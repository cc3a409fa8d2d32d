"""TEST INFRASTRUCTURE: caller-built job tables for zxc_b200_decode_blocks (include/zxc_b200.h) and what every job of
such a table must produce.  Shared by tests/test_device_abi_gpu.py (the compiled kernel on the device) and
tests/test_simt_layouts.py (the kernel source on the CPU warp emulator).

A job table is a numpy structured array of JOB_DT, the layout of zxc_b200_job_t (the dtype bench.py uses).  A `Case`
is a source buffer holding one or more frames back to back, the jobs of all their blocks in frame order with the
outputs packed end to end, and the bytes those outputs must hold."""
import ctypes as C
import os

import numpy as np

import zxc_corpus as zc

JOB_DT = np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("src_len", "<u4"), ("dst_cap", "<u4")])
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class Info(C.Structure):
    _fields_ = [("decoded_size", C.c_uint64), ("block_size", C.c_uint32), ("n_blocks", C.c_uint32),
                ("dict_id", C.c_uint32), ("has_checksum", C.c_int), ("seekable", C.c_int), ("global_hash", C.c_uint32)]


def plan(prod, frame):
    """(jobs, Info) from the product's host walk of a frame in host memory (no device needed)"""
    fb = np.frombuffer(bytes(frame), np.uint8)
    L = prod.lib
    L.zxc_b200_plan_frame.restype = C.c_int64
    L.zxc_b200_plan_frame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    info = Info()
    nb = L.zxc_b200_plan_frame(fb.ctypes.data, fb.size, None, 0, C.byref(info))
    assert nb >= 0, nb
    jobs = np.zeros(max(nb, 1), JOB_DT)
    assert L.zxc_b200_plan_frame(fb.ctypes.data, fb.size, jobs.ctypes.data, nb, None) == nb
    return jobs[:nb], info


def pow2_at_least(n):
    b = 4096
    while b < n:
        b *= 2
    return b


class Case:
    """frames (with their expected output) concatenated into one source; jobs in frame order, outputs packed"""

    def __init__(self, prod, frames, dict=None, dict_huf=None, verify=0):
        srcs, jobs, want, so, do = [], [], [], 0, 0
        self.has_checksum = True
        for fr, exp in frames:
            fb = bytes(fr)
            j, info = plan(prod, fb)
            assert int(j["dst_cap"].astype(np.int64).sum()) == len(exp)
            self.has_checksum &= bool(info.has_checksum)
            j = j.copy()
            j["src_off"] += so
            j["dst_off"] += do
            srcs.append(fb)
            jobs.append(j)
            want.append(bytes(exp))
            so += len(fb)
            do += len(exp)
        self.src = np.frombuffer(b"".join(srcs), np.uint8)
        self.jobs = np.concatenate(jobs) if jobs else np.zeros(0, JOB_DT)
        self.want = np.frombuffer(b"".join(want), np.uint8)
        self.dict, self.dict_huf = dict, dict_huf
        assert not verify or self.has_checksum
        self.verify = verify
        self.block_size = pow2_at_least(int(self.jobs["dst_cap"].max()) if self.jobs.size else 0)

    def expected(self, jobs=None, ref_off=None):
        """[(status, bytes)] per job for an undamaged source: every job fills its window"""
        jobs = self.jobs if jobs is None else jobs
        ref_off = self.jobs["dst_off"] if ref_off is None else ref_off
        return [(int(c), self.want[int(o):int(o) + int(c)]) for c, o in zip(jobs["dst_cap"], ref_off)]


def laid_out(jobs, gap=0, order=None, base=0):
    """(new jobs, ref_off): the output windows placed one after the other in frame order with `gap` bytes between
    them, starting at `base`; rows then permuted by `order`.  ref_off[i] is row i's original dst_off."""
    caps = jobs["dst_cap"].astype(np.uint64)
    out = jobs.copy()
    out["dst_off"] = base + np.concatenate([[0], np.cumsum(caps + gap)[:-1]]).astype(np.uint64) if jobs.size else []
    ref = jobs["dst_off"].copy()
    if order is not None:
        out, ref = out[order], ref[order]
    return out, ref


def oracle_verdicts(orc, src, jobs, dict=None, dict_huf=None, verify=0):
    """[(status, bytes or None)] per job from the scalar per-block decoder at each job's own dst_cap"""
    src = np.ascontiguousarray(src)
    dp = np.frombuffer(dict, np.uint8) if dict else None
    hp = np.frombuffer(dict_huf, np.uint8) if dict_huf is not None else None
    res = []
    for j in jobs:
        so, sl, cap = int(j["src_off"]), int(j["src_len"]), int(j["dst_cap"])
        out = np.zeros(cap + 64, np.uint8)
        r = orc.lib.zxo_decode_block(src.ctypes.data + so, sl, out.ctypes.data, cap,
                                     dp.ctypes.data if dp is not None else None, dp.size if dp is not None else 0,
                                     hp.ctypes.data if hp is not None else None, verify)
        res.append((int(r), out[:r].copy() if r >= 0 else None))
    return res


def damage(src, jobs, rng, n):
    """copy of `src` with `n` seeded byte changes inside the jobs' payloads, checksum words included (block headers
    untouched: the host walk, not the kernel, judges those)"""
    s = src.copy()
    for _ in range(n):
        j = jobs[int(rng.integers(0, jobs.size))]
        lo = int(j["src_off"]) + 8
        hi = int(j["src_off"]) + int(j["src_len"])
        if hi > lo:
            s[int(rng.integers(lo, hi))] ^= int(rng.integers(1, 256))
    return s


def windows_mask(size, jobs, base=0):
    m = np.zeros(size, bool)
    for j in jobs:
        a = base + int(j["dst_off"])
        m[a:a + int(j["dst_cap"])] = True
    return m


# A kernel status that differs from the scalar decoder's on purpose goes here with its reason.  None so far: at the
# job's own dst_cap the kernel reports exactly what zxo_decode_block reports.
STATUS_MAP = {}


def check(dst, base, jobs, status, expected, sentinel, what=""):
    """per-job status and bytes against `expected`, and every byte of `dst` outside the windows still `sentinel`"""
    assert len(status) == jobs.size
    bad = []
    for i, (s, (es, eb)) in enumerate(zip(status, expected)):
        s = STATUS_MAP.get(int(s), int(s))
        if s != es:
            bad.append((i, "status", s, es))
        elif s >= 0:
            a = base + int(jobs[i]["dst_off"])
            if not np.array_equal(dst[a:a + s], eb):
                bad.append((i, "bytes", s, int(np.argmax(dst[a:a + s] != eb))))
    assert not bad, (what, len(bad), bad[:8])
    outside = ~windows_mask(dst.size, jobs, base)
    n_changed = int((dst[outside] != sentinel).sum())
    assert n_changed == 0, (what, "bytes written outside the job windows", n_changed,
                            np.nonzero(outside & (dst != sentinel))[0][:8] - base)
    return len(expected)


# ---- inputs ------------------------------------------------------------------------------------------------------
GOLDEN_MIX = ["all_256_values", "all_zeros_4k", "all_zeros_64k", "glo_pivco_wide_l7", "long_match_64k",
              "max_offset_128k", "multiblock_mixed", "multiblock_text", "one_byte", "random_256", "random_4k",
              "random_64k", "seekable_1block", "seekable_4blocks", "short_matches_4k", "text_1k", "text_64k",
              "text_64k_bs2m", "text_64k_level1", "text_64k_level2", "text_64k_level3", "text_64k_level4",
              "text_64k_level5", "text_64k_level6", "text_8k_bs4k"]
GOLDEN_CHECKSUM = ["long_match_checksum", "random_4k_checksum", "seekable_checksum", "text_1k_checksum",
                   "zeros_4k_checksum"]


# tests/golden/format vectors without a dictionary: GLO with an RLE literal section at level 3, 16-bit offsets, Huffman
GOLDEN_FORMAT = ["03_block_ghi", "04_block_glo", "05_block_glo_huffman", "07_multiple_blocks", "10_glo_offset16",
                 "11_glo_rle", "13_glo_huffman_wide"]


def golden(name, orc=None):
    """(frame, expected output) of a conformance vector; a format vector (name in GOLDEN_FORMAT) has no stored output,
    so the oracle (pinned against it by tests/test_oracle.py) supplies it"""
    if name in GOLDEN_FORMAT:
        fr = open(os.path.join(G, "format", name + ".zxc"), "rb").read()
        r, out = orc.decompress(fr, 1 << 20)
        assert r > 0, (name, r)
        return fr, out.tobytes()
    fr = open(os.path.join(G, "valid", name + ".zxc"), "rb").read()
    exp = open(os.path.join(G, "valid", name + ".expected"), "rb").read()
    return fr, exp


def mixed_input(n=1 << 20, seed=1):
    """text, incompressible stretches (RAW blocks), short periods (offsets below 32), a 1500-byte period (matches far
    longer than the 4 KiB ring), a varying byte before every four 0xAA (literal runs: RLE sections) and a repeat
    exactly 65536 bytes back; the random stretch and the run pattern each cover whole 64 KiB blocks"""
    rng = np.random.default_rng(seed)
    rle = np.full((n // 40 + 80000) // 5 * 5, 0xAA, np.uint8)
    rle[::5] = rng.integers(0, 256, rle.size // 5, dtype=np.uint8)
    far = zc.gen_random(65536 + 64, seed=seed + 6)
    far[65536:] = far[:64]
    parts = [zc.silesia_shaped(n // 8, seed=seed), zc.gen_random(n // 16 + 140000, seed=seed + 1),
             zc.gen_periodic(n // 32, 7, seed=seed + 2), zc.gen_periodic(n // 32, 3, seed=seed + 3),
             zc.gen_periodic(n // 16, 1500, seed=seed + 4), rle, far, zc.gen_text(n // 8, seed=seed + 7)]
    return np.resize(np.concatenate(parts)[int(rng.integers(0, 64)):], n)


def dict_records(d, n_records=24, record=4096, seed=100):
    """records that open with the dictionary repeated (a match at the record's first byte reaches back to the
    dictionary's first byte and runs through its last), then its last and first bytes, and end with all of it"""
    k = min(len(d), 40)
    head = d * (48 // len(d) + 1)
    recs = [(head + d[-k:] + d[:k] + zc.gen_text(3000, seed=seed + i).tobytes() + d)[:record] for i in range(n_records)]
    return np.frombuffer(b"".join(recs), np.uint8)


def golden_dict_huf():
    """the shared Huffman table of the conformance text dictionary (tests/golden/valid/dict_text.zxd)"""
    b = open(os.path.join(G, "valid", "dict_text.zxd"), "rb").read()
    n = int.from_bytes(b[6:8], "little")
    return b[16 + n:16 + n + 128]


def assert_block_kinds(orc, frames):
    """the frames hold RAW, GHI and GLO blocks, RLE and Huffman sections and offsets below 32 between them"""
    tot = {}
    for fr in frames:
        rc, st = orc.stats(fr)
        assert rc == 0, rc
        for k, v in st.items():
            tot[k] = tot.get(k, 0) + v
    for k in ("raw_blocks", "ghi_blocks", "glo_blocks", "rle_blocks", "huf_blocks", "off_lt32"):
        assert tot[k] > 0, (k, tot)
    return tot
