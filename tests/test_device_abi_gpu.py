"""The device-resident entry points of include/zxc_b200.h -- zxc_b200_plan_frame, zxc_b200_decode_scratch_size,
zxc_b200_decode_blocks, zxc_b200_reduce_status -- called the way bench.py and the multi-GPU pipeline call them:
caller-owned device buffers and a caller-built job table.  Every job's status and bytes are checked against the
original input (valid frames) or against the scalar per-block decoder zxo_decode_block at the job's own dst_cap
(damaged frames), and every destination byte outside the job windows must keep the sentinel it was filled with.

Frames come from the GPU encoder and from the conformance vectors; none of these tests needs the reference build
except the one optional encoder-identity test.  tests/test_simt_layouts.py runs the same matrix on the CPU emulator."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import zxc_corpus as zc
import zxc_jobs as zj
from test_oracle import golden_dicts

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

DST_SHIFTS = (0, 1, 2, 3, 4, 7, 8, 15)
SRC_SHIFTS = (0, 1, 3, 8, 13)
SENTINELS = (0xA5, 0x5A)
GUARD = 4096  # bytes of sentinel either side of the outermost windows
UNSET = 0x7AAAAAAA  # status a job has not written
LEVELS = (1, 3, 6, 7)  # GHI, GLO, Huffman literals, Huffman tokens; every frame also holds RAW blocks


class Api:
    def __init__(self, prod):
        self.L = L = prod.lib
        L.zxc_b200_decode_scratch_size.restype = C.c_size_t
        L.zxc_b200_decode_scratch_size.argtypes = [C.c_uint32]
        L.zxc_b200_decode_blocks.restype = C.c_int
        L.zxc_b200_decode_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                             C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_int,
                                             C.c_void_p]
        L.zxc_b200_reduce_status.restype = C.c_int64
        L.zxc_b200_reduce_status.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.zxc_b200_launch_count.restype = C.c_uint64
        L.zxc_b200_plan_frame.restype = C.c_int64
        L.zxc_b200_plan_frame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]

    def scratch_size(self, bs):
        return int(self.L.zxc_b200_decode_scratch_size(bs))

    def decode(self, *a):
        return self.L.zxc_b200_decode_blocks(*a)

    def reduce(self, d_status, d_jobs, n, stream=None):
        return self.L.zxc_b200_reduce_status(d_status, d_jobs, n, stream)

    def launches(self):
        return int(self.L.zxc_b200_launch_count())


@pytest.fixture(scope="module")
def api(prod):
    return Api(prod)


def dev_bytes(b):
    return torch.from_numpy(np.frombuffer(bytes(b), np.uint8).copy()).cuda()


def dev_jobs(jobs):
    return torch.from_numpy(np.ascontiguousarray(jobs).view(np.uint8).copy()).cuda()


class Launch:
    """Device buffers for one zxc_b200_decode_blocks call: the source `src_shift` bytes past an allocation's start, the
    destination `dst_shift` bytes past a 4 KiB guard band, both filled around the data (source: 0xEE, destination:
    the sentinel); the dictionary and its Huffman table in allocations of their own."""

    def __init__(self, api, src, jobs, block_size, src_shift=0, dst_shift=0, sentinel=0xA5, dict=None, dict_huf=None,
                 dict_shift=None, verify=0, scratch=None):
        self.api, self.jobs, self.bs, self.verify, self.sentinel = api, np.ascontiguousarray(jobs), block_size, verify, sentinel
        src = np.array(src, np.uint8)  # a writable copy for torch.from_numpy
        self.s = torch.full((src_shift + src.size + 64,), 0xEE, dtype=torch.uint8, device="cuda")
        self.s[src_shift:src_shift + src.size].copy_(torch.from_numpy(src))
        self.src_ptr = self.s.data_ptr() + src_shift
        end = int((self.jobs["dst_off"] + self.jobs["dst_cap"]).max()) if self.jobs.size else 0
        self.base = GUARD + dst_shift
        self.d = torch.full((self.base + end + GUARD,), sentinel, dtype=torch.uint8, device="cuda")
        self.d_jobs = dev_jobs(self.jobs) if self.jobs.size else torch.zeros(32, dtype=torch.uint8, device="cuda")
        self.status = torch.full((max(self.jobs.size, 1),), UNSET, dtype=torch.int32, device="cuda")
        self.ss = api.scratch_size(block_size)
        self.scratch = scratch if scratch is not None else torch.empty(self.ss, dtype=torch.uint8, device="cuda")
        self.dict_ptr, self.dict_size, self.huf_ptr = None, 0, None
        if dict:
            if dict_shift is None:  # exact-size allocation
                self.dd = dev_bytes(dict)
                self.dict_ptr = self.dd.data_ptr()
            else:
                self.dd = torch.full((dict_shift + len(dict) + 64,), 0xCC, dtype=torch.uint8, device="cuda")
                self.dd[dict_shift:dict_shift + len(dict)].copy_(torch.from_numpy(np.frombuffer(dict, np.uint8).copy()))
                self.dict_ptr = self.dd.data_ptr() + dict_shift
            self.dict_size = len(dict)
        if dict_huf is not None:
            self.hh = dev_bytes(dict_huf)
            self.huf_ptr = self.hh.data_ptr()

    def run(self, stream=None, sync=True, presync=True):
        if presync:  # the fills above ran on torch's current stream
            torch.cuda.synchronize()
        st = stream.cuda_stream if stream is not None else None
        rc = self.api.decode(self.src_ptr, self.d.data_ptr() + self.base, self.d_jobs.data_ptr(), self.jobs.size,
                             self.status.data_ptr(), self.dict_ptr, self.dict_size, self.huf_ptr, self.scratch.data_ptr(),
                             self.ss, self.bs, self.verify, st)
        assert rc == 0, rc
        if sync:
            (stream or torch.cuda.current_stream()).synchronize()
        return self

    def result(self):
        return self.status.cpu().numpy()[:self.jobs.size], self.d.cpu().numpy()

    def check(self, expected, what=""):
        st, dst = self.result()
        return zj.check(dst, self.base, self.jobs, st, expected, self.sentinel, what)


def gpu_frames(prod, data, levels=LEVELS, bs=65536, checksum=0, **kw):
    out = []
    for lv in levels:
        fr = prod.compress(data, level=lv, block_size=bs, checksum=checksum, **kw)
        assert not isinstance(fr, int), (lv, fr)
        out.append((fr, data.tobytes()))
    return out


@pytest.fixture(scope="module")
def mixed(prod, orc):
    """GPU-encoded frames of the mixed input at levels 1, 3, 6, 7 followed by the conformance vectors, one table"""
    data = zj.mixed_input(600000, seed=2)
    frames = gpu_frames(prod, data) + [zj.golden(n, orc) for n in zj.GOLDEN_MIX + zj.GOLDEN_FORMAT]
    zj.assert_block_kinds(orc, [f for f, _ in frames])
    return zj.Case(prod, frames)


@pytest.fixture(scope="module")
def mixed_cks(prod, orc):
    data = zj.mixed_input(300000, seed=3)
    frames = gpu_frames(prod, data, checksum=1) + [zj.golden(n) for n in zj.GOLDEN_CHECKSUM]
    return zj.Case(prod, frames, verify=1)


# ---- layouts and guard bands ------------------------------------------------------------------------------------
def test_layouts_and_guard_bands(api, mixed, mixed_cks):
    """every destination shift with two seeded source shifts over RAW, GHI, GLO and Huffman blocks (al16 false in
    ring_flush, the aligned and unaligned section loads), under two sentinels; the checksummed frames with verify on"""
    rng = np.random.default_rng(1)
    n = 0
    for case in (mixed, mixed_cks):
        for i, ds in enumerate(DST_SHIFTS):
            for ss in rng.choice(SRC_SHIFTS, 2, replace=False):
                L = Launch(api, case.src, case.jobs, case.block_size, src_shift=int(ss), dst_shift=ds,
                           sentinel=SENTINELS[i & 1], verify=case.verify).run()
                n += L.check(case.expected(), (ds, int(ss)))
    assert n > 0


def test_gaps_and_orders(api, mixed):
    """gaps of 0, 1, 13 and 4101 bytes between windows; rows in frame order, reversed and in a seeded permutation"""
    rng = np.random.default_rng(2)
    n = mixed.jobs.size
    for gap in (0, 1, 13, 4096 + 5):
        for name, order in (("frame", None), ("reversed", np.arange(n)[::-1]), ("seeded", rng.permutation(n))):
            jobs, ref_off = zj.laid_out(mixed.jobs, gap=gap, order=order)
            L = Launch(api, mixed.src, jobs, mixed.block_size, dst_shift=gap % 16, sentinel=SENTINELS[gap & 1]).run()
            L.check(mixed.expected(jobs, ref_off), (gap, name))


# ---- job tables -------------------------------------------------------------------------------------------------
def test_rank_slices_as_the_pipeline_builds_them(api, prod):
    """Block ranges of one frame rebased with zxc_b200/shard.py, each rank's compressed slice in an allocation of its
    own, and every rank decoding straight into its view of one shared output buffer, as rank 0 of bench.py's one-frame
    pipeline decodes into the gather buffer.  The shared buffer's base is shifted by 0, 3 and 13 bytes, so the ranks'
    views are misaligned too; the whole buffer must hold the input, its guard bands the sentinel."""
    from zxc_b200 import shard
    data = zj.mixed_input(1 << 20, seed=4)
    bs = 65536
    case = zj.Case(prod, gpu_frames(prod, data, levels=(3,), bs=bs, seekable=1))
    comp = case.jobs["src_len"].astype(np.int64)
    total = data.size
    ss = api.scratch_size(bs)
    scratch = torch.empty(ss, dtype=torch.uint8, device="cuda")
    want_all = torch.from_numpy(case.want.copy()).cuda()
    for world, shift, sentinel in ((2, 0, 0xA5), (3, 3, 0x5A), (5, 13, 0xA5)):
        base = GUARD + shift
        d_all = torch.full((base + total + GUARD,), sentinel, dtype=torch.uint8, device="cuda")
        for r, (b0, b1) in enumerate(shard.partition_blocks(comp, world)):
            lo, hi, dlo, dhi = shard.rank_slice(comp, bs, total, b0, b1)
            sub = shard.rebase_jobs(case.jobs, b0, b1, lo, dlo)
            if sub.size == 0:
                continue
            mine = torch.from_numpy(case.src[lo:hi].copy()).cuda()
            view = d_all[base + dlo:base + dhi]
            d_jobs = dev_jobs(sub)
            status = torch.full((sub.size,), UNSET, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            assert api.decode(mine.data_ptr(), view.data_ptr(), d_jobs.data_ptr(), sub.size, status.data_ptr(), None, 0,
                              None, scratch.data_ptr(), ss, bs, 0, None) == 0
            torch.cuda.synchronize()
            assert np.array_equal(status.cpu().numpy(), sub["dst_cap"].astype(np.int32)), (world, r)
            assert api.reduce(status.data_ptr(), d_jobs.data_ptr(), sub.size, None) == dhi - dlo
        assert torch.equal(d_all[base:base + total], want_all), world
        assert bool((d_all[:base] == sentinel).all()) and bool((d_all[base + total:] == sentinel).all()), world
        del d_all


def test_one_source_two_windows_and_the_short_tail(api, mixed):
    jobs = mixed.jobs
    twice = np.concatenate([jobs, jobs[::-1]])
    lay, ref_off = zj.laid_out(twice, gap=7)
    Launch(api, mixed.src, lay, mixed.block_size, dst_shift=3).run().check(mixed.expected(lay, ref_off), "twice")
    tails = jobs[jobs["dst_cap"] % 4096 != 0]
    assert tails.size > 0
    lay, ref_off = zj.laid_out(tails, gap=1)
    Launch(api, mixed.src, lay, mixed.block_size, dst_shift=5).run().check(mixed.expected(lay, ref_off), "tails")


def test_windows_smaller_than_the_block(api, mixed, orc):
    """dst_cap below what a block produces: zxo_decode_block's verdict at that cap, nothing written past the window"""
    rng = np.random.default_rng(5)
    for k in (1, 7, 16, 17, 4095):
        short = mixed.jobs.copy()
        short["dst_cap"] = np.maximum(short["dst_cap"].astype(np.int64) - k, 1).astype(np.uint32)
        lay, _ = zj.laid_out(short, gap=int(rng.integers(0, 20)))
        want = zj.oracle_verdicts(orc, mixed.src, lay)
        assert sum(s < 0 for s, _ in want) > 10
        L = Launch(api, mixed.src, lay, mixed.block_size, dst_shift=int(rng.integers(0, 16)),
                   sentinel=SENTINELS[k & 1]).run()
        L.check(want, ("short", k))


# ---- block sizes ------------------------------------------------------------------------------------------------
def test_every_block_size(api, prod, simt_stride):
    """4 KiB .. 2 MiB blocks, each frame ending in a partial block of 1, 15, 16 or 17 bytes, decoded with exactly the
    scratch zxc_b200_decode_scratch_size reports"""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    for k in range(12, 22):
        bs = 1 << k
        frames = []
        for i, tail in enumerate((1, 15, 16, 17)):
            data = zj.mixed_input(2 * bs + tail + 1024, seed=k * 7 + i)[:2 * bs + tail]
            frames += gpu_frames(prod, data, levels=(LEVELS[i],), bs=bs, checksum=i & 1)
        case = zj.Case(prod, frames)
        assert {int(c) for c in case.jobs["dst_cap"]} == {bs, 1, 15, 16, 17}
        assert api.scratch_size(bs) >= sm * 7 * 4 * simt_stride(bs) + 32
        L = Launch(api, case.src, case.jobs, bs, dst_shift=k % 16, sentinel=SENTINELS[k & 1]).run()
        L.check(case.expected(), bs)
        del L
        torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def simt_stride():
    """per-warp scratch stride from the kernel source's own formula (tests/simt build)"""
    import zxc_simt as zs
    lib = zs.lib()
    lib.simt_scratch_stride.restype = C.c_uint32
    lib.simt_scratch_stride.argtypes = [C.c_uint32]
    return lambda bs: int(lib.simt_scratch_stride(bs))


# ---- dictionaries -----------------------------------------------------------------------------------------------
DICT_SIZES = (1, 7, 8, 9, 16, 17, 31, 4096, 65535)


def dict_frames(prod, size, level, huf):
    d = zc.gen_text(size, seed=size).tobytes()
    data = zj.dict_records(d)
    fr = prod.compress(data, level=level, block_size=4096, dict=d, dict_huf=huf)
    assert not isinstance(fr, int), (size, level, fr)
    return d, data, fr


@pytest.mark.parametrize("size", DICT_SIZES)
def test_dictionaries(api, prod, orc, size):
    """levels 1, 3, 5, 6 (6 with the dictionary's shared Huffman table in its own allocation); records open with the
    dictionary's last and first bytes; the dictionary in an exact-size allocation and at an odd address"""
    huf = zj.golden_dict_huf()
    for level in (1, 3, 5, 6):
        h = huf if level == 6 else None
        d, data, fr = dict_frames(prod, size, level, h)
        case = zj.Case(prod, [(fr, data.tobytes())], dict=d, dict_huf=h)
        no_dict = zj.oracle_verdicts(orc, case.src, case.jobs)
        assert any(s < 0 for s, _ in no_dict), "no block refers to the dictionary"
        if h is not None and size <= 31:  # its blocks decode their literals with the dictionary's table
            assert all(s == -15 for s, _ in zj.oracle_verdicts(orc, case.src, case.jobs, d, None))
        for i, dshift in enumerate((None, 3)):
            L = Launch(api, case.src, case.jobs, case.block_size, src_shift=i * 5, dst_shift=i * 9 + level,
                       sentinel=SENTINELS[i], dict=d, dict_huf=h, dict_shift=dshift).run()
            L.check(case.expected(), (size, level, dshift))


def test_dictionary_size_limit(prod):
    assert prod.compress(zc.gen_text(8192), level=3, dict=zc.gen_text(65536).tobytes()) == -17  # DICT_TOO_LARGE


def test_golden_dictionary_vectors(api, prod):
    dicts = golden_dicts()
    for name in ("dict_http", "dict_seekable_l7"):
        fr, exp = zj.golden(name)
        d, h = dicts[int.from_bytes(fr[7:11], "little")]
        case = zj.Case(prod, [(fr, exp)], dict=d, dict_huf=h)
        for ds in DST_SHIFTS:
            Launch(api, case.src, case.jobs, case.block_size, src_shift=ds % 5, dst_shift=ds, sentinel=SENTINELS[ds & 1],
                   dict=d, dict_huf=h, dict_shift=None if ds & 1 else ds).run().check(case.expected(), (name, ds))


def test_dictionary_frames_match_the_reference(prod, ref):
    """optional (needs oracle/_ref): the GPU encoder's dictionary frames are the reference's, byte for byte"""
    huf = zj.golden_dict_huf()
    for size in DICT_SIZES:
        for level in (1, 3, 5, 6):
            h = huf if level == 6 else None
            d, data, fr = dict_frames(prod, size, level, h)
            want = ref.compress(data, level=level, block_size=4096, dict=d, dict_huf=h)
            assert np.array_equal(fr, want), (size, level)


# ---- per-job verdicts on damaged frames -------------------------------------------------------------------------
def _damaged(api, orc, case, trials, seed, verify, per_trial=(1, 5)):
    rng = np.random.default_rng(seed)
    lay, _ = zj.laid_out(case.jobs, gap=3)
    clean = zj.oracle_verdicts(orc, case.src, lay, case.dict, case.dict_huf, verify)
    hit = 0
    for t in range(trials):
        src = zj.damage(case.src, case.jobs, rng, int(rng.integers(*per_trial)))
        want = zj.oracle_verdicts(orc, src, lay, case.dict, case.dict_huf, verify)
        L = Launch(api, src, lay, case.block_size, dst_shift=t % 16, sentinel=SENTINELS[t & 1], dict=case.dict,
                   dict_huf=case.dict_huf, verify=verify).run()
        L.check(want, ("damaged", seed, t))
        hit += sum(1 for a, b in zip(want, clean) if a[0] != b[0] or (a[0] >= 0 and not np.array_equal(a[1], b[1])))
    return hit


def test_damaged_blocks_per_job_verdicts(api, prod, orc, mixed, mixed_cks):
    """seeded payload damage (block headers intact): every job's status is zxo_decode_block's, and so are its bytes
    where it succeeds.  Frames with and without checksums, verify off and on (the checksum word can be hit too)"""
    hit = _damaged(api, orc, mixed, 40, 1, 0, per_trial=(3, 12))
    for verify in (0, 1):
        hit += _damaged(api, orc, mixed_cks, 25, 2 + verify, verify, per_trial=(3, 12))
    for size, level in ((9, 3), (31, 6), (4096, 1), (4096, 6)):
        h = zj.golden_dict_huf() if level == 6 else None
        d, data, fr = dict_frames(prod, size, level, h)
        hit += _damaged(api, orc, zj.Case(prod, [(fr, data.tobytes())], dict=d, dict_huf=h), 12, size + level, 0)
    assert hit >= 400, hit


def test_damaged_checksum_word(api, orc, mixed_cks):
    rng = np.random.default_rng(9)
    src = mixed_cks.src.copy()
    for j in mixed_cks.jobs:
        src[int(j["src_off"]) + int(j["src_len"]) - 1 - int(rng.integers(0, 4))] ^= 0x41
    for verify in (0, 1):
        want = zj.oracle_verdicts(orc, src, mixed_cks.jobs, verify=verify)
        assert all((s == -7) == bool(verify) for s, _ in want)
        Launch(api, src, mixed_cks.jobs, mixed_cks.block_size, dst_shift=3, verify=verify).run().check(want, verify)


# ---- 64-bit offsets ---------------------------------------------------------------------------------------------
def test_offsets_above_4gib(api, prod):
    """the frame at byte 2^32 + 7 of a source a little over 4 GiB; windows near and above 2^32 of a 4.6 GiB output,
    one of them straddling 2^32.  A 32-bit truncation of either offset would read the wrong bytes or write at the
    window's offset modulo 2^32, which must keep its sentinel."""
    data = zj.mixed_input(300 * 4096 - 123, seed=6)
    fr = gpu_frames(prod, data, levels=(3,), bs=4096)[0][0]
    case = zj.Case(prod, [(fr, data.tobytes())])
    jobs = case.jobs.copy()
    n = jobs.size
    assert n >= 300
    S = 1 << 32
    src_at = S + 7
    d_src = torch.empty(src_at + case.src.size + 64, dtype=torch.uint8, device="cuda")
    d_src[src_at:src_at + case.src.size].copy_(torch.from_numpy(case.src.copy()))
    jobs["src_off"] += src_at
    # windows: the first 40 just below 2^32 (the 40th straddles it), the rest spread over the next 600 MiB
    caps = jobs["dst_cap"].astype(np.int64)
    offs = np.empty(n, np.int64)
    offs[:40] = S - 39 * 4096 - 2000 + np.arange(40) * 4096
    offs[40:] = S + 4096 + np.arange(n - 40) * ((600 << 20) // (n - 40)) + np.arange(n - 40) % 13
    assert offs[39] < S < offs[39] + caps[39]
    jobs["dst_off"] = offs
    size = int(offs[-1] + caps[-1]) + GUARD
    sentinel = 0xA5
    d_dst = torch.full((size,), sentinel, dtype=torch.uint8, device="cuda")
    d_jobs = dev_jobs(jobs)
    status = torch.full((n,), UNSET, dtype=torch.int32, device="cuda")
    ss = api.scratch_size(4096)
    scratch = torch.empty(ss, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    assert api.decode(d_src.data_ptr(), d_dst.data_ptr(), d_jobs.data_ptr(), n, status.data_ptr(), None, 0, None,
                      scratch.data_ptr(), ss, 4096, 0, None) == 0
    torch.cuda.synchronize()
    assert np.array_equal(status.cpu().numpy(), caps)
    want = torch.from_numpy(case.want.copy()).cuda()
    ref_off = case.jobs["dst_off"].astype(np.int64)
    n_sent_in = 0
    for i in range(n):
        o, c, r = int(offs[i]), int(caps[i]), int(ref_off[i])
        assert torch.equal(d_dst[o:o + c], want[r:r + c]), i
        n_sent_in += int((want[r:r + c] == sentinel).sum())
        if o + c > S:  # where a truncated offset would have written the part above 2^32
            assert bool((d_dst[max(o, S) - S:o + c - S] == sentinel).all()), i
    # nothing else changed: the sentinel count is what the windows leave
    assert int((d_dst == sentinel).sum()) == size - int(caps.sum()) + n_sent_in
    assert api.reduce(status.data_ptr(), d_jobs.data_ptr(), n, None) == int(caps.sum())
    del d_src, d_dst, scratch
    torch.cuda.empty_cache()


# ---- grid and streams -------------------------------------------------------------------------------------------
def _small_jobs(case, n):
    """n rows cycled from the case's blocks of at most 4 KiB, windows packed"""
    small = case.jobs[case.jobs["dst_cap"] <= 4096]
    rows = small[np.arange(n) % small.size]
    return zj.laid_out(rows)


def test_job_counts_around_the_resident_grid(api, mixed):
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    R = sm * 7 * 4
    for n in (1, 31, R - 1, R, R + 1, 100003):
        jobs, ref_off = _small_jobs(mixed, n)
        L = Launch(api, mixed.src, jobs, 4096, dst_shift=n % 16, sentinel=SENTINELS[n & 1]).run()
        st = L.status.cpu().numpy()
        assert np.array_equal(st, jobs["dst_cap"].astype(np.int32)), n
        want = np.concatenate([mixed.want[int(o):int(o) + int(c)] for o, c in zip(ref_off, jobs["dst_cap"])])
        end = L.base + want.size
        assert torch.equal(L.d[L.base:end], torch.from_numpy(want).cuda()), n
        assert bool((L.d[:L.base] == L.sentinel).all()) and bool((L.d[end:] == L.sentinel).all()), n
        assert api.reduce(L.status.data_ptr(), L.d_jobs.data_ptr(), n, None) == want.size


def test_two_launches_on_one_scratch(api, mixed):
    """the work counters live in the scratch tail: a second launch must not depend on anyone re-zeroing them"""
    jobs, ref_off = zj.laid_out(mixed.jobs, gap=2)
    a = Launch(api, mixed.src, jobs, mixed.block_size, dst_shift=1)
    b = Launch(api, mixed.src, jobs[::-1].copy(), mixed.block_size, dst_shift=6, sentinel=0x5A, scratch=a.scratch)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    a.run(stream=s, sync=False, presync=False)
    b.run(stream=s, sync=False, presync=False)
    with torch.cuda.stream(s):  # the same launch again, on counters b left behind
        a.status.fill_(UNSET)
        a.d.fill_(a.sentinel)
    a.run(stream=s, sync=False, presync=False)
    s.synchronize()
    a.check(mixed.expected(jobs, ref_off), "a")
    b.check(mixed.expected(jobs[::-1], ref_off[::-1]), "b")


def test_two_streams_in_flight(api, mixed, mixed_cks):
    """two launches at once on two non-default streams, each with its own scratch, status and output; the host waits
    on each stream alone"""
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    j1, r1 = _small_jobs(mixed, 50000)
    j2, r2 = zj.laid_out(mixed_cks.jobs, gap=9, order=np.random.default_rng(3).permutation(mixed_cks.jobs.size))
    a = Launch(api, mixed.src, j1, 4096, dst_shift=2)
    b = Launch(api, mixed_cks.src, j2, mixed_cks.block_size, dst_shift=11, sentinel=0x5A, verify=1)
    torch.cuda.synchronize()
    n0 = api.launches()
    for L, s in ((a, s1), (b, s2)):
        assert api.decode(L.src_ptr, L.d.data_ptr() + L.base, L.d_jobs.data_ptr(), L.jobs.size, L.status.data_ptr(),
                          None, 0, None, L.scratch.data_ptr(), L.ss, L.bs, L.verify, s.cuda_stream) == 0
    assert api.launches() - n0 == 2
    s2.synchronize()
    b.check(mixed_cks.expected(j2, r2), "stream 2")
    s1.synchronize()
    a.check(mixed.expected(j1, r1), "stream 1")
    assert api.reduce(b.status.data_ptr(), b.d_jobs.data_ptr(), j2.size, s2.cuda_stream) == int(j2["dst_cap"].sum())


# ---- reduce_status ----------------------------------------------------------------------------------------------
def reduce_ref(status, caps):
    bad = np.nonzero((status < 0) | (status.astype(np.int64) != caps.astype(np.int64)))[0]
    if bad.size:
        s = int(status[bad[0]])
        return s if s < 0 else -8
    return int(caps.astype(np.int64).sum())


def test_reduce_status(api):
    rng = np.random.default_rng(4)
    cases = []
    for n in (1, 255, 256, 257, 1000, 70000):
        caps = rng.integers(1, 65537, n).astype(np.uint32)
        cases.append((caps.astype(np.int32), caps))
    base = cases[-1]
    for idx in (0, 69999, 65536 + 17, 256, 511, 512, 30000):
        for val in (-8, -2, -13, "mismatch"):
            st = base[0].copy()
            st[idx] = int(base[1][idx]) - 1 if val == "mismatch" else val
            cases.append((st, base[1]))
    st = base[0].copy()  # several bad jobs in different 256-job blocks: the lowest index decides
    for idx, v in ((60000, -9), (40000, -7), (300, 5), (44444, -13)):
        st[idx] = v
    cases.append((st, base[1]))
    st = base[0].copy()
    st[1000], st[999] = -10, int(base[1][999]) + 1
    cases.append((st, base[1]))
    big = np.full(70000, 65536, np.uint32)  # all good, sum above 2^32
    cases.append((big.astype(np.int32), big))
    for st, caps in cases:
        jobs = np.zeros(caps.size, zj.JOB_DT)
        jobs["dst_cap"] = caps
        d_st = torch.from_numpy(st.copy()).cuda()
        d_jobs = dev_jobs(jobs)
        s = torch.cuda.Stream()
        torch.cuda.synchronize()
        assert api.reduce(d_st.data_ptr(), d_jobs.data_ptr(), st.size, s.cuda_stream) == reduce_ref(st, caps)
    assert reduce_ref(big.astype(np.int32), big) == 70000 * 65536 > 1 << 32
    d = torch.zeros(8, dtype=torch.int32, device="cuda")
    assert api.reduce(d.data_ptr(), d.data_ptr(), 0, None) == 0


# ---- API edges --------------------------------------------------------------------------------------------------
def test_api_edges(api, prod, mixed, simt_stride):
    L = Launch(api, mixed.src, mixed.jobs, mixed.block_size)
    a = [L.src_ptr, L.d.data_ptr() + L.base, L.d_jobs.data_ptr(), mixed.jobs.size, L.status.data_ptr(), None, 0, None,
         L.scratch.data_ptr(), L.ss, L.bs, 0, None]
    torch.cuda.synchronize()
    n0 = api.launches()
    for k in (0, 1, 2, 4, 8):  # d_src, d_dst, d_jobs, d_status, d_scratch
        b = list(a)
        b[k] = None
        assert api.decode(*b) == -12, k
    # scratch below its 32-byte tail, and below what the grid of this launch needs
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    need = min((mixed.jobs.size + 3) // 4, sm * 7) * 4 * simt_stride(mixed.block_size) + 32
    assert need <= L.ss
    for small in (0, 31, 32, need - 8):
        b = list(a)
        b[9] = small
        assert api.decode(*b) == -1, small
    b = list(a)
    b[3] = 0
    assert api.decode(*b) == 0
    torch.cuda.synchronize()
    assert api.launches() == n0
    assert bool((L.status == UNSET).all())
    # plan_frame: max_jobs one short
    fr = zj.golden("multiblock_mixed")[0]
    fb = np.frombuffer(fr, np.uint8)
    nb = api.L.zxc_b200_plan_frame(fb.ctypes.data, fb.size, None, 0, None)
    jobs = np.zeros(nb, zj.JOB_DT)
    assert api.L.zxc_b200_plan_frame(fb.ctypes.data, fb.size, jobs.ctypes.data, nb - 1, None) == -2
    assert api.L.zxc_b200_plan_frame(fb.ctypes.data, fb.size, jobs.ctypes.data, nb, None) == nb


# ---- the unit walk ----------------------------------------------------------------------------------------------
@pytest.mark.skipif(os.environ.get("ZXC_B200_UNITS") == "1", reason="already the unit walk")
def test_unit_walk_layouts_and_guard_bands():
    """The output-centric body (opt-in, ZXC_B200_UNITS=1, read once per process) has its own output alignment
    branch: the layout, gap and short-window tests again in a child process that selects it."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, ZXC_B200_UNITS="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-p", "no:cacheprovider",
                        "-k", "layouts_and_guard_bands or gaps_and_orders or smaller_than_the_block"],
                       cwd=here, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and " passed" in r.stdout, (r.stdout[-3000:], r.stderr[-2000:])
