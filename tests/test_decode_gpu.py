"""GPU parity tests proper: the CUDA decode path, called through the C ABI (libzxc.so.4),
against (a) the reference's conformance vectors, (b) the oracle / the unmodified reference on
seeded synthetic inputs, (c) size-independent properties at larger sizes."""
import ctypes as C
import glob
import json
import os

import numpy as np
import pytest

import zxc_corpus as zc
import zxc_ctypes as z
from test_oracle import CASES, G, GC_DICT, INVALID, VALID, golden_dicts, make_case

pytestmark = pytest.mark.gpu

HUFFMAN_VECTORS = {"glo_pivco_wide_l7", "dict_seekable_l7", "text_64k_level6"}


def frame_uses_huffman(orc, frame):
    rc, st = orc.stats(frame)
    return rc == 0 and st["huf_blocks"] > 0


@pytest.mark.parametrize("name", VALID)
def test_conformance_valid(prod, orc, name):
    frame = open(os.path.join(G, "valid", name + ".zxc"), "rb").read()
    exp = open(os.path.join(G, "valid", name + ".expected"), "rb").read()
    did = int.from_bytes(frame[7:11], "little") if frame[6] & 0x40 else 0
    d, h = golden_dicts().get(did, (None, None))
    r, out = prod.decompress(frame, len(exp), checksum=1, dict=d, dict_huf=h)  # exact-size dst
    assert r == len(exp), z.ERR.get(r, r)
    assert out.tobytes() == exp


@pytest.mark.parametrize("name", sorted(INVALID))
def test_conformance_invalid(prod, name):
    frame = open(os.path.join(G, "invalid", name + ".zxc"), "rb").read()
    ds = prod.lib.zxc_get_decompressed_size(frame, len(frame)) if frame else 0
    cap = ds if 0 < ds <= (1 << 20) else (1 << 20)  # conformance/test_conformance.c:287-297
    out = np.zeros(cap, np.uint8)
    o = z.DecompressOpts(checksum_enabled=1)
    r = prod.lib.zxc_decompress(frame if frame else b"\0", len(frame), out.ctypes.data, cap, C.byref(o))
    assert r == INVALID[name], (name, z.ERR.get(r, r))


def test_golden_format_frames(prod, orc):
    for p in sorted(glob.glob(os.path.join(G, "format", "*.zxc"))):
        frame = open(p, "rb").read()
        n = prod.lib.zxc_get_decompressed_size(frame, len(frame))
        d = GC_DICT if frame[6] & 0x40 else None
        if os.path.basename(p).startswith("12_"):
            continue  # needs the reference trainer's shared table (zxc_train_dict_huf), not a fixture
        r0, o0 = orc.decompress(frame, n, checksum=1, dict=d)
        r1, o1 = prod.decompress(frame, n, checksum=1, dict=d)
        assert r0 == r1 == n, (p, r0, r1)
        assert np.array_equal(o0, o1), p


@pytest.mark.parametrize("kind,n", CASES)
@pytest.mark.parametrize("level", [1, 2, 3, 4, 5, 6, 7])
def test_differential_vs_reference(prod, ref, kind, n, level):
    data = make_case(kind, n)
    for bs, cks, seek in ((4096, 1, 0), (65536, 0, 1), (0, 0, 0), (2 << 20, 1, 1)):
        frame = ref.compress(data, level=level, block_size=bs, checksum=cks, seekable=seek)
        r, out = prod.decompress(frame, data.size, checksum=cks)
        assert r == data.size, (kind, level, bs, z.ERR.get(r, r))
        assert np.array_equal(out, data), (kind, level, bs)


def test_mutation_parity_with_reference(prod, ref):
    data = zc.silesia_shaped(1 << 20, seed=5)[:200000]
    rng = np.random.default_rng(3)
    for level, bs in ((3, 4096), (1, 4096), (5, 65536)):
        frame = ref.compress(data, level=level, block_size=bs, checksum=1, seekable=0)
        same = 0
        trials = 120
        for t in range(trials):
            f = frame.copy()
            pos = int(rng.integers(16, f.size - 12))
            f[pos] ^= int(rng.integers(1, 256))
            cks = t & 1
            r0, o0 = ref.decompress(f, data.size, checksum=cks)
            r1, o1 = prod.decompress(f, data.size, checksum=cks)
            assert (r0 < 0) == (r1 < 0), (level, t, pos, r0, r1)
            if r0 >= 0:
                assert r0 == r1 and np.array_equal(o0, o1)
            same += r0 == r1
        assert same >= trials * 0.9, (level, same)


def test_damaged_block_that_decodes_past_block_size(prod, ref):
    """The reference gives each block block_size + ZXC_DECOMPRESS_TAIL_PAD of room (zxc_dispatch.c:902) and asks about
    the caller's capacity afterwards, so this frame (one extras byte changed: block 1 grows past 64 KiB) is
    DST_TOO_SMALL with an exact buffer and CORRUPT_DATA (footer) with a roomy one."""
    data = zc.silesia_shaped(8 << 20, seed=33)[:300000]
    f = ref.compress(data, level=1, block_size=65536).copy()
    f[90026] = 76
    for cap in (300000, 300000 + 2111, 400000):
        r0, _ = ref.decompress(f, cap)
        r1, _ = prod.decompress(f, cap)
        assert r0 == r1 and r0 < 0, (cap, r0, r1)
    assert ref.decompress(f, 300000)[0] == -2 and ref.decompress(f, 400000)[0] == -8
    rng = np.random.default_rng(11)
    same = trials = 0
    for t in range(60):  # varint-area damage in general: verdicts must agree, not just their sign
        g = ref.compress(data, level=1 + (t % 5), block_size=65536).copy()
        for _ in range(2):
            g[int(rng.integers(16, g.size - 12))] = int(rng.integers(0, 256))
        r0, o0 = ref.decompress(g, 300000)
        r1, o1 = prod.decompress(g, 300000)
        assert (r0 < 0) == (r1 < 0), (t, r0, r1)
        if r0 >= 0:
            assert r0 == r1 and np.array_equal(o0, o1)
        trials += 1
        same += r0 == r1
    assert same >= trials - 3, (same, trials)


def test_capacity_semantics(prod, ref):
    data = zc.silesia_shaped(1 << 20, seed=8)[:300000]
    frame = ref.compress(data, level=3, block_size=65536, seekable=1)
    for cap in (data.size - 1, 65536, 65535, 1):
        r0, _ = ref.decompress(frame, cap)
        r1, _ = prod.decompress(frame, cap)
        assert r0 == r1 == -2, (cap, r0, r1)
    r, out = prod.decompress(frame, data.size + 5000)
    assert r == data.size and np.array_equal(out, data)


def test_seekable_ranges(prod, ref):
    data = zc.silesia_shaped(2 << 20, seed=6)[:1500007]
    for bs, level in ((65536, 3), (4096, 1)):
        frame = ref.compress(data, level=level, block_size=bs, checksum=1, seekable=1)
        fb = frame.tobytes()
        h = prod.lib.zxc_seekable_open(fb, len(fb))
        assert h
        rng = np.random.default_rng(1)
        spans = [(0, data.size), (0, 1), (data.size - 1, 1), (bs - 1, 2), (bs, bs), (12345, 300000)]
        spans += [(int(o), int(min(l, data.size - o))) for o, l in zip(rng.integers(0, data.size - 1, 8), rng.integers(1, 400000, 8))]
        for off, ln in spans:
            out = np.zeros(ln, np.uint8)
            fn = prod.lib.zxc_seekable_decompress_range if (off & 1) else prod.lib.zxc_seekable_decompress_range_mt
            args = (h, out.ctypes.data, ln, off, ln) + (() if (off & 1) else (4,))
            r = fn(*args)
            assert r == ln, (off, ln, z.ERR.get(r, r))
            assert np.array_equal(out, data[off:off + ln]), (off, ln)
        out = np.zeros(16, np.uint8)
        assert prod.lib.zxc_seekable_decompress_range(h, out.ctypes.data, 16, data.size - 8, 16) == -3
        assert prod.lib.zxc_seekable_decompress_range(h, out.ctypes.data, 8, 0, 16) == -2
        assert prod.lib.zxc_seekable_decompress_range(h, out.ctypes.data, 16, 0, 0) == 0
        prod.lib.zxc_seekable_free(h)


def test_dictionary_frames(prod, ref):
    rng = np.random.default_rng(12)
    words = [b"\"user_id\":", b"\"timestamp\":", b"\"status\":\"ok\"", b"\"payload\":{", b"\"region\":\"eu-west\"", b"},{"]
    dict_bytes = b"".join(words[i % len(words)] + b"," for i in range(400))[:16384]
    recs = b"".join(b"{" + b",".join(words[int(k)] + str(int(v)).encode() for k, v in zip(rng.integers(0, 6, 20), rng.integers(0, 1 << 20, 20))) + b"}\n"
                    for _ in range(3000))
    data = np.frombuffer(recs, np.uint8)
    for level, bs in ((5, 4096), (3, 65536), (1, 4096)):
        frame = ref.compress(data, level=level, block_size=bs, seekable=1, dict=dict_bytes)
        assert prod.lib.zxc_get_dict_id(frame.ctypes.data, frame.size) == ref.lib.zxc_dict_id(dict_bytes, len(dict_bytes), None)
        r, out = prod.decompress(frame, data.size, dict=dict_bytes)
        assert r == data.size and np.array_equal(out, data), (level, bs, z.ERR.get(r, r))
        assert prod.decompress(frame, data.size)[0] == -15                      # DICT_REQUIRED
        assert prod.decompress(frame, data.size, dict=dict_bytes[:-1])[0] == -16  # DICT_MISMATCH
        fb = frame.tobytes()
        h = prod.lib.zxc_seekable_open(fb, len(fb))
        out = np.zeros(5000, np.uint8)
        assert prod.lib.zxc_seekable_decompress_range(h, out.ctypes.data, 5000, 7777, 5000) == -15
        assert prod.lib.zxc_seekable_set_dict(h, dict_bytes, len(dict_bytes), None) == 0
        assert prod.lib.zxc_seekable_decompress_range(h, out.ctypes.data, 5000, 7777, 5000) == 5000
        assert np.array_equal(out, data[7777:12777])
        prod.lib.zxc_seekable_free(h)


def test_block_api(prod, ref):
    data = zc.silesia_shaped(1 << 20, seed=9)
    cctx = ref.lib.zxc_create_cctx(None)
    dctx = prod.lib.zxc_create_dctx()
    for n, level, cks in ((4096, 5, 0), (65536, 3, 1), (100000, 1, 0), (700, 3, 1), (1 << 20, 4, 0)):
        src = data[:n]
        cap = int(ref.lib.zxc_compress_block_bound(n))
        blk = np.zeros(cap, np.uint8)
        o = z.CompressOpts(level=level, checksum_enabled=cks)
        r = ref.lib.zxc_compress_block(cctx, src.ctypes.data, n, blk.ctypes.data, cap, C.byref(o))
        assert r > 0
        do = z.DecompressOpts(checksum_enabled=cks)
        out = np.zeros(n, np.uint8)
        for fn in (prod.lib.zxc_decompress_block, prod.lib.zxc_decompress_block_safe):
            out[:] = 0
            rr = fn(dctx, blk.ctypes.data, r, out.ctypes.data, n, C.byref(do))
            assert rr == n, (n, level, z.ERR.get(rr, rr))
            assert np.array_equal(out, src)
        if cks:
            blk[20] ^= 1
            assert prod.lib.zxc_decompress_block(dctx, blk.ctypes.data, r, out.ctypes.data, n, C.byref(do)) == -7
    assert prod.lib.zxc_decompress_block(dctx, None, 10, out.ctypes.data, 10, None) == -12
    prod.lib.zxc_free_dctx(dctx)
    ref.lib.zxc_free_cctx(cctx)


def test_dctx_and_inplace(prod, ref):
    data = zc.silesia_shaped(1 << 20, seed=10)[:777777]
    frame = ref.compress(data, level=3, block_size=65536, checksum=1)
    dctx = prod.lib.zxc_create_dctx()
    out = np.zeros(data.size, np.uint8)
    o = z.DecompressOpts(checksum_enabled=1)
    for _ in range(2):
        assert prod.lib.zxc_decompress_dctx(dctx, frame.ctypes.data, frame.size, out.ctypes.data, out.size, C.byref(o)) == data.size
        assert np.array_equal(out, data)
    prod.lib.zxc_free_dctx(dctx)
    prod.lib.zxc_decompress_inplace_bound.restype = C.c_size_t
    ref.lib.zxc_decompress_inplace_bound.restype = C.c_size_t
    b = prod.lib.zxc_decompress_inplace_bound(frame.ctypes.data, frame.size)
    assert b == ref.lib.zxc_decompress_inplace_bound(frame.ctypes.data, frame.size)
    buf = np.zeros(b, np.uint8)
    buf[b - frame.size:] = frame
    prod.lib.zxc_decompress_inplace.restype = C.c_int64
    prod.lib.zxc_decompress_inplace.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p]
    assert prod.lib.zxc_decompress_inplace(buf.ctypes.data, b, frame.size, C.byref(o)) == data.size
    assert np.array_equal(buf[:data.size], data)


def test_large_roundtrip_properties(prod, ref):
    """256 MiB Silesia-shaped, 64 KiB blocks, level 3: decode == original, through both the frame
    and the seekable entry, and a checksum of block checksums survives erasure of one block."""
    n = 256 << 20
    data = zc.silesia_shaped(n, seed=21)
    frame = zc.compress_ref_mt(ref, data, level=3, block_size=65536, checksum=1)
    r, out = prod.decompress(frame, n, checksum=1)
    assert r == n
    assert np.array_equal(out, data)
    # damage one payload byte in the middle: exactly that block must fail with BAD_CHECKSUM
    f2 = frame.copy()
    f2[f2.size // 2] ^= 0x40
    assert prod.decompress(f2, n, checksum=1)[0] == ref.decompress(f2, n, checksum=1)[0]
    h = prod.lib.zxc_seekable_open(frame.ctypes.data, frame.size)
    part = np.zeros(64 << 20, np.uint8)
    assert prod.lib.zxc_seekable_decompress_range_mt(h, part.ctypes.data, part.size, 100 << 20, part.size, 0) == part.size
    assert np.array_equal(part, data[100 << 20:164 << 20])
    prod.lib.zxc_seekable_free(h)


def test_pinned_pipelined_frame_path(prod, ref):
    """Page-locked caller buffers take the chunked H2D / decode / D2H pipeline (zxg_decode_pipelined)."""
    torch = pytest.importorskip("torch")
    n = 200 << 20
    data = zc.silesia_shaped(n, seed=33)
    frame = zc.compress_ref_mt(ref, data, level=3, block_size=65536, checksum=1)
    h_frame = torch.from_numpy(frame).pin_memory()
    h_out = torch.empty(n, dtype=torch.uint8).pin_memory()
    o = z.DecompressOpts(checksum_enabled=1)
    r = prod.lib.zxc_decompress(h_frame.data_ptr(), h_frame.numel(), h_out.data_ptr(), n, C.byref(o))
    assert r == n
    assert np.array_equal(h_out.numpy(), data)
    # a damaged block in a late chunk is still reported with the reference's code
    f2 = h_frame.clone().pin_memory()
    f2[int(f2.numel() * 0.9)] ^= 0x10
    r0, _ = ref.decompress(f2.numpy(), n, checksum=1)
    assert prod.lib.zxc_decompress(f2.data_ptr(), f2.numel(), h_out.data_ptr(), n, C.byref(o)) == r0 < 0


def test_huffman_sections(prod, ref, orc):
    """PivCo literal (level 6+) and token (level 7) sections, incl. the shared dictionary table."""
    import ctypes as C
    data = zc.silesia_shaped(6 << 20, seed=51, offset=120 << 20)
    for level, bs in ((6, 65536), (7, 65536), (6, 4096), (7, 1 << 20)):
        frame = zc.compress_ref_mt(ref, data, level=level, block_size=bs, checksum=1)
        rc, st = orc.stats(frame)
        assert st["huf_blocks"] > 0
        r, out = prod.decompress(frame, data.size, checksum=1)
        assert r == data.size, z.ERR.get(r, r)
        assert np.array_equal(out, data)
    # mutation parity on a Huffman frame
    small = data[:150000]
    frame = ref.compress(small, level=7, block_size=65536, checksum=0)
    rng = np.random.default_rng(5)
    for t in range(80):
        f = frame.copy()
        pos = int(rng.integers(16, f.size - 12))
        f[pos] ^= int(rng.integers(1, 256))
        r0, o0 = ref.decompress(f, small.size)
        r1, o1 = prod.decompress(f, small.size)
        assert (r0 < 0) == (r1 < 0), (t, pos, r0, r1)
        if r0 >= 0:
            assert r0 == r1 and np.array_equal(o0, o1)


def test_frames_with_short_non_final_blocks(prod, ref):
    """The reference decoder accepts any split into blocks of at most block_size (zxc_dispatch.c:912-1001); its
    encoder never emits one, so the frame is stitched from single-block frames of irregular pieces."""
    import struct
    data = zc.silesia_shaped(1 << 20, seed=21)[:400000]
    bs = 65536
    rng = np.random.default_rng(4)
    for level in (1, 3, 6):
        cuts, p = [], 0
        while p < data.size:
            n = int(rng.integers(1, bs + 1)) if len(cuts) % 3 else bs  # mix of full and short blocks
            cuts.append((p, min(data.size, p + n)))
            p += n
        head, eof, blocks = None, None, []
        for a, b in cuts:
            fr = ref.compress(data[a:b], level=level, block_size=bs).tobytes()
            head, eof = fr[:16], fr[-20:-12]
            blocks.append(fr[16:-20])
        frame = np.frombuffer(head + b"".join(blocks) + eof + struct.pack("<QI", data.size, 0), np.uint8)
        r0, o0 = ref.decompress(frame, data.size)
        assert r0 == data.size and np.array_equal(o0, data), ("reference", level, r0)
        r1, o1 = prod.decompress(frame, data.size)
        assert r1 == data.size, (level, z.ERR.get(r1, r1))
        assert np.array_equal(o1, data), level
        # exact verdicts on capacity: one byte short fails the same way in both
        r0s, _ = ref.decompress(frame, data.size - 1)
        r1s, _ = prod.decompress(frame, data.size - 1)
        assert r0s == r1s, (level, r0s, r1s)


def test_deep_skewed_huffman_table_rank_words(prod, ref, orc):
    """ADVICE r1 (high): a Kraft-complete code with lengths 1,2,...,10,11,11 has eleven bitmap levels, each carrying
    every symbol when the runs are all ones -- 11*n/8 bytes of runs, the worst case for the decoder's rank table
    (one word per 32 run bits per node).  The table is sized for that now; the frame must decode exactly as the
    reference decodes it."""
    import struct
    n = 65536
    tmpl = ref.compress(np.zeros(n, np.uint8), level=3, block_size=n).tobytes()
    head, eof = tmpl[:16], tmpl[-20:-12]
    lens = bytearray(128)
    for s, l in enumerate([1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 11]):
        lens[s >> 1] |= l << (4 * (s & 1))
    runs = bytes([0xFF]) * (11 * (n // 8))
    lit = bytes(lens) + runs
    payload = struct.pack("<IIBBBB", 0, n, 2, 0, 0, 0) + struct.pack("<I", len(lit)) + lit + bytes(32)
    hdr = bytearray(struct.pack("<BBB", 1, 0, 0) + struct.pack("<I", len(payload)) + b"\0")
    hdr[7] = orc.lib.zxo_hash8(bytes(hdr))
    frame = np.frombuffer(head + bytes(hdr) + payload + eof + struct.pack("<QI", n, 0), np.uint8)
    r0, o0 = ref.decompress(frame, n)
    r1, o1 = prod.decompress(frame, n)
    assert r1 == r0, (r0, z.ERR.get(r1, r1))
    if r0 == n:
        assert np.array_equal(o0, o1) and int(o1[0]) == 11 and int(o1.min()) == int(o1.max())


ALT_BODY_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "alt_body.json")

# RECORD = True: the reference library encodes and judges the damaged frames, and what it answered is written to
# ALT_BODY_GOLDEN (tests/golden/make_fixtures.py reference).  RECORD = False: the GPU encoder makes the frames, each
# checked against the reference's sha256, and the GPU decoder must give the reference's verdicts and bytes.
_ALT_BODY = r"""
import sys, json, hashlib, numpy as np
sys.path.insert(0, %r)
GOLDEN, RECORD = %r, %r
import zxc_corpus as zc, zxc_ctypes as z
from test_oracle import CASES, make_case
sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
lib = z.ZxcLib(z.REF_SO if RECORD else z.PRODUCT_SO)
rec = {"frames": [], "damaged": []} if RECORD else json.load(open(GOLDEN))
frames, verdicts = iter(rec["frames"]), iter(rec["damaged"])
def frame(data, level, bs, seekable=0):
    fr = lib.compress(data, level=level, block_size=bs, seekable=seekable)
    assert not isinstance(fr, int), fr
    if RECORD:
        rec["frames"].append(sha(fr))
    else:
        assert sha(fr) == next(frames), ("frame differs from the reference's", level, bs, data.size)
    return fr
n_ok = 0
for kind, n in CASES:
    data = make_case(kind, n)
    for level in (1, 3, 5, 6):
        for bs in (4096, 65536):
            fr = frame(data, level, bs)
            r, out = lib.decompress(fr, data.size)
            assert r == data.size and np.array_equal(out, data), (kind, level, bs, r)
            n_ok += 1
data = zc.silesia_shaped(8 << 20, seed=33)
fr = frame(data, 3, 65536, seekable=1)
r, out = lib.decompress(fr, data.size)
assert r == data.size and np.array_equal(out, data)
rng = np.random.default_rng(2)
for t in range(40):  # damaged frames: same verdict as the reference
    f = frame(data[:300000], 3 if t & 1 else 1, 65536).copy()
    for _ in range(int(rng.integers(1, 4))):
        f[int(rng.integers(16, f.size - 12))] = int(rng.integers(0, 256))
    r1, o1 = lib.decompress(f, 300000)
    if RECORD:
        rec["damaged"].append([int(r1), sha(o1) if r1 > 0 else None])
        continue
    r0, h0 = next(verdicts)
    assert r0 == r1, (t, r0, r1)
    if r0 > 0:
        assert sha(o1) == h0
if RECORD:
    json.dump(rec, open(GOLDEN, "w"))
print("alt-body ok", n_ok)
"""


@pytest.mark.parametrize("env", [{"ZXC_B200_UNITS": "1"}, {"ZXC_B200_DECODE_V2": "1"}], ids=["unit-walk-forced", "block-cooperative"])
def test_alternative_decode_bodies_stay_bit_exact(env):
    """The output-centric body outside its default domain and the block-cooperative kernel (off by default, DESIGN.md
    3c) are selected by environment variables read once per process, so they run in a child process."""
    import subprocess
    import sys
    e = dict(os.environ)
    e.update(env)
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", _ALT_BODY % (here, ALT_BODY_GOLDEN, False)], env=e, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "alt-body ok" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])
