"""CPU-only: pins the oracle restatement (oracle/zxc_oracle.c) against the reference's own
known-answer vectors (tests/golden/, copied from conformance/ and tests/format/golden/) and,
when oracle/_ref is built, differentially against the unmodified reference library."""
import glob
import json
import os

import numpy as np
import pytest

import zxc_corpus as zc
import zxc_ctypes as z

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GC_DICT = (b"GET /api/v1/users/ HTTP/1.1\r\nHost: api.example.com\r\n"
           b"Accept: application/json\r\nUser-Agent: zxc-client\r\n")  # tests/format/golden_cases.h


def load_zxd(path):
    """minimal .zxd reader (docs/FORMAT.md 12.4): -> (content, huf128, dict_id)"""
    b = open(path, "rb").read()
    n = int.from_bytes(b[6:8], "little")
    return b[16:16 + n], b[16 + n:16 + n + 128], int.from_bytes(b[8:12], "little")


def golden_dicts():
    d = {}
    for p in glob.glob(os.path.join(G, "valid", "*.zxd")):
        c, h, i = load_zxd(p)
        d[i] = (c, h)
    return d


VALID = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(G, "valid", "*.zxc")))
INVALID = json.load(open(os.path.join(G, "invalid", "expected.json")))


def test_fixture_inventory():
    assert len(VALID) == 33 and len(INVALID) == 20  # conformance/ as of reference 0.13.3


@pytest.mark.parametrize("name", VALID)
def test_oracle_conformance_valid(orc, name):
    frame = open(os.path.join(G, "valid", name + ".zxc"), "rb").read()
    exp = open(os.path.join(G, "valid", name + ".expected"), "rb").read()
    did = int.from_bytes(frame[7:11], "little") if frame[6] & 0x40 else 0
    d, h = golden_dicts().get(did, (None, None))
    if d is not None:
        assert orc.dict_id(d, h) == did
    r, out = orc.decompress(frame, len(exp), checksum=1, dict=d, dict_huf=h)  # exact-size buffer
    assert r == len(exp)
    assert out.tobytes() == exp


@pytest.mark.parametrize("name", sorted(INVALID))
def test_oracle_conformance_invalid(orc, name):
    frame = open(os.path.join(G, "invalid", name + ".zxc"), "rb").read()
    cap = 1 << 20
    if len(frame) == 0:
        r = orc.lib.zxo_decompress(b"\0", 0, np.empty(8, np.uint8).ctypes.data, 8, 1, None, 0, None)
    else:
        r, _ = orc.decompress(frame, cap, checksum=1)
    assert r == INVALID[name], (name, z.ERR.get(r))


def test_oracle_golden_format_decode(orc):
    """tests/format/golden/*.zxc decode (inputs are deterministic, tests/format/golden_cases.h)."""
    phrase = (b"the quick brown fox jumps over the lazy dog. ZXC compresses repeated "
              b"patterns efficiently and decompresses them very fast. ")
    text = lambda n: bytes(phrase[i % len(phrase)] for i in range(n))
    fr = lambda n: open(os.path.join(G, "format", n), "rb").read()
    r, o = orc.decompress(fr("01_empty_eof_only.zxc"), 0)
    assert r == 0
    for name in ("03_block_ghi.zxc", "04_block_glo.zxc", "06_checksum_per_block.zxc"):
        r, o = orc.decompress(fr(name), 8192, checksum=1)
        assert r == 8192 and o.tobytes() == text(8192), name
    for name in ("07_multiple_blocks.zxc", "08_seekable_table.zxc"):
        n = 5 * 4096 + 777
        r, o = orc.decompress(fr(name), n, checksum=1)
        assert r == n and o.tobytes() == text(n), name
    req = (b"GET /api/v1/users/4242/profile HTTP/1.1\r\nHost: api.example.com\r\n"
           b"Accept: application/json\r\nUser-Agent: zxc-client\r\n\r\n")
    r, o = orc.decompress(fr("09_block_dict.zxc"), 4096, dict=GC_DICT)
    assert r == 4096 and o.tobytes() == bytes(req[i % len(req)] for i in range(4096))
    # 11_glo_rle: a varying byte then four 0xAA, repeated
    r, o = orc.decompress(fr("11_glo_rle.zxc"), 16384)
    assert r == 16384 and all(o[i] == 0xAA for i in range(16384) if i % 5)
    # Huffman cases decode to the right size with a skewed alphabet
    r, o = orc.decompress(fr("05_block_glo_huffman.zxc"), 16384)
    assert r == 16384 and set(o.tobytes()) <= set(b"abcdefg")
    r, o = orc.decompress(fr("13_glo_huffman_wide.zxc"), 16384)
    assert r == 16384 and int(o.max()) < 220


def dict_id_cases():
    """(n, content, huf128) triples, seeded"""
    rng = np.random.default_rng(7)
    for n in list(range(1, 40)) + [47, 48, 49, 111, 112, 113, 114, 223, 224, 225, 300, 4096, 65537]:
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        huf = rng.integers(0, 256, 128, dtype=np.uint8).tobytes()
        yield n, b, huf


def test_hashes_against_reference(orc):
    """zxc_dict_id of the reference for dict_id_cases(), without and with the Huffman table, is stored in
    tests/golden/reference/dict_ids.json (tests/golden/make_fixtures.py)"""
    want = json.load(open(os.path.join(G, "reference", "dict_ids.json")))
    got = [[n, orc.lib.zxo_dict_id(b, n, None), orc.lib.zxo_dict_id(b, n, huf)] for n, b, huf in dict_id_cases()]
    assert got == want


CASES = [("silesia", 3 << 20), ("text", 300000), ("random", 70000), ("numeric", 200000),
         ("binrec", 150000), ("period1", 100000), ("period7", 100000), ("period300", 90000),
         ("runs", 120000), ("tiny", 1), ("small", 37), ("zeros", 200000)]


def make_case(kind, n):
    if kind == "silesia":
        return zc.silesia_shaped(n, seed=11)
    if kind == "text":
        return zc.gen_text(n)
    if kind == "random":
        return zc.gen_random(n)
    if kind == "numeric":
        return zc.gen_numeric(n)
    if kind == "binrec":
        return zc.gen_binary_records(n)
    if kind.startswith("period"):
        return zc.gen_periodic(n, int(kind[6:]))
    if kind == "runs":
        return zc.gen_runs(n)
    if kind == "zeros":
        return np.zeros(n, np.uint8)
    return zc.gen_text(n, seed=9)


@pytest.mark.parametrize("kind,n", CASES)
@pytest.mark.parametrize("level", [1, 3, 5, 6, 7])
def test_oracle_vs_reference_differential(orc, ref, kind, n, level):
    data = make_case(kind, n)
    for bs, cks in ((4096, 1), (65536, 0), (0, 0)):
        frame = ref.compress(data, level=level, block_size=bs, checksum=cks, seekable=1)
        assert not isinstance(frame, int), frame
        r0, o0 = ref.decompress(frame, data.size, checksum=cks)
        r1, o1 = orc.decompress(frame, data.size, checksum=cks)
        assert r0 == data.size == r1
        assert np.array_equal(o1, data) and np.array_equal(o0, data)


def test_oracle_error_parity_on_mutations(orc, ref):
    """Same verdict class as the reference on randomly damaged frames: both reject or both
    produce identical bytes (exact codes are only contractual for the pinned vectors)."""
    data = zc.silesia_shaped(1 << 20, seed=5)[: 200000]
    frame = ref.compress(data, level=3, block_size=4096, checksum=1, seekable=0)
    rng = np.random.default_rng(3)
    agree = 0
    for t in range(300):
        f = frame.copy()
        pos = int(rng.integers(16, f.size - 12))
        f[pos] ^= int(rng.integers(1, 256))
        r0, o0 = ref.decompress(f, data.size, checksum=1)
        r1, o1 = orc.decompress(f, data.size, checksum=1)
        assert (r0 < 0) == (r1 < 0), (t, pos, r0, r1)
        if r0 >= 0:
            assert r0 == r1 and np.array_equal(o0, o1)
        agree += r0 == r1
    assert agree >= 285  # identical code in the vast majority of cases


def test_stitched_frame_equals_single_call(ref):
    data = zc.silesia_shaped(3 << 20, seed=2)
    a = zc.compress_ref_mt(ref, data, level=3, block_size=65536, checksum=1, slice_bytes=1 << 20)
    b = ref.compress(data, level=3, block_size=65536, checksum=1, seekable=1)
    assert a.size == b.size and np.array_equal(a, b)


def test_corpus_shape(orc, ref):
    """SURVEY 8(d)-2 acceptance: L3 ratio 40-50 %, 2.5k-5k sequences per 64 KiB block."""
    data = zc.silesia_shaped(212 << 20, seed=1)
    frame = zc.compress_ref_mt(ref, data, level=3, block_size=65536)
    ratio = frame.size / data.size
    rc, st = orc.stats(frame)
    assert rc == 0
    assert 0.40 <= ratio <= 0.50, ratio
    assert 2500 <= st["sequences"] / st["blocks"] <= 5000
