"""CPU tests of the decode kernels' SOURCE: zxc_b200/csrc/zxc_decode.cuh (and the headers it includes) compiled
unchanged for the host on the fiber warp emulator of tests/simt/ -- one emulated warp per block runs decode_job()
exactly as zxc_decode_kernel does, with the lanes resumed in a random order between warp-level primitives -- and
compared with the unmodified reference (oracle/_ref) and the conformance vectors.  This is test infrastructure: it
checks the kernels' logic where there is no GPU; the -m gpu tests check the compiled kernels through the C ABI."""
import os

import numpy as np
import pytest

import zxc_corpus as zc
import zxc_ctypes as z
import zxc_simt as zs
from test_oracle import CASES, G, GC_DICT, VALID, golden_dicts, make_case


def _check(prod, frame, want, **kw):
    st, out, oob, _ = zs.decode_frame(prod, frame, **kw)
    assert oob == 0, "stores outside the destination"
    assert all(s >= 0 for s in st), [z.ERR.get(s, s) for s in st if s < 0][:3]
    assert np.array_equal(out, want)


@pytest.mark.parametrize("kind,n", [(k, min(n, 1 << 20)) for k, n in CASES])
@pytest.mark.parametrize("level", [1, 3, 5, 6, 7])
def test_kernel_source_vs_reference(prod, ref, kind, n, level):
    data = make_case(kind, n)
    for bs, cks in ((4096, 1), (65536, 0), (2 << 20, 1)):
        frame = ref.compress(data, level=level, block_size=bs, checksum=cks, seekable=1)
        _check(prod, frame, data, verify=cks, seed=level * 131 + bs)


@pytest.mark.parametrize("name", VALID)
def test_kernel_source_conformance_vectors(prod, name):
    frame = open(os.path.join(G, "valid", name + ".zxc"), "rb").read()
    exp = np.frombuffer(open(os.path.join(G, "valid", name + ".expected"), "rb").read(), np.uint8)
    did = int.from_bytes(frame[7:11], "little") if frame[6] & 0x40 else 0
    d, h = golden_dicts().get(did, (None, None))
    for units in (0, 1):  # sequence-centric body, then the output-centric one (small blocks / dictionaries use it)
        _check(prod, frame, exp, dict=d, dict_huf=h, verify=1, units=units, seed=17 + units)


def test_kernel_source_dictionary_records(prod, ref):
    recs = zc.records(256, record_size=4096, seed=7)
    d = zc.train_dict_ref(ref, recs, record_size=4096, n_samples=128, cap=16384)
    for level in (3, 5):
        frame = ref.compress(recs, level=level, block_size=4096, checksum=0, seekable=1, dict=d)
        for units in (0, 1):
            _check(prod, frame, recs, dict=d, units=units, seed=5)


def test_kernel_source_is_schedule_independent(prod, ref):
    """same bytes whatever order the lanes run in between two warp primitives (seed 0 = lane order)"""
    data = zc.silesia_shaped(1 << 19, seed=21)
    frame = ref.compress(data, level=3, block_size=65536, checksum=0, seekable=1)
    for seed in (0, 1, 2, 3, 99):
        for units in (0, 1):
            _check(prod, frame, data, units=units, seed=seed)


def test_kernel_source_damaged_blocks_fail_like_the_reference(prod, ref):
    """single-byte damage inside block payloads: a block the reference rejects is rejected with the same code by the
    kernel source, a frame the reference still decodes gives the same bytes"""
    data = zc.silesia_shaped(3 * 65536, seed=5)
    rng = np.random.default_rng(11)
    for level in (3, 6):
        frame = ref.compress(data, level=level, block_size=65536, checksum=0, seekable=0)
        fb = bytearray(frame.tobytes())
        body_lo, body_hi = 16 + 8, len(fb) - 12 - 8
        checked = 0
        for _ in range(60):
            pos = int(rng.integers(body_lo, body_hi))
            b = bytearray(fb)
            b[pos] ^= int(rng.integers(1, 256))
            r_ref, out_ref = ref.decompress(bytes(b), data.size)
            try:
                st, out, oob, _ = zs.decode_frame(prod, bytes(b), seed=3)
            except AssertionError:
                continue  # the damage hit a block header: the host walk decides, not the kernel
            assert oob == 0
            if len(st) != 3:
                continue
            bad = [s for s, cap in zip(st, (65536, 65536, 65536)) if s < 0 or s != cap]
            if r_ref == data.size:
                assert not bad and np.array_equal(out, out_ref)
            else:
                assert bad, (pos, "the reference rejects, the kernel source accepts")
                if bad[0] < 0:
                    # a block that outgrows its room is OVERFLOW for the kernel; the host turns it into the reference's
                    # DST_TOO_SMALL where the frame driver would have (zxc_api.c), so the two count as one here
                    room = {-2: -10}
                    assert room.get(bad[0], bad[0]) == room.get(r_ref, r_ref), (pos, z.ERR.get(bad[0], bad[0]), z.ERR.get(r_ref, r_ref))
            checked += 1
        assert checked >= 40


def test_kernel_source_differential_fuzz_smoke(ref):
    """a short fixed-seed run of the open-ended emulator fuzz tools (tests/simt_fuzz.py, tests/simt_fuzz_dict.py);
    both draw their frames and verdicts from the reference library"""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    for tool, secs in (("simt_fuzz.py", "12"), ("simt_fuzz_dict.py", "8")):
        r = subprocess.run([sys.executable, os.path.join(here, tool), "1", secs], stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-1500:]


@pytest.mark.skipif(bool(os.environ.get("ZXC_SIMT_SO")), reason="already running a variant build")
def test_kernel_source_with_bulk_copy_staging():
    """The opt-in TMA flavour of the kernel (token / offset / literal sections staged through shared memory by
    cp.async.bulk, ring flushed by bulk stores: -DZXC_STAGE=1 -DZXC_STAGE_LIT=1 -DZXC_BULK_FLUSH=1) through the same
    tests.  The emulator performs a bulk load when it is issued and a bulk store only when it is waited for, and keeps
    the mbarriers' books: one copy in flight per barrier, every wait on the parity it names, nothing in flight at
    the end of a block."""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    so = os.path.join(here, "simt", "libzxc_simt_decode_staged.so")
    r = subprocess.run(["make", "-s", "SO=" + so, "EXTRA=-DZXC_STAGE=1 -DZXC_STAGE_LIT=1 -DZXC_BULK_FLUSH=1"],
                       cwd=os.path.join(here, "simt"), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    env = dict(os.environ, ZXC_SIMT_SO=so)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider"],
                       env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:]
