"""CPU tests of the decode kernel's SOURCE under caller-built job tables, the way zxc_b200_decode_blocks receives them
(include/zxc_b200.h): output windows at any byte alignment, gaps between them, rows in any order, windows shorter than
the block, small dictionaries, and per-job verdicts on damaged blocks against the scalar per-block decoder
(zxo_decode_block).  The kernel's decode_job() runs unchanged on the warp emulator of tests/simt/; the bytes around the
windows must come back untouched.  Frames: the conformance vectors always, reference-made frames when oracle/_ref is
built.  tests/test_device_abi_gpu.py runs the same matrix on the device."""
import numpy as np
import pytest

import zxc_corpus as zc
import zxc_jobs as zj
import zxc_simt as zs
from test_oracle import golden_dicts

DST_SHIFTS = (0, 1, 2, 3, 4, 7, 8, 15)
SRC_SHIFTS = (0, 1, 3, 8, 13)


def run(case, jobs, src=None, src_shift=0, dst_shift=0, sentinel=0x5A, units=0, seed=1, verify=None, dict=None,
        dict_huf=None, block_size=None):
    """-> (status, dst, jobs as launched): the source moved up by src_shift, the windows by dst_shift"""
    src = case.src if src is None else src
    s = np.concatenate([np.full(src_shift, 0xEE, np.uint8), src])
    j = jobs.copy()
    j["src_off"] += src_shift
    j["dst_off"] += dst_shift
    end = int((j["dst_off"] + j["dst_cap"]).max()) if j.size else 0
    dst = np.full(end + 80, sentinel, np.uint8)
    st, oob, _ = zs.decode_jobs(s, j, dst, block_size or case.block_size, dict=case.dict if dict is None else dict,
                                dict_huf=case.dict_huf if dict_huf is None else dict_huf,
                                verify=case.verify if verify is None else verify, units=units, seed=seed)
    assert oob == 0, "stores outside the destination buffer"
    return st, dst, j


def ref_frames(ref, levels=(1, 3, 6, 7), n=300000, bs=65536, checksum=0, seed=1):
    data = zj.mixed_input(n, seed=seed)
    return [(ref.compress(data, level=lv, block_size=bs, checksum=checksum), data.tobytes()) for lv in levels]


@pytest.fixture(scope="module")
def golden_mix(prod, orc):
    return zj.Case(prod, [zj.golden(n, orc) for n in zj.GOLDEN_MIX + zj.GOLDEN_FORMAT])


@pytest.fixture(scope="module")
def golden_cks(prod):
    return zj.Case(prod, [zj.golden(n) for n in zj.GOLDEN_CHECKSUM], verify=1)


def _layouts(case, units, seed):
    rng = np.random.default_rng(seed)
    n = 0
    for ds in DST_SHIFTS:
        for ss in rng.choice(SRC_SHIFTS, 2, replace=False):
            st, dst, j = run(case, case.jobs, src_shift=int(ss), dst_shift=ds, units=units, seed=ds + 1)
            n += zj.check(dst, 0, j, st, case.expected(), 0x5A, (ds, int(ss), units))
    return n


@pytest.mark.parametrize("units", [0, 1], ids=["sequence-walk", "unit-walk"])
def test_misaligned_windows_golden(golden_mix, golden_cks, units):
    """every destination shift, each with two source shifts: the 16-byte head / byte tail of ring_flush (al16 false)
    and the unit walk's own alignment branch; the checksum vectors with verify on"""
    assert _layouts(golden_mix, units, 3) > 0
    assert _layouts(golden_cks, units, 4) > 0


@pytest.mark.parametrize("units", [0, 1], ids=["sequence-walk", "unit-walk"])
def test_misaligned_windows_reference_frames(prod, ref, orc, units):
    """GHI (level 1), GLO with RLE literals (3), Huffman literals (6) and tokens (7), RAW blocks, short periods and
    matches longer than the ring, in one table"""
    frames = ref_frames(ref)
    zj.assert_block_kinds(orc, [f for f, _ in frames])
    case = zj.Case(prod, frames)
    _layouts(case, units, 5)


def test_gaps_and_permutations(golden_mix):
    rng = np.random.default_rng(8)
    n = golden_mix.jobs.size
    for gap in (0, 1, 13, 4096 + 5):
        for name, order in (("frame", None), ("reversed", np.arange(n)[::-1]), ("seeded", rng.permutation(n))):
            jobs, ref_off = zj.laid_out(golden_mix.jobs, gap=gap, order=order)
            for units in (0, 1):
                st, dst, j = run(golden_mix, jobs, dst_shift=gap % 7, units=units, seed=gap + 1)
                zj.check(dst, 0, j, st, golden_mix.expected(jobs, ref_off), 0x5A, (gap, name, units))


def test_same_source_twice_and_subsets(prod, golden_mix):
    """one source block decoded to two windows; a block range rebased the way zxc_b200/shard.py slices a frame"""
    from zxc_b200 import shard
    jobs = golden_mix.jobs
    twice = np.concatenate([jobs, jobs])
    lay, ref_off = zj.laid_out(twice, gap=3)
    st, dst, j = run(golden_mix, lay, dst_shift=1)
    zj.check(dst, 0, j, st, golden_mix.expected(lay, ref_off), 0x5A, "twice")
    # one frame of many blocks, sliced by block range and rebased
    fr, exp = zj.golden("multiblock_mixed")
    case = zj.Case(prod, [(fr, exp)])
    comp = case.jobs["src_len"]
    for b0, b1 in ((0, 5), (5, 16), (15, 16), (3, 3)):
        lo, hi, dlo, dhi = shard.rank_slice(comp, case.jobs["dst_cap"][0], len(exp), b0, b1)
        sub = shard.rebase_jobs(case.jobs, b0, b1, lo, dlo)
        if sub.size == 0:
            continue
        st, dst, j = run(case, sub, src=case.src[lo:hi], dst_shift=5)
        want = [(int(c), case.want[dlo + int(o):dlo + int(o) + int(c)]) for c, o in zip(sub["dst_cap"], sub["dst_off"])]
        zj.check(dst, 0, j, st, want, 0x5A, (b0, b1))
        assert sum(st) == dhi - dlo


@pytest.mark.parametrize("units", [0, 1], ids=["sequence-walk", "unit-walk"])
def test_short_windows_against_the_oracle(golden_mix, orc, units):
    """dst_cap below what a block produces: the verdict zxo_decode_block gives at that cap, nothing past the window"""
    jobs = golden_mix.jobs.copy()
    rng = np.random.default_rng(12 + units)
    n = 0
    for k in (1, 7, 16, 17, 4095):
        short = jobs.copy()
        short["dst_cap"] = np.maximum(short["dst_cap"].astype(np.int64) - k, 1).astype(np.uint32)
        lay, _ = zj.laid_out(short, gap=int(rng.integers(0, 20)))
        want = zj.oracle_verdicts(orc, golden_mix.src, lay)
        st, dst, j = run(golden_mix, lay, dst_shift=int(rng.integers(0, 16)), units=units)
        n += zj.check(dst, 0, j, st, want, 0x5A, ("short", k, units))
        assert any(s < 0 for s, _ in want)
    assert n > 0


def _dict_case(prod, ref, size, level, huf):
    d = zc.gen_text(size, seed=size).tobytes()
    data = zj.dict_records(d)
    fr = ref.compress(data, level=level, block_size=4096, dict=d, dict_huf=huf)
    assert not isinstance(fr, int), fr
    return zj.Case(prod, [(fr, data.tobytes())], dict=d, dict_huf=huf), d


def test_small_dictionaries_golden(prod):
    """the conformance dictionary vectors (one with the dictionary's shared Huffman table) at every alignment"""
    dicts = golden_dicts()
    for name in ("dict_http", "dict_seekable_l7"):
        fr, exp = zj.golden(name)
        did = int.from_bytes(fr[7:11], "little")
        d, h = dicts[did]
        case = zj.Case(prod, [(fr, exp)], dict=d, dict_huf=h)
        for ds in DST_SHIFTS:
            for units in (0, 1):
                st, dst, j = run(case, case.jobs, src_shift=ds % 5, dst_shift=ds, units=units)
                zj.check(dst, 0, j, st, case.expected(), 0x5A, (name, ds, units))


DICT_SIZES = (1, 7, 8, 9, 16, 17, 31, 4096, 65535)


@pytest.mark.parametrize("size", DICT_SIZES)
def test_small_dictionaries_reference_frames(prod, ref, size):
    huf = zj.golden_dict_huf()
    for level in (1, 3, 5, 6):
        case, d = _dict_case(prod, ref, size, level, huf if level == 6 else None)
        for ds in (0, 3, 8):
            st, dst, j = run(case, case.jobs, dst_shift=ds, src_shift=ds % 3, units=ds & 1)
            zj.check(dst, 0, j, st, case.expected(), 0x5A, (size, level, ds))


def _damaged(case, orc, trials, seed, verify, per_trial=(1, 4), units=0):
    rng = np.random.default_rng(seed)
    lay, _ = zj.laid_out(case.jobs, gap=5)
    clean = zj.oracle_verdicts(orc, case.src, lay, case.dict, case.dict_huf, verify)
    hit = 0
    for t in range(trials):
        src = zj.damage(case.src, case.jobs, rng, int(rng.integers(*per_trial)))
        want = zj.oracle_verdicts(orc, src, lay, case.dict, case.dict_huf, verify)
        st, dst, j = run(case, lay, src=src, dst_shift=t % 16, verify=verify, units=units, seed=t + 1)
        zj.check(dst, 0, j, st, want, 0x5A, ("damaged", t))
        hit += sum(1 for a, b in zip(want, clean) if a[0] != b[0] or (a[0] >= 0 and not np.array_equal(a[1], b[1])))
    return hit


def test_damaged_blocks_golden(golden_mix, golden_cks, orc):
    """seeded payload damage; every job's status equals zxo_decode_block's, and its bytes where it succeeds"""
    hit = _damaged(golden_mix, orc, 60, 1, 0)
    hit += _damaged(golden_mix, orc, 20, 2, 0, units=1)
    for verify in (0, 1):  # checksummed blocks: damage anywhere including the checksum word, checked or not
        hit += _damaged(golden_cks, orc, 100, 3 + verify, verify)
    assert hit >= 300, hit


def test_damaged_checksum_word(golden_cks, orc):
    """only the trailing checksum damaged: BAD_CHECKSUM with verify, the intact output without"""
    rng = np.random.default_rng(9)
    src = golden_cks.src.copy()
    for j in golden_cks.jobs:
        src[int(j["src_off"]) + int(j["src_len"]) - 1 - int(rng.integers(0, 4))] ^= 0x41
    for verify in (0, 1):
        want = zj.oracle_verdicts(orc, src, golden_cks.jobs, verify=verify)
        assert all((s == -7) == bool(verify) for s, _ in want)
        st, dst, j = run(golden_cks, golden_cks.jobs, src=src, dst_shift=3, verify=verify)
        zj.check(dst, 0, j, st, want, 0x5A, verify)


def test_damaged_blocks_reference_frames(prod, ref, orc):
    """GHI, GLO, RLE, Huffman and dictionary blocks, with and without checksums"""
    hit = 0
    for cks in (0, 1):
        case = zj.Case(prod, ref_frames(ref, n=200000, checksum=cks, seed=7 + cks), verify=cks)
        hit += _damaged(case, orc, 25, 20 + cks, cks, per_trial=(1, 6))
    case, _ = _dict_case(prod, ref, 31, 6, zj.golden_dict_huf())
    hit += _damaged(case, orc, 25, 30, 0)
    case, _ = _dict_case(prod, ref, 4096, 3, None)
    hit += _damaged(case, orc, 25, 31, 0)
    assert hit >= 200, hit
