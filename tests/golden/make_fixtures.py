#!/usr/bin/env python3
"""Regenerates tests/golden/ from the reference tree (run in the build container only).

Copies the reference's own known-answer DATA (not source):
  * conformance/valid/*.zxc + .expected + .zxd   -> tests/golden/valid/     (decode KAT)
  * conformance/invalid/*.zxc                    -> tests/golden/invalid/   (reject KAT)
    with the pinned error table of conformance/test_conformance.c:228-249
    transcribed to tests/golden/invalid/expected.json
  * tests/format/golden/*.zxc + golden.sha256    -> tests/golden/format/    (encoder KAT)
and generates seeded differential fixtures with the UNMODIFIED reference library
(oracle/_ref/libzxc_ref.so): tests/golden/diff/*.bin (input) + *.zxc (frame).
`make_fixtures.py bench` and `make_fixtures.py reference` record, with that library, what bench.py
(tests/golden/bench/), tests/test_oracle.py and tests/test_decode_gpu.py (tests/golden/reference/) compare with
the reference.
/root/reference does not exist on the GPU box; tests read only tests/golden/.
"""
import json, os, shutil, sys, glob, ctypes
import numpy as np

REF = os.environ.get("ZXC_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))

INVALID = {  # conformance/test_conformance.c:228-249
    "all_0xff_garbage": -4, "bad_block_checksum": -7, "bad_block_size_field": -14,
    "bad_block_type": -13, "bad_checksum_algo": -6, "bad_enc_lit": -8, "bad_eof_compsize": -6,
    "bad_header_crc": -6, "bad_magic": -4, "bad_version": -5, "corrupt_payload": -7,
    "dict_required": -15, "ghi_forged_offset": -9, "glo_forged_enc_off": -8,
    "glo_insufficient_slack": -8, "magic_then_zeros": -5, "too_short_4bytes": -3,
    "truncated_header_only": -3, "truncated_mid_block": -3, "zero_length": -3,
}


def copy_tree(src_glob, dst):
    os.makedirs(dst, exist_ok=True)
    for f in sorted(glob.glob(src_glob)):
        shutil.copy(f, dst)


def main():
    copy_tree(f"{REF}/conformance/valid/*", f"{HERE}/valid")
    copy_tree(f"{REF}/conformance/invalid/*.zxc", f"{HERE}/invalid")
    with open(f"{HERE}/invalid/expected.json", "w") as f:
        json.dump(INVALID, f, indent=1, sort_keys=True)
    copy_tree(f"{REF}/tests/format/golden/*.zxc", f"{HERE}/format")
    with open(f"{REF}/tests/format/golden.sha256") as f, open(f"{HERE}/format/golden.sha256", "w") as g:
        for line in f:
            h, p = line.split()
            g.write(f"{h}  {os.path.basename(p)}\n")
    print("fixtures copied")


def bench_records():
    """What bench.py compares with the reference, so that it runs without the reference library:
    tests/golden/bench/records_dict.bin (the reference trainer's dictionary for the dictionary leg) and
    tests/golden/bench/reference.json (sha256 of the reference's frames for bench.py's default inputs)."""
    import hashlib
    sys.path.insert(0, os.path.dirname(HERE))
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    import bench
    import zxc_corpus as zc
    import zxc_ctypes as z
    ref = z.ZxcLib(z.REF_SO)
    out = os.path.join(HERE, "bench")
    os.makedirs(out, exist_ok=True)
    sha = lambda a: hashlib.sha256(memoryview(np.ascontiguousarray(a))).hexdigest()
    recs = zc.records(bench.DICT_TRAIN_SAMPLES, bench.DICT_REC)  # all the trainer reads
    d = zc.train_dict_ref(ref, recs, bench.DICT_REC)
    with open(os.path.join(out, "records_dict.bin"), "wb") as f:
        f.write(d)
    sub = recs[: bench.DICT_IDENTITY_RECORDS * bench.DICT_REC]
    rec = {"dict_level5": sha(ref.compress(sub, level=5, block_size=bench.DICT_REC, seekable=1, dict=d))}
    del recs, sub
    data = bench.shard_input(bench.DEFAULT_GIB, 0)
    rec[bench.frame_key(bench.DEFAULT_GIB, 0, bench.LEVEL)] = sha(zc.compress_ref_mt(ref, data, level=bench.LEVEL, block_size=bench.BLOCK))
    enc = data[: bench.ENCODE_BYTES]
    for level in (6, bench.LEVEL):
        rec[bench.frame_key(bench.ENCODE_BYTES / (1 << 30), 0, level)] = sha(zc.compress_ref_mt(ref, enc, level=level, block_size=bench.BLOCK))
    with open(os.path.join(out, "reference.json"), "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
    print("bench records written")


def reference_records():
    """tests/golden/reference/dict_ids.json: the reference's zxc_dict_id over test_oracle.dict_id_cases();
    tests/golden/reference/alt_body.json: its frames (sha256) and verdicts in test_decode_gpu's alternative-body test"""
    sys.path.insert(0, os.path.dirname(HERE))
    import zxc_ctypes as z
    from test_oracle import dict_id_cases
    ref = z.ZxcLib(z.REF_SO)
    out = os.path.join(HERE, "reference")
    os.makedirs(out, exist_ok=True)
    ids = [[n, ref.lib.zxc_dict_id(b, n, None), ref.lib.zxc_dict_id(b, n, huf)] for n, b, huf in dict_id_cases()]
    with open(os.path.join(out, "dict_ids.json"), "w") as f:
        json.dump(ids, f)
    import subprocess
    from test_decode_gpu import _ALT_BODY, ALT_BODY_GOLDEN
    subprocess.run([sys.executable, "-c", _ALT_BODY % (os.path.dirname(HERE), ALT_BODY_GOLDEN, True)], check=True)
    print("reference records written")


if __name__ == "__main__":
    if sys.argv[1:] == ["bench"]:
        bench_records()
    elif sys.argv[1:] == ["reference"]:
        reference_records()
    else:
        main()
