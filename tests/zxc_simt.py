"""TEST INFRASTRUCTURE: ctypes binding of tests/simt/libzxc_simt_decode.so -- the product's decode DEVICE code compiled
for the CPU on the fiber warp emulator (tests/simt/).  decode_frame() plans a frame with the product's host code
(zxc_b200_plan_frame, no device needed) and runs decode_job() once per block on an emulated warp; decode_jobs() runs a
caller-built job table the same way."""
import ctypes as C
import os
import subprocess

import numpy as np

import zxc_ctypes as z

HERE = os.path.dirname(os.path.abspath(__file__))
SIMT_DIR = os.path.join(HERE, "simt")
SIMT_SO = os.environ.get("ZXC_SIMT_SO") or os.path.join(SIMT_DIR, "libzxc_simt_decode.so")  # variant builds: make SO=... EXTRA=-D...


class Job(C.Structure):
    _fields_ = [("src_off", C.c_uint64), ("dst_off", C.c_uint64), ("src_len", C.c_uint32), ("dst_cap", C.c_uint32)]


class Info(C.Structure):
    _fields_ = [("decoded_size", C.c_uint64), ("block_size", C.c_uint32), ("n_blocks", C.c_uint32),
                ("dict_id", C.c_uint32), ("has_checksum", C.c_int), ("seekable", C.c_int), ("global_hash", C.c_uint32)]


def build():
    if os.environ.get("ZXC_SIMT_SO"):
        return
    r = subprocess.run(["make", "-s"], cwd=SIMT_DIR, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(SIMT_SO)
        _lib.simt_decode_blocks.restype = C.c_uint64
        _lib.simt_decode_blocks.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p,
                                            C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_uint64,
                                            C.c_void_p]
    return _lib


def decode_frame(prod, frame, dict=None, dict_huf=None, verify=0, units=0, seed=1, max_blocks=None):
    """(per-block status list, decoded bytes ndarray, oob_writes, rendezvous) for the blocks of `frame`."""
    fb = frame.tobytes() if isinstance(frame, np.ndarray) else bytes(frame)
    prod.lib.zxc_b200_plan_frame.restype = C.c_int64
    prod.lib.zxc_b200_plan_frame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    info = Info()
    nb = prod.lib.zxc_b200_plan_frame(fb, len(fb), None, 0, C.byref(info))
    assert nb >= 0, nb
    jobs = (Job * max(nb, 1))()
    assert prod.lib.zxc_b200_plan_frame(fb, len(fb), jobs, nb, None) == nb
    if max_blocks is not None:
        nb = min(nb, max_blocks)
    total = int(jobs[nb - 1].dst_off + jobs[nb - 1].dst_cap) if nb else 0
    out = np.full(max(total, 1), 0x5A, np.uint8)  # a byte no job writes reads back as 0x5A, not as a plausible 0
    status = (C.c_int32 * max(nb, 1))()
    oob = C.c_int(0)
    src = np.frombuffer(fb, np.uint8)
    d = np.frombuffer(dict, np.uint8) if dict else None
    h = np.frombuffer(dict_huf, np.uint8) if dict_huf else None
    rv = lib().simt_decode_blocks(src.ctypes.data, src.size, out.ctypes.data, total, jobs, nb, status,
                                  d.ctypes.data if d is not None else None, d.size if d is not None else 0,
                                  h.ctypes.data if h is not None else None, max(info.block_size, 4096),
                                  1 if (verify and info.has_checksum) else 0, units, seed, C.byref(oob))
    return list(status)[:nb], out[:total], oob.value, rv


def decode_jobs(src, jobs, dst, block_size, dict=None, dict_huf=None, verify=0, units=0, seed=1):
    """Run a caller-built job table (numpy structured array laid out like zxc_b200_job_t) over the source bytes `src`
    into `dst` (uint8 ndarray, updated in place: bytes no job writes keep their value).  -> (per-job status list,
    writes outside dst, rendezvous)"""
    src = np.ascontiguousarray(src, np.uint8)
    jobs = np.ascontiguousarray(jobs)
    assert dst.flags.c_contiguous and dst.dtype == np.uint8
    n = int(jobs.size)
    status = (C.c_int32 * max(n, 1))()
    oob = C.c_int(0)
    d = np.frombuffer(dict, np.uint8) if dict else None
    h = np.frombuffer(dict_huf, np.uint8) if dict_huf is not None else None
    rv = lib().simt_decode_blocks(src.ctypes.data, src.size, dst.ctypes.data, dst.size, jobs.ctypes.data, n, status,
                                  d.ctypes.data if d is not None else None, d.size if d is not None else 0,
                                  h.ctypes.data if h is not None else None, block_size, 1 if verify else 0, units, seed,
                                  C.byref(oob))
    return list(status)[:n], oob.value, rv
