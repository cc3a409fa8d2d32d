#!/usr/bin/env python3
"""bench.py -- ZXC block decode on B200: decompress GB/s (uncompressed bytes) and HBM roofline.

One "step" = one pass of the hot path (decode every block of the shard) over synthetic input.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--gib G] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): seekable ZXC frame, 64 KiB blocks, level 3, over the
Silesia-shaped synthetic corpus (oracle/zxc_corpus.c), G GiB decoded per GPU (default 4; 8 at N = 8 = configs[4]'s 64 GiB).
Frames are produced by this library's GPU encoder, whose frames are byte-identical to the reference
encoder's (BASELINE.md section 3): for the default inputs the frame's sha256 is checked against the reference's
(tests/golden/bench/reference.json) before anything is timed.  At N > 1 every rank owns the contiguous block range [rank*G GiB, (rank+1)*G GiB) of the frame
(weak scaling: independent seekable blocks, no data-path collective).

  value        decode-only, compressed input and output resident in HBM, CUDA events on the
               launching stream, max over ranks; inputs (G GiB + its frame) are far larger than L2.
  e2e          same metric through the reference-facing C ABI call zxc_decompress() with HOST
               (pinned) buffers: H2D of the frame and D2H of the output inside the timed region.
  roofline     algorithmic bytes per launch (C + U: on-disk block bytes read once + decoded bytes
               written once, SURVEY 8(d)) / average launch time, vs MEASURED_PEAKS.json hbm_gbs.
  e2e_pageable the same call with ordinary (pageable) numpy buffers: the library stages them through its own
               NUMA-local pinned bounce buffers and copy pools.
  cpu_baseline the reference's own SIMD CPU path (zxc_seekable_decompress_range_mt, all host
               threads; zxc_decompress 1 thread) on the same frame, same run, rank 0 at N=1; only where
               the reference library was built (oracle/_ref), otherwise reported as not measured.
  dict         (N=1) BASELINE configs[3]: the reference trainer's dictionary (tests/golden/bench/records_dict.bin), 1 Mi x 4 KiB records, level 5, one frame with
               block_size 4096 -- decode-only value + roofline, e2e through zxc_seekable_set_dict +
               zxc_seekable_decompress_range_mt, the reference's CPU figure for the same calls.
  encode       (N=1) BASELINE configs[2]: level 6 over 1 GiB through zxc_compress, frame compared with the reference's.
  pipeline     (N>1) north_star's multi-GPU path from ONE seekable frame held by rank 0 (N x G GiB; 64 GiB at N=8):
               NCCL scatter of compressed block ranges -> decode -> NCCL gather into rank 0, each phase timed on
               the device (max over ranks), output verified on rank 0.
  Every rank binds itself to its GPU's NUMA node before it allocates pinned host memory.
  --impl reference   times only that CPU path, same metric / config (needs oracle/_ref).
  --dump-outputs DIR after the timed steps, rank 0 writes what the last timed step computed as DIR/<name>.npy:
               block_status (per-block result of zxc_b200_decode_blocks), block_sums (per-block byte sums of the
               decoded output) and decoded_sample (decoded bytes at 8 Mi fixed, seeded positions), float64 / float32.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

BLOCK = 65536
LEVEL = 3
DEFAULT_GIB = 4.0
ENCODE_BYTES = 1 << 30  # input of the encode leg: the first GiB of rank 0's shard
DICT_REC = 4096
DICT_RECORDS = 1 << 20
DICT_TRAIN_SAMPLES = 4096  # the stored dictionary was trained on the first 4096 records
DICT_IDENTITY_RECORDS = 2048
DUMP_SAMPLE = 1 << 23
GOLDEN = os.path.join(ROOT, "tests", "golden", "bench")


class Job(C.Structure):
    _fields_ = [("src_off", C.c_uint64), ("dst_off", C.c_uint64), ("src_len", C.c_uint32), ("dst_cap", C.c_uint32)]


class Info(C.Structure):
    _fields_ = [("decoded_size", C.c_uint64), ("block_size", C.c_uint32), ("n_blocks", C.c_uint32),
                ("dict_id", C.c_uint32), ("has_checksum", C.c_int), ("seekable", C.c_int), ("global_hash", C.c_uint32)]


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dram_traffic(decoded_bytes):
    """dram__bytes_read.sum + dram__bytes_write.sum of the decode kernel, per launch: taken from the committed ncu
    capture (profiles/r02_decode_traffic.json, written from the --set full capture named inside it) and scaled to this
    launch's decoded bytes (the capture decodes a shorter frame of the same corpus)."""
    p = os.path.join(ROOT, "profiles", "r02_decode_traffic.json")
    try:
        t = json.load(open(p))
        per_byte = (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["decoded_bytes"]
        return int(per_byte * decoded_bytes), f"profiles/r02_decode_traffic.json <- {t['source']}"
    except Exception:
        return None, "no committed capture"


class ClockSampler:
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md recipe).  NVML is polled
    every 2 ms from a thread (the timed region is ~0.15 s, too short for nvidia-smi's 100 ms loop);
    nvidia-smi is the fallback when the NVML binding is missing."""

    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []  # one (sm_mhz, reasons_bitmask) per sample
        self.max_mhz = None
        self.stop_flag = False
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.lines.append((mhz, mask))
            except Exception:
                pass
            time.sleep(0.002)

    def _pump(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mhz = float(f[0])
                self.max_mhz = float(f[1])
            except ValueError:
                continue
            mask = 0
            for (name, bit), v in zip((("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
                                       ("sw_power_cap", 0x4)), f[3:7]):
                if v.lower().startswith("active"):
                    mask |= bit
            self.lines.append((mhz, mask))

    def stop(self):
        self.stop_flag = True
        if self.nvml is None and not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"]}
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        else:
            self.t.join(timeout=1)
        sm = [m for m, _ in self.lines]
        mask = 0
        for _, k in self.lines:
            mask |= k
        reasons = sorted(name for name, bit in self.REASONS if mask & bit)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def shard_input(gib, rank, seed=1):
    """this rank's slice of the Silesia-shaped stream"""
    import zxc_corpus as zc
    n = int(gib * (1 << 30))
    n -= n % (1 << 20)
    return zc.silesia_shaped(n, seed=seed, offset=rank * n)


def frame_key(gib, rank, level):
    return f"frame_gib{gib:g}_rank{rank}_level{level}"


def sha256(a):
    import hashlib
    return hashlib.sha256(memoryview(np.ascontiguousarray(a))).hexdigest()


def reference_sha(key):
    """sha256 of the reference encoder's frame for `key`, or None when none is stored"""
    return json.load(open(os.path.join(GOLDEN, "reference.json"))).get(key)


def build_shard(lib, gib, rank, on_gpu):
    """(data ndarray, frame ndarray) for this rank's slice; the frame from `lib`'s encoder (one 1 GiB call after the
    other on the GPU, parallel slices on the CPU) stitched into one seekable frame, and checked against the
    reference's frame where its sha256 is stored."""
    import zxc_corpus as zc
    t0 = time.time()
    data = shard_input(gib, rank)
    t1 = time.time()
    kw = {"threads": 1, "slice_bytes": min(1 << 30, data.size)} if on_gpu else {}
    frame = zc.compress_ref_mt(lib, data, level=LEVEL, block_size=BLOCK, checksum=0, **kw)
    t2 = time.time()
    want = reference_sha(frame_key(gib, rank, LEVEL))
    identical = None if want is None else sha256(frame) == want
    assert identical is not False, "the frame differs from the reference encoder's frame"
    return data, frame, {"gen_s": round(t1 - t0, 2), "compress_s": round(t2 - t1, 2),
                         "frame_identical_to_reference": identical}


def load_ref():
    import zxc_ctypes as z
    return z.ZxcLib(z.REF_SO) if z.have_ref() else None


def cpu_reference_decode(ref, frame, n, threads, reps):
    """best-of-reps GB/s of zxc_seekable_decompress_range_mt over the whole frame (output pre-faulted)."""
    out = np.zeros(n, dtype=np.uint8)
    h = ref.lib.zxc_seekable_open(frame.ctypes.data, frame.size)
    assert h
    best = None
    for _ in range(reps):
        t = time.perf_counter()
        r = ref.lib.zxc_seekable_decompress_range_mt(h, out.ctypes.data, n, 0, n, threads)
        dt = time.perf_counter() - t
        assert r == n, r
        best = dt if best is None or dt < best else best
    ref.lib.zxc_seekable_free(h)
    return n / best / 1e9, out

def bind_to_gpu_numa(index):
    """Pin this process (and the pinned host buffers it allocates next) to the NUMA node of GPU `index`:
    /sys/bus/pci/devices/<bdf>/numa_node -> that node's cpulist.  On the 8-GPU hosts GPUs 0-3 hang off node 0 and
    4-7 off node 1; unbound ranks put every pinned buffer on one node and the 8-rank e2e collapses (round 1)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return {"node": None, "bdf": bdf}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"node": node, "bdf": bdf, "cpus": len(allowed)}
    except Exception as e:  # noqa: BLE001
        return {"node": None, "error": repr(e)}


def pipeline_leg(lib, dist, dev, stream, rank, world, frame, jv, data, steps, block):
    """north_star's multi-GPU data path from ONE seekable frame held by rank 0 (SURVEY 8(e), zxc_seekable.c:999-1108):
    partition by the SEK prefix sums (balanced compressed bytes) -> NCCL scatter of compressed block ranges ->
    per-rank decode of the rebased job table -> NCCL gather of decoded ranges into rank 0 (which decodes its own
    range straight into the gather buffer).  Every phase is timed on the device, max over ranks."""
    import torch
    from zxc_b200 import shard
    n = data.size
    # ---- untimed: assemble the frame on rank 0's GPU from the per-rank slices (bodies back to back)
    body_lo = int(jv["src_off"][0])
    body_hi = int(jv["src_off"][-1]) + int(jv["src_len"][-1])
    sizes = torch.tensor([body_hi - body_lo, len(jv)], dtype=torch.int64, device=dev)
    all_sizes = [torch.zeros_like(sizes) for _ in range(world)]
    dist.all_gather(all_sizes, sizes)
    body_sizes = [int(t[0]) for t in all_sizes]
    nblocks = [int(t[1]) for t in all_sizes]
    assert len(set(nblocks)) == 1
    nbr = nblocks[0]
    comp_local = torch.from_numpy(jv["src_len"].astype(np.int64)).to(dev)
    comp_all = torch.empty(world * nbr, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(comp_all, comp_local)
    comp_all = comp_all.cpu().numpy()
    body_off = np.concatenate([[0], np.cumsum(body_sizes)])
    total = n * world
    d_body = torch.from_numpy(frame[body_lo:body_hi]).to(dev)
    d_frame = torch.empty(16 + int(body_off[-1]), dtype=torch.uint8, device=dev) if rank == 0 else None
    if rank == 0:
        d_frame[:16].copy_(torch.from_numpy(frame[:16]).to(dev))
    shard.gather_ranges_p2p(d_body, d_frame, [(16 + int(body_off[r]), 16 + int(body_off[r + 1])) for r in range(world)], dist)
    if rank == 0:
        d_frame[16:16 + body_sizes[0]].copy_(d_body)
    del d_body
    # ---- the partition every rank derives from the block table
    parts = shard.partition_blocks(comp_all, world)
    src_rng, dst_rng = [], []
    for (b0, b1) in parts:
        lo, hi, dlo, dhi = shard.rank_slice(comp_all, block, total, b0, b1)
        src_rng.append((lo, hi))
        dst_rng.append((dlo, dhi))
    b0, b1 = parts[rank]
    lo, hi = src_rng[rank]
    dlo, dhi = dst_rng[rank]
    nb = b1 - b0
    jobs = np.zeros(nb, dtype=np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("src_len", "<u4"), ("dst_cap", "<u4")]))
    offs = 16 + np.concatenate([[0], np.cumsum(comp_all)])
    jobs["src_off"] = offs[b0:b1] - lo
    jobs["src_len"] = comp_all[b0:b1]
    jobs["dst_off"] = (np.arange(b0, b1, dtype=np.int64) * block) - dlo
    jobs["dst_cap"] = np.minimum(block, total - np.arange(b0, b1, dtype=np.int64) * block)
    d_jobs = torch.from_numpy(jobs.view(np.uint8)).to(dev)
    d_status = torch.empty(nb, dtype=torch.int32, device=dev)
    ss = lib.zxc_b200_decode_scratch_size(block)
    d_scr = torch.empty(ss, dtype=torch.uint8, device=dev)
    d_all = torch.empty(total, dtype=torch.uint8, device=dev) if rank == 0 else None
    d_out = d_all[dlo:dhi] if rank == 0 else torch.empty(dhi - dlo, dtype=torch.uint8, device=dev)

    def run_once(ev):
        ev[0].record(stream)
        mine = shard.scatter_ranges_p2p(d_frame, src_rng, dist, dev)
        ev[1].record(stream)
        rc = lib.zxc_b200_decode_blocks(mine.data_ptr(), d_out.data_ptr(), d_jobs.data_ptr(), nb, d_status.data_ptr(),
                                        None, 0, None, d_scr.data_ptr(), ss, block, 0, stream.cuda_stream)
        assert rc == 0, rc
        ev[2].record(stream)
        shard.gather_ranges_p2p(d_out, d_all, dst_rng, dist)
        ev[3].record(stream)
        return mine
    mk = lambda: [torch.cuda.Event(enable_timing=True) for _ in range(4)]  # noqa: E731
    for _ in range(2):
        run_once(mk())
    torch.cuda.synchronize(dev)
    assert lib.zxc_b200_reduce_status(d_status.data_ptr(), d_jobs.data_ptr(), nb, stream.cuda_stream) == dhi - dlo
    # verify on rank 0: per-MiB wrapping sums of the gathered output against every rank's original slice
    def sums(t):
        return t.view(torch.int64).view(-1, 131072).sum(dim=1)
    mine_sums = sums(torch.from_numpy(data).to(dev))
    all_sums = torch.empty(world * mine_sums.numel(), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(all_sums, mine_sums)
    ok = True
    if rank == 0:
        ok = bool(torch.equal(sums(d_all), all_sums))
    del mine_sums, all_sums
    dist.barrier()
    acc = np.zeros(4)
    for _ in range(steps):
        ev = mk()
        dist.barrier()
        torch.cuda.synchronize(dev)
        run_once(ev)
        torch.cuda.synchronize(dev)
        acc += [ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]), ev[0].elapsed_time(ev[3])]
    t = torch.tensor(acc / steps, dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sc, de, ga, tot = [float(x) for x in t.tolist()]
    frame_bytes = int(offs[-1])
    return {"frame": f"one seekable frame, {total / 2**30:g} GiB decoded / {frame_bytes / 2**30:.2f} GiB on disk, held by rank 0",
            "partition": "contiguous block ranges balanced by compressed bytes (SEK prefix sums)",
            "scatter_ms": round(sc, 3), "decode_ms": round(de, 3), "gather_ms": round(ga, 3), "total_ms": round(tot, 3),
            "gbs_decode_only": round(total / (de * 1e-3) / 1e9, 1), "gbs_with_exchange": round(total / (tot * 1e-3) / 1e9, 1),
            "scatter_gbs_out_of_root": round((frame_bytes - (src_rng[0][1] - src_rng[0][0])) / (sc * 1e-3) / 1e9, 1),
            "gather_gbs_into_root": round((total - (dst_rng[0][1] - dst_rng[0][0])) / (ga * 1e-3) / 1e9, 1),
            "nvlink_peer_copy_ref_gbs": 770.0, "collective": "NCCL grouped ncclSend/ncclRecv (batch_isend_irecv), 1 GiB messages",
            "verified_on_rank0": ok, "steps": steps}


def dict_leg(lib, prod, ref, dev, stream, threads, n_records, steps, peak):
    """BASELINE.json configs[3]: 16 KiB dictionary (the reference's trainer over the first 4096 records, stored in
    tests/golden/bench/records_dict.bin), n x 4 KiB records, level 5, one seekable frame with block_size 4096.
    value = decode-only from HBM; e2e = zxc_seekable_set_dict + zxc_seekable_decompress_range_mt of THIS library
    with host buffers; cpu = the same two calls of the reference, where it was built."""
    import torch
    import zxc_corpus as zc
    REC = DICT_REC
    assert n_records >= DICT_TRAIN_SAMPLES, f"--dict-records must be at least {DICT_TRAIN_SAMPLES}"
    data = zc.records(n_records, REC)
    dict_bytes = open(os.path.join(GOLDEN, "records_dict.bin"), "rb").read()
    dsz = len(dict_bytes)
    frame = prod.compress(data, level=5, block_size=REC, seekable=1, dict=dict_bytes)  # GPU encoder
    assert not isinstance(frame, int), frame
    sub = data[: DICT_IDENTITY_RECORDS * REC]
    identical = sha256(prod.compress(sub, level=5, block_size=REC, seekable=1, dict=dict_bytes)) == reference_sha("dict_level5")
    n = data.size
    nb = lib.zxc_b200_plan_frame(frame.ctypes.data, frame.size, None, 0, None)
    jobs = np.zeros(nb * C.sizeof(Job), dtype=np.uint8)
    assert lib.zxc_b200_plan_frame(frame.ctypes.data, frame.size, jobs.ctypes.data, nb, None) == nb == n_records
    jv = jobs.view(np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("src_len", "<u4"), ("dst_cap", "<u4")]))
    comp_bytes = int(jv["src_len"].astype(np.int64).sum())
    d_src = torch.from_numpy(frame).to(dev)
    d_dst = torch.empty(n, dtype=torch.uint8, device=dev)
    d_jobs = torch.from_numpy(jobs).to(dev)
    d_status = torch.empty(nb, dtype=torch.int32, device=dev)
    d_dict = torch.from_numpy(np.frombuffer(dict_bytes, np.uint8).copy()).to(dev)
    ss = lib.zxc_b200_decode_scratch_size(REC)
    d_scr = torch.empty(ss, dtype=torch.uint8, device=dev)

    def step():
        rc = lib.zxc_b200_decode_blocks(d_src.data_ptr(), d_dst.data_ptr(), d_jobs.data_ptr(), nb, d_status.data_ptr(),
                                        d_dict.data_ptr(), dsz, None, d_scr.data_ptr(), ss, REC, 0, stream.cuda_stream)
        assert rc == 0, rc
    for _ in range(3):
        step()
    torch.cuda.synchronize(dev)
    assert lib.zxc_b200_reduce_status(d_status.data_ptr(), d_jobs.data_ptr(), nb, stream.cuda_stream) == n
    assert np.array_equal(d_dst.cpu().numpy(), data), "dict leg: decoded records differ"
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    del d_src, d_dst, d_scr
    # e2e through the seekable API (host buffers, pinned)
    h_frame = torch.from_numpy(frame).pin_memory()
    h_out = torch.empty(n, dtype=torch.uint8).pin_memory()

    def seek_run(L, fptr, flen, optr, reps):
        h = L.zxc_seekable_open(fptr, flen)
        assert h
        assert L.zxc_seekable_set_dict(h, dict_bytes, dsz, None) == 0
        best = None
        for _ in range(reps):
            t = time.perf_counter()
            r = L.zxc_seekable_decompress_range_mt(h, optr, n, 0, n, threads)
            dt = time.perf_counter() - t
            assert r == n, r
            best = dt if best is None or dt < best else best
        L.zxc_seekable_free(h)
        return n / best / 1e9
    e2e = seek_run(prod.lib, h_frame.data_ptr(), h_frame.numel(), h_out.data_ptr(), 3)
    assert np.array_equal(h_out.numpy(), data), "dict leg: e2e output differs"
    cpu = None
    if ref is not None:
        out = np.zeros(n, dtype=np.uint8)
        cpu = round(seek_run(ref.lib, frame.ctypes.data, frame.size, out.ctypes.data, 3), 3)
        assert np.array_equal(out, data)
    achieved = (comp_bytes + n) / (ms * 1e-3) / 1e9
    return {"workload": f"zxc_dict decode: {dsz} B dictionary (reference trainer), {n_records} x 4 KiB records, level 5, "
                        "block_size 4096, one seekable frame",
            "value": round(n / (ms * 1e-3) / 1e9, 2), "unit": "GB/s", "ms_per_step": round(ms, 4), "steps": steps,
            "blocks": int(nb), "ratio": round(frame.size / n, 4), "encoder_identical_to_reference": identical,
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "algorithmic_bytes_per_launch": comp_bytes + n,
                         "note": "C + U per record; the dictionary is read once per SM and excluded (SURVEY 8(d))"},
            "e2e": {"value": round(e2e, 2), "unit": "GB/s", "h2d_bytes_per_step": int(frame.size), "d2h_bytes_per_step": int(n),
                    "api": "zxc_seekable_open + zxc_seekable_set_dict + zxc_seekable_decompress_range_mt, pinned host buffers"},
            "cpu_baseline": {"value": cpu, "unit": "GB/s", "cores": threads, "kind": "reference",
                             "sample": "the same frame, zxc_seekable_set_dict + zxc_seekable_decompress_range_mt, best of 3"
                                       if cpu is not None else "not measured: reference library not built (oracle/_ref)"}}


def dump_outputs(out_dir, d_dst, d_status):
    """what the last timed step left in HBM: the per-block verdicts, per-block byte sums of the decoded output and the
    decoded bytes at DUMP_SAMPLE positions drawn with a fixed seed (the whole output is GiBs)"""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = d_dst.numel()
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    sample = d_dst[torch.from_numpy(idx).to(d_dst.device)].cpu().numpy()
    np.save(os.path.join(out_dir, "decoded_sample.npy"), sample.astype(np.float32))
    nfull = n - n % BLOCK
    sums = d_dst[:nfull].view(-1, BLOCK).sum(dim=1, dtype=torch.int64).cpu().numpy()
    if nfull < n:
        sums = np.append(sums, int(d_dst[nfull:].sum(dtype=torch.int64)))
    np.save(os.path.join(out_dir, "block_sums.npy"), sums.astype(np.float64))
    np.save(os.path.join(out_dir, "block_status.npy"), d_status.cpu().numpy().astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gib", type=float, default=0.0, help="decoded GiB per GPU (default: 4 = configs[1]; 8 at N = 8 so that the eight "
                    "GPUs hold configs[4]'s 64 GiB frame)")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--decode-only", action="store_true", help="development: skip the cpu_baseline, dict and encode legs")
    ap.add_argument("--dict-records", type=int, default=DICT_RECORDS, help="records of the configs[3] dictionary leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gib <= 0:
        args.gib = 8.0 if world >= 8 else DEFAULT_GIB
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import zxc_corpus as zc
    import zxc_ctypes as z

    ref = load_ref()
    threads = zc.host_threads()
    config = {"workload": f"seekable decode, {args.gib:g} GiB/GPU Silesia-shaped synthetic, 64 KiB blocks, level 3",
              "block_size": BLOCK, "level": LEVEL, "gib_per_gpu": args.gib, "sharding": f"block-range x{world}",
              "l2_policy": "inputs (frame + output) >> 126 MB L2, no flush needed"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        if ref is None:
            raise SystemExit("--impl reference needs oracle/_ref/libzxc_ref.so: build() compiles it where the reference sources are")
        data, frame, prep = build_shard(ref, args.gib, 0, on_gpu=False)
        n = data.size
        out = np.zeros(n, dtype=np.uint8)
        h = ref.lib.zxc_seekable_open(frame.ctypes.data, frame.size)
        for _ in range(args.warmup):
            ref.lib.zxc_seekable_decompress_range_mt(h, out.ctypes.data, n, 0, n, threads)
        t = time.perf_counter()
        for _ in range(args.steps):
            r = ref.lib.zxc_seekable_decompress_range_mt(h, out.ctypes.data, n, 0, n, threads)
            assert r == n
        dt = (time.perf_counter() - t) / args.steps
        ref.lib.zxc_seekable_free(h)
        assert np.array_equal(out, data)
        gbs = n / dt / 1e9
        line = {"impl": "reference", "metric": "decompress GB/s (uncompressed)", "value": round(gbs, 3), "unit": "GB/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": round(gbs, 3), "unit": "GB/s", "cores": threads, "kind": "reference",
                                 "sample": f"whole {args.gib:g} GiB frame per step, zxc_seekable_decompress_range_mt, {threads} threads"},
                "e2e": {"value": round(gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "prep": prep}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    lib = C.CDLL(z.PRODUCT_SO)  # fails loudly if the CUDA library is missing
    prod = z.ZxcLib(z.PRODUCT_SO)
    lib.zxc_b200_plan_frame.restype = C.c_int64
    lib.zxc_b200_plan_frame.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.zxc_b200_decode_scratch_size.restype = C.c_size_t
    lib.zxc_b200_decode_scratch_size.argtypes = [C.c_uint32]
    lib.zxc_b200_decode_blocks.restype = C.c_int
    lib.zxc_b200_decode_blocks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                           C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, C.c_void_p]
    lib.zxc_b200_reduce_status.restype = C.c_int64
    lib.zxc_b200_reduce_status.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    lib.zxc_b200_launch_count.restype = C.c_uint64

    data, frame, prep = build_shard(prod, args.gib, rank, on_gpu=True)
    n = data.size
    info = Info()
    nb = lib.zxc_b200_plan_frame(frame.ctypes.data, frame.size, None, 0, C.byref(info))
    assert nb > 0 and info.decoded_size == n, (nb, info.decoded_size)
    jobs = np.zeros(nb * C.sizeof(Job), dtype=np.uint8)
    assert lib.zxc_b200_plan_frame(frame.ctypes.data, frame.size, jobs.ctypes.data, nb, None) == nb
    jv = jobs.view(np.dtype([("src_off", "<u8"), ("dst_off", "<u8"), ("src_len", "<u4"), ("dst_cap", "<u4")]))
    comp_bytes = int(jv["src_len"].astype(np.int64).sum())
    algo_bytes = comp_bytes + n  # C + U per launch

    h_frame = torch.from_numpy(frame).pin_memory()
    d_src = h_frame.to(dev, non_blocking=True)
    d_dst = torch.empty(n, dtype=torch.uint8, device=dev)
    d_jobs = torch.from_numpy(jobs).to(dev)
    d_status = torch.empty(nb, dtype=torch.int32, device=dev)
    scratch_size = lib.zxc_b200_decode_scratch_size(BLOCK)
    d_scratch = torch.empty(scratch_size, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step():
        rc = lib.zxc_b200_decode_blocks(d_src.data_ptr(), d_dst.data_ptr(), d_jobs.data_ptr(), nb, d_status.data_ptr(),
                                        None, 0, None, d_scratch.data_ptr(), scratch_size, BLOCK, 0, stream.cuda_stream)
        assert rc == 0, rc

    sampler = ClockSampler(local_rank)
    sampler.start()  # nvidia-smi takes ~0.5 s to deliver its first line: start it ahead of the warm-up
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize(dev)
    total = lib.zxc_b200_reduce_status(d_status.data_ptr(), d_jobs.data_ptr(), nb, stream.cuda_stream)
    assert total == n, f"decode verdict {total} != {n}"
    if not args.no_verify:
        got = d_dst.cpu().numpy()
        assert np.array_equal(got, data), "decoded bytes differ from the original"
        del got

    t_wait = time.time()
    while len(sampler.lines) < 2 and time.time() - t_wait < 3.0:
        step()  # keep the GPU under load until the sampler is live (untimed)
        torch.cuda.synchronize(dev)
    sampler.lines.clear()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    launches0 = lib.zxc_b200_launch_count()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    evs[0].record(stream)
    for i in range(args.steps):
        step()
        evs[i + 1].record(stream)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    launches = int(lib.zxc_b200_launch_count() - launches0)
    total_ms = evs[0].elapsed_time(evs[-1])
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_dst, d_status)

    t_ms = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(t_ms.item()) / args.steps
    value = (n * world) / (ms_per_step * 1e-3) / 1e9

    # ---- e2e through the C ABI with host (pinned) buffers: H2D + decode + D2H every step
    h_out = torch.empty(n, dtype=torch.uint8).pin_memory()
    e2e_steps = args.steps
    for _ in range(2):
        r = prod.lib.zxc_decompress(h_frame.data_ptr(), h_frame.numel(), h_out.data_ptr(), n, None)
        assert r == n, r
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r = prod.lib.zxc_decompress(h_frame.data_ptr(), h_frame.numel(), h_out.data_ptr(), n, None)
    torch.cuda.synchronize(dev)
    e2e_dt = (time.perf_counter() - t0) / e2e_steps
    assert r == n
    if not args.no_verify:
        assert np.array_equal(h_out.numpy(), data), "e2e output differs"
    t_e = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = (n * world) / float(t_e.item()) / 1e9

    # ---- the same call with ordinary (pageable) numpy buffers: what an existing libzxc caller passes in
    del h_out  # 4-8 GiB of pinned memory per rank: give it back before the pageable buffer is touched
    p_out = np.zeros(n, dtype=np.uint8)  # pre-faulted
    r = prod.lib.zxc_decompress(frame.ctypes.data, frame.size, p_out.ctypes.data, n, None)
    assert r == n, r
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = prod.lib.zxc_decompress(frame.ctypes.data, frame.size, p_out.ctypes.data, n, None)
    pg_dt = (time.perf_counter() - t0) / args.steps
    assert r == n
    if not args.no_verify:
        assert np.array_equal(p_out, data), "pageable e2e output differs"
    del p_out
    t_p = torch.tensor([pg_dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_p, op=dist.ReduceOp.MAX)
    e2e_pageable = (n * world) / float(t_p.item()) / 1e9

    # ---- supplementary (N > 1): ONE zxc_decompress call on rank 0 fanned out over all N devices by the library itself
    # (ZXC_B200_DEVICES, zxc_api.c decode_multi) -- what a single-process caller of the drop-in gets from the box;
    # the other ranks idle at the barrier meanwhile
    one_call = None
    if world > 1:
        # the waiting ranks poll a flag file instead of sitting in an NCCL barrier kernel on the GPUs rank 0 is using
        flag = "/tmp/zxc_bench_one_call_%s.done" % os.environ.get("MASTER_PORT", "0")
        if rank == 0 and os.path.exists(flag):
            os.unlink(flag)
        dist.barrier()
        torch.cuda.synchronize(dev)
        if rank == 0:
            mine = os.sched_getaffinity(0)
            os.sched_setaffinity(0, all_cpus)  # the stripes' copy pools bind themselves to their own device's node
            os.environ["ZXC_B200_DEVICES"] = str(world)
            try:
                h_out = torch.empty(n, dtype=torch.uint8).pin_memory()
                p_out = np.zeros(n, dtype=np.uint8)
                rates = {}
                for name, src_p, src_n, dst_p in (("page_locked", h_frame.data_ptr(), h_frame.numel(), h_out.data_ptr()),
                                                  ("pageable", frame.ctypes.data, frame.size, p_out.ctypes.data)):
                    for _ in range(2):
                        r = prod.lib.zxc_decompress(src_p, src_n, dst_p, n, None)
                        assert r == n, r
                    t0 = time.perf_counter()
                    for _ in range(3):
                        r = prod.lib.zxc_decompress(src_p, src_n, dst_p, n, None)
                    rates[name] = n / ((time.perf_counter() - t0) / 3) / 1e9
                    assert r == n
                if not args.no_verify:
                    assert np.array_equal(h_out.numpy(), data) and np.array_equal(p_out, data), "one-call output differs"
                one_call = {"devices": world, "decoded_bytes": int(n), "unit": "GB/s",
                            "page_locked": round(rates["page_locked"], 2), "pageable": round(rates["pageable"], 2),
                            "api": "one zxc_decompress(host frame, host dst) call on rank 0, ZXC_B200_DEVICES=%d: block stripes "
                                   "fork-joined over the devices inside the library" % world}
                del h_out, p_out
            finally:
                del os.environ["ZXC_B200_DEVICES"]
                os.sched_setaffinity(0, mine)
                open(flag, "w").close()
        else:
            t_wait = time.perf_counter()
            while not os.path.exists(flag) and time.perf_counter() - t_wait < 600:
                time.sleep(0.05)
        dist.barrier()
        if rank == 0:
            os.unlink(flag)

    # ---- supplementary: NVLink gather of decoded output (N > 1), bounded slice
    gather = None
    if world > 1:
        sl = min(n, 1 << 30)
        outs = torch.empty(sl * world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(outs, d_dst[:sl])
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        e0.record()
        for _ in range(3):
            dist.all_gather_into_tensor(outs, d_dst[:sl])
        e1.record()
        torch.cuda.synchronize(dev)
        g_ms = torch.tensor([e0.elapsed_time(e1) / 3], dtype=torch.float64, device=dev)
        dist.all_reduce(g_ms, op=dist.ReduceOp.MAX)
        gather = {"collective": "nccl all_gather of decoded ranges", "bytes_per_rank": sl,
                  "gbs_per_rank_in": round(sl * (world - 1) / (float(g_ms.item()) * 1e-3) / 1e9, 1)}
        del outs
    pipeline = None
    if world > 1:
        del d_scratch
        torch.cuda.empty_cache()
        pipeline = pipeline_leg(lib, dist, dev, stream, rank, world, frame, jv, data, args.steps, BLOCK)

    if rank == 0:
        peak, peak_src = measured_peak()
        traffic, traffic_src = dram_traffic(n)
        avg_launch_ms = float(np.mean(per_launch_ms))
        achieved = algo_bytes / (avg_launch_ms * 1e-3) / 1e9
        line = {"metric": "decompress GB/s (uncompressed)", "value": round(value, 2), "unit": "GB/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config,
                "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                             "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                             "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": algo_bytes, "compressed_bytes": comp_bytes,
                             "decoded_bytes": n, "kernel": "zxc_decode_kernel<false,false> (sequence-centric body)",
                             "avg_launch_ms": round(avg_launch_ms, 4),
                             "decoded_only_frac": round((n / (avg_launch_ms * 1e-3) / 1e9) / peak, 4)},
                "e2e": {"value": round(e2e_value, 2), "unit": "GB/s", "h2d_bytes_per_step": int(frame.size),
                        "d2h_bytes_per_step": int(n), "api": "zxc_decompress(host frame, host dst), pinned host buffers",
                        "steps": e2e_steps},
                "e2e_pageable": {"value": round(e2e_pageable, 2), "unit": "GB/s",
                                 "api": "zxc_decompress(host frame, host dst), ordinary pageable buffers (staged through the "
                                        "library's NUMA-local pinned bounce buffers and copy pool)"},
                "gpu_launches": launches, "clocks": clocks, "ratio": round(frame.size / n, 4), "blocks_per_gpu": int(nb),
                "prep": prep}
        if gather:
            line["gather"] = gather
        if pipeline:
            line["pipeline"] = pipeline
        if one_call:
            line["e2e_one_call"] = one_call
        line["numa"] = numa
        if world == 1 and not args.decode_only:
            os.sched_setaffinity(0, all_cpus)  # the CPU baseline may use every host core again
            threads = zc.host_threads()
            reps = 3
            if ref is not None:
                mt, out = cpu_reference_decode(ref, frame, n, threads, reps)
                sample_n = min(n, 256 << 20)
                sf = zc.compress_ref_mt(ref, data[:sample_n], level=LEVEL, block_size=BLOCK)
                o1 = np.zeros(sample_n, dtype=np.uint8)
                t = time.perf_counter()
                r1 = ref.lib.zxc_decompress(sf.ctypes.data, sf.size, o1.ctypes.data, sample_n, None)
                st = sample_n / (time.perf_counter() - t) / 1e9
                assert r1 == sample_n
                line["cpu_baseline"] = {"value": round(mt, 3), "unit": "GB/s", "cores": threads, "kind": "reference",
                                        "sample": f"whole {args.gib:g} GiB frame, zxc_seekable_decompress_range_mt best of {reps}",
                                        "single_thread_gbs": round(st, 3)}
            else:
                line["cpu_baseline"] = {"value": None, "unit": "GB/s", "kind": "reference",
                                        "sample": "not measured: reference library not built (oracle/_ref)"}
            # ---- supplementary: the encoder, BASELINE.json configs[2] (level 6, 1 GiB, frame bit-exact vs the
            # reference) and the same input at level 3; through zxc_compress with host buffers
            enc_n = min(n, ENCODE_BYTES)
            src_v = data[:enc_n]
            cap = int(prod.lib.zxc_compress_bound(enc_n))
            enc_out = np.zeros(cap, dtype=np.uint8)

            def encode_leg(level):
                o = z.CompressOpts(level=level, block_size=BLOCK, seekable=1)
                r_enc = prod.lib.zxc_compress(src_v.ctypes.data, enc_n, enc_out.ctypes.data, cap, C.byref(o))  # warm-up
                t = time.perf_counter()
                r_enc = prod.lib.zxc_compress(src_v.ctypes.data, enc_n, enc_out.ctypes.data, cap, C.byref(o))
                enc_dt = time.perf_counter() - t
                want = reference_sha(frame_key(enc_n / (1 << 30), 0, level))
                cpu_gbs = None
                if ref is not None:
                    t = time.perf_counter()
                    ref_frame = zc.compress_ref_mt(ref, src_v, level=level, block_size=BLOCK)
                    cpu_gbs = round(enc_n / (time.perf_counter() - t) / 1e9, 3)
                    want = sha256(ref_frame)
                return {"level": level, "bytes_in": int(enc_n), "gbs_in_e2e": round(enc_n / enc_dt / 1e9, 3),
                        "identical_to_reference": None if want is None else r_enc > 0 and sha256(enc_out[:r_enc]) == want,
                        "ratio": round(r_enc / enc_n, 4),
                        "cpu_reference_gbs_in": cpu_gbs, "cpu_threads": threads}

            del d_src, d_dst
            torch.cuda.empty_cache()
            line["dict"] = dict_leg(lib, prod, ref, dev, stream, threads, args.dict_records, args.steps, peak)
            line["encode"] = encode_leg(6)
            line["encode"]["note"] = "configs[2]: optimal parser + Huffman sections on the GPU; levels 1-7 all encode on the GPU"
            line["encode"]["level3"] = encode_leg(LEVEL)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
