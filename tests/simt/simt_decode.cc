/*
 * TEST INFRASTRUCTURE -- tests/simt/simt_decode.cc
 *
 * Compiles the product's decode DEVICE code (zxc_b200/csrc/zxc_decode.cuh and what it includes) for the CPU on top
 * of the fiber warp emulator in this directory and exposes one entry point that decodes a job table the way
 * zxc_decode_kernel does: one (emulated) warp per job, decode_job<UNITS>() unchanged.  Used by
 * tests/test_simt_decode.py to check the kernel source bit-for-bit against the reference without a GPU and under
 * randomised lane scheduling.  Never linked into libzxc.so.
 */
#include <cuda_runtime.h>

#include <vector>

extern "C" { uint64_t simt_stat[32]; }
#define ZXC_STAT(i, v) do { const uint64_t zv_ = (uint64_t)(v); if (simt::g_warp->current == 0) simt_stat[i] += zv_; } while (0)

#include <stdio.h>
uint32_t simt_bar_issued[64], simt_bar_waited[64];
uint32_t simt_bar_base;
void simt_stage_fail(const char* what) {
    fprintf(stderr, "simt stage check failed: %s\n", what);
    abort();
}

#include "zxc_decode.cuh"
SimtStore simt_stores[64];
u32 simt_n_stores;

alignas(16) u8 smem[DECODE_SMEM_BYTES];

namespace {
const u32 PAD = 256;
}

extern "C" uint64_t simt_decode_blocks(const u8* src, uint64_t src_size, u8* dst, uint64_t dst_size,
                                       const zxc_b200_job_t* jobs, u32 n_jobs, i32* status, const u8* dict, u32 dict_size,
                                       const u8* dict_huf, u32 block_cap, u32 flags, int units, uint64_t seed,
                                       int* oob_writes) {
    /* device buffers with a guard band either side: word loads may touch a few bytes outside, stores must not */
    std::vector<u8> in(src_size + 2 * PAD, 0xA5), out(dst_size + 2 * PAD, 0x5A), dct((size_t)dict_size + 128 + 2 * PAD, 0x33);
    memcpy(in.data() + PAD, src, src_size);
    memcpy(out.data() + PAD, dst, dst_size); /* the caller's bytes: what a job does not write must come back unchanged */
    if (dict && dict_size) memcpy(dct.data() + PAD, dict, dict_size);
    if (dict_huf) memcpy(dct.data() + PAD + dict_size, dict_huf, 128);
    const u32 stride = scr_stride(block_cap);
    std::vector<u8> scratch((size_t)stride + 2 * PAD, 0x77);
    unsigned long long counter = 0;
    DecodeParams P;
    memset(&P, 0, sizeof P);
    P.src = in.data() + PAD;
    P.dst = out.data() + PAD;
    P.jobs = jobs;
    P.status = status;
    P.dict = (dict && dict_size) ? dct.data() + PAD : nullptr;
    P.dict_huf = dict_huf ? dct.data() + PAD + dict_size : nullptr;
    P.scratch = scratch.data() + PAD;
    P.counter = &counter;
    P.n_jobs = n_jobs;
    P.dict_size = dict_size;
    P.scratch_stride = stride;
    P.flags = flags;
    P.block_cap = block_cap;
    uint64_t rendezvous = 0;
    for (u32 j = 0; j < n_jobs; j++) {
        const zxc_b200_job_t job = jobs[j];
        u8* scr = P.scratch + 256; /* the lead-in zxc_decode_kernel leaves */
        u8* ring = smem;
        auto body = [&](unsigned lane) {
#if ZXC_STAGE
            simt_bar_base = smem_addr(ring) + RING_BYTES + ST_OFF_BAR;
            st_init(smem_addr(ring) + RING_BYTES, lane);
#endif
            const bool has_dict = P.dict != nullptr && P.dict_size != 0;
            const int r = units ? (has_dict ? decode_job<true, true>(P, job, scr, ring, lane) : decode_job<true, false>(P, job, scr, ring, lane))
                                : (has_dict ? decode_job<false, true>(P, job, scr, ring, lane) : decode_job<false, false>(P, job, scr, ring, lane));
            flush_wait(lane);
            __syncwarp();
            if (lane == 0) status[j] = r;
        };
        rendezvous += simt::run_warp(body, 0, 0, CTA_THREADS, seed ? seed + j : 0);
        if (simt_n_stores) simt_stage_fail("a bulk store was still in flight when the warp finished");
        for (int b = 0; b < 64; b++)
            if (simt_bar_issued[b] != simt_bar_waited[b]) simt_stage_fail("a bulk copy was still in flight when the block ended");
    }
    int bad = 0;
    for (u32 k = 0; k < PAD; k++) bad += (out[k] != 0x5A) + (out[PAD + dst_size + k] != 0x5A);
    if (oob_writes) *oob_writes = bad;
    memcpy(dst, out.data() + PAD, dst_size);
    return rendezvous;
}

extern "C" u32 simt_scratch_stride(u32 block_cap) { return scr_stride(block_cap); }
