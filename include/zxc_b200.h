/*
 * zxc_b200.h -- ADDITIVE device-resident entry points of the B200 build.
 *
 * The reference C API (zxc_buffer.h, zxc_seekable.h) takes host pointers, so
 * every call pays PCIe both ways.  These entry points expose the same block
 * decode with the compressed frame and the output already in HBM: the host
 * walks the frame once into a job table (one entry per block), the kernel
 * decodes all jobs in one launch.  They are what bench.py times for the
 * HBM-resident `value`, and what a multi-GPU caller shards by block range.
 *
 * Nothing here exists in the reference; adding symbols passes its ABI policy
 * (abidiff --no-added-syms, .github/workflows/abi-check.yml:128).
 *
 * Pointers named d_* are DEVICE pointers on the current CUDA device.
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 */
#ifndef ZXC_B200_H
#define ZXC_B200_H

#include <stddef.h>
#include <stdint.h>

#include "zxc_export.h"
#include "zxc_opts.h"

#ifdef __cplusplus
extern "C" {
#endif

/* One independent block = one unit of work (a CTA of the block-cooperative kernel, or a warp of
 * the general kernel).  Replaces the reference's
 * zxc_seek_mt_job_t (src/lib/zxc_seekable.c:802-815). */
typedef struct {
    uint64_t src_off; /* byte offset of the 8-byte block header inside the source buffer */
    uint64_t dst_off; /* byte offset of the block's first decoded byte inside the output */
    uint32_t src_len; /* on-disk size: header + payload (+4 checksum when the frame has them) */
    uint32_t dst_cap; /* bytes the block may produce (block_size, or the tail remainder) */
} zxc_b200_job_t;

/* What the host learnt from walking a frame. */
typedef struct {
    uint64_t decoded_size;  /* footer value */
    uint32_t block_size;    /* from the file header */
    uint32_t n_blocks;      /* data blocks found before EOF */
    uint32_t dict_id;       /* 0 = none */
    int has_checksum;       /* file flag 0x80 */
    int seekable;           /* a valid SEK table was found and used */
    uint32_t global_hash;   /* footer value (0 without checksums) */
} zxc_b200_frame_info_t;

/* Number of usable CUDA devices (0 when there is no driver / no device). */
ZXC_EXPORT int zxc_b200_device_count(void);

/* Walk a frame held in HOST memory and fill jobs[0..n) (dst offsets assume every
 * block but the last decodes to block_size, which the decode then verifies).
 * Always the sequential header walk of zxc_decompress_frame (src/lib/zxc_dispatch.c:912-1001),
 * so damaged block headers are reported exactly as the reference reports them; the SEK
 * table is only probed to fill info->seekable.  jobs may be NULL to query the count.  Returns the number of blocks or a negative zxc_error_t. */
ZXC_EXPORT int64_t zxc_b200_plan_frame(const void* frame, size_t frame_size, zxc_b200_job_t* jobs,
                                       size_t max_jobs, zxc_b200_frame_info_t* info);

/* Bytes of device scratch zxc_b200_decode_blocks needs for blocks of at most
 * block_size decoded bytes (RLE / Huffman literal sections are expanded there). */
ZXC_EXPORT size_t zxc_b200_decode_scratch_size(uint32_t block_size);

/* Decode n_jobs blocks, device to device, on `stream` (asynchronous).
 *   d_src     base of the compressed bytes the jobs index into
 *   d_dst     base of the output
 *   d_jobs    job table in device memory
 *   d_status  one int32 per job: decoded byte count, or a negative zxc_error_t
 *   d_dict    dictionary content or NULL; d_dict_huf its 128-byte table or NULL
 *   d_scratch zxc_b200_decode_scratch_size(block_size) bytes
 *   verify_checksums  non-zero: jobs carry a trailing rapidhash fold, check it
 * Returns ZXC_OK once the launch is enqueued, or a negative code: ZXC_ERROR_NULL_INPUT when d_src, d_dst, d_jobs,
 * d_status or d_scratch is NULL; ZXC_ERROR_MEMORY when scratch_size is below what this launch needs (then nothing
 * is launched and d_status is untouched).  n_jobs == 0 launches nothing.
 *
 * What a caller may rely on (tests/test_device_abi_gpu.py, tests/test_simt_layouts.py):
 *   - no alignment is required of d_src, d_dst, d_dict, d_dict_huf or of any src_off / dst_off;
 *   - offsets are full 64-bit byte offsets (buffers beyond 4 GiB);
 *   - the job table is any list of jobs: any order, a subset of a frame's blocks with rebased offsets, gaps or
 *     overlaps between source ranges, the same source block decoded to several windows.  Output windows
 *     [dst_off, dst_off + dst_cap) of different jobs must not overlap;
 *   - a job writes nothing outside its window, whatever its block holds.  Its status is what the reference's block
 *     decoder gives for that block at that dst_cap, including DST_TOO_SMALL / OVERFLOW when dst_cap is too small;
 *     its bytes are valid only where the status is >= 0, and only the first `status` of them;
 *   - every job's dst_cap is at most block_size, which sizes the scratch (it need not be the frame's block size);
 *   - d_dict_huf may live in an allocation of its own; it need not follow the dictionary;
 *   - jobs without a dictionary reference ignore d_dict; a block that refers to one needs it;
 *   - one scratch serves any number of launches in stream order without being cleared (its last 32 bytes hold the
 *     launch's work counters, which every launch resets); launches that may run at the same time, on different
 *     streams, each need their own scratch, status and output. */
ZXC_EXPORT int zxc_b200_decode_blocks(const void* d_src, void* d_dst, const zxc_b200_job_t* d_jobs,
                                      uint32_t n_jobs, int32_t* d_status, const void* d_dict,
                                      uint32_t dict_size, const void* d_dict_huf, void* d_scratch,
                                      size_t scratch_size, uint32_t block_size,
                                      int verify_checksums, void* stream);

/* Reduce a status array (device) to the reference's frame verdict: total bytes
 * if every job produced exactly its dst_cap (a 64-bit sum), else the code of the
 * failing job with the lowest index (ZXC_ERROR_CORRUPT_DATA for a size mismatch).
 * 0 for n_jobs == 0.  Synchronises `stream`. */
ZXC_EXPORT int64_t zxc_b200_reduce_status(const int32_t* d_status, const zxc_b200_job_t* d_jobs,
                                          uint32_t n_jobs, void* stream);

/* Kernels launched by this library since load (for bench.py's gpu_launches). */
ZXC_EXPORT uint64_t zxc_b200_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* ZXC_B200_H */
