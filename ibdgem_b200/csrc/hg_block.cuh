// hg_block.cuh — the chunked-block pipeline of the batched hiddengem kernels (viterbi_fused_kernel in hidden.cu,
// posterior_fwd_kernel / posterior_bwd_kernel in posterior.cu).  The recursions are sequential in bins and
// independent across tables, but the caller's arrays are table-major.  So a block takes 32 tables; eight worker warps
// move 16-bin chunks between global and shared memory with coalesced accesses (a table's chunk is 384 contiguous
// bytes) and do the per-bin work that is parallel over bins; ONE solver warp (lane = table) walks each chunk in
// shared memory.  Chunks are double buffered: buffer b = chunk & 1 (or, walking backwards, the chunk's rank & 1).
#pragma once

#include <stdint.h>

namespace ibdgem {

constexpr int HG_TABLES = 32, HG_BINS = 16, HG_ROW = HG_BINS * 3 + 1;  // padded row: lanes hit distinct banks
constexpr int HG_WORKERS = 256, HG_THREADS = HG_WORKERS + 32;         // thread 0-31: the solver warp
constexpr int HG_NLD = HG_TABLES * HG_BINS * 3 / HG_WORKERS;  // doubles of a chunk each worker moves
constexpr int HG_NBIN = HG_TABLES * HG_BINS / HG_WORKERS;     // bins of a chunk each worker handles
constexpr int HG_HEAD_SMEM = 2 * HG_TABLES * 8;               // s_start, s_len

// The block's tables [blockIdx.x * 32, + 32): start and length into shared memory (0 past n_tables).  Synchronises
// the block; returns the number of chunks of its longest table.
__device__ __forceinline__ int block_tables(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len,
                                            int64_t *s_start, int64_t *s_len) {
    if (threadIdx.x < HG_TABLES) {
        const int tb = blockIdx.x * HG_TABLES + threadIdx.x;
        s_start[threadIdx.x] = tb < n_tables ? start[tb] : 0;
        s_len[threadIdx.x] = tb < n_tables ? len[tb] : 0;
    }
    __syncthreads();
    int64_t blk_bins = 0;
    for (int k = 0; k < HG_TABLES; k++) blk_bins = max(blk_bins, s_len[k]);
    return (int)((blk_bins + HG_BINS - 1) / HG_BINS);
}

// A worker's share of chunk c of the block's tables, rows [t][bin * 3 + state] of the caller's table-major arrays.
struct ChunkLoader {
    const int64_t *s_start, *s_len;
    int w;  // worker index, 0..HG_WORKERS-1
    // raw likelihoods into registers; rows past a table's end read as 0
    __device__ __forceinline__ void fetch(const double *__restrict__ lik, int c, double (&pre)[HG_NLD]) const {
        const int64_t i0 = (int64_t)c * HG_BINS;
#pragma unroll
        for (int k = 0; k < HG_NLD; k++) {
            const int idx = k * HG_WORKERS + w;
            const int t = idx / (HG_BINS * 3), d = idx % (HG_BINS * 3);
            pre[k] = (i0 + d / 3 < s_len[t]) ? __ldcs(lik + (s_start[t] + i0) * 3 + d) : 0.0;
        }
    }
    __device__ __forceinline__ void store(const double (&pre)[HG_NLD], double (*buf)[HG_ROW]) const {
#pragma unroll
        for (int k = 0; k < HG_NLD; k++) {
            const int idx = k * HG_WORKERS + w;
            buf[idx / (HG_BINS * 3)][idx % (HG_BINS * 3)] = pre[k];
        }
    }
    // a chunk in shared memory back to global memory; rows past a table's end are not written
    __device__ __forceinline__ void write(int c, const double (*buf)[HG_ROW], double *__restrict__ out) const {
        const int64_t i0 = (int64_t)c * HG_BINS;
#pragma unroll
        for (int k = 0; k < HG_NLD; k++) {
            const int idx = k * HG_WORKERS + w;
            const int t = idx / (HG_BINS * 3), d = idx % (HG_BINS * 3);
            if (i0 + d / 3 < s_len[t]) __stcs(out + (s_start[t] + i0) * 3 + d, buf[t][d]);
        }
    }
};

// Named barriers: 1 + b = chunk in buffer b is ready for the solver (workers arrive, solver syncs);
//                 3 + b = chunk in buffer b is solved (solver arrives, workers sync); 5 = workers only.
__device__ __forceinline__ void arrive_ready(int b) {
    if (b == 0) asm volatile("bar.arrive 1, %0;" ::"n"(HG_THREADS) : "memory");
    else asm volatile("bar.arrive 2, %0;" ::"n"(HG_THREADS) : "memory");
}
__device__ __forceinline__ void sync_ready(int b) {
    if (b == 0) asm volatile("bar.sync 1, %0;" ::"n"(HG_THREADS) : "memory");
    else asm volatile("bar.sync 2, %0;" ::"n"(HG_THREADS) : "memory");
}
__device__ __forceinline__ void arrive_solved(int b) {
    if (b == 0) asm volatile("bar.arrive 3, %0;" ::"n"(HG_THREADS) : "memory");
    else asm volatile("bar.arrive 4, %0;" ::"n"(HG_THREADS) : "memory");
}
__device__ __forceinline__ void sync_solved(int b) {
    if (b == 0) asm volatile("bar.sync 3, %0;" ::"n"(HG_THREADS) : "memory");
    else asm volatile("bar.sync 4, %0;" ::"n"(HG_THREADS) : "memory");
}
__device__ __forceinline__ void sync_workers() { asm volatile("bar.sync 5, %0;" ::"n"(HG_WORKERS) : "memory"); }

}  // namespace ibdgem
