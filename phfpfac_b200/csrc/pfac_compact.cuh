// Stable expansion of a record buffer (DESIGN.md §3.8): each input record yields 0..G output records, written in
// input order.  The batch and flow split pass (pfac_batch.cuh, G = 1) and the verify pass of mixed case-rule sets
// (pfac_rules.cuh) are this pass with their own records.  Two launches over the input count the kernel before
// left in Result::count:
//   count kernel  outputs of each CTA's contiguous range of input records -> blk[blockIdx.x]; blk[gridDim.x] = n
//   write kernel  the outputs of the CTAs before it, then a block scan of the per-record counts of each chunk of
//                 kCompactThreads records; the last CTA writes Result::count and the caller's count
// A tripped watchdog leaves the records unspecified: n reads as 0, nothing is read, and the caller gets the error.
// If the n input records exceeded their buffer, Result::count and the caller's count are overflow(n), a capacity
// with which one rescan fits; nothing is written.
//
// A pass is a per-thread object over its kernel parameters `p` (with blk, result and count_out) and supplies
//   in_cap                 the input buffer's capacity
//   setup(lo, hi)          per CTA, before a barrier: anything count() needs about the range [lo, hi)
//   count(i)               outputs of input record i
//   write(i, at)           those outputs from out[at] on (called after count(i) with a non-zero result)
//   overflow(n)            the count passed on when n > in_cap
#pragma once
#include "pfac_kernel.cuh"

#if defined(__CUDACC__)

namespace pfac {

constexpr int kCompactThreads = 256;

// This CTA's contiguous range [lo, hi) of the n input records
__device__ __forceinline__ void compact_range(unsigned long long n, unsigned long long &lo, unsigned long long &hi)
{
    const unsigned long long per = (n + gridDim.x - 1) / gridDim.x;
    lo = min(n, (unsigned long long)blockIdx.x * per);
    hi = min(n, lo + per);
}

template <class Pass>
__device__ __forceinline__ void compact_count(Pass ps)
{
    __shared__ unsigned long long s_sum[kCompactThreads / 32];
    pdl_launch_next();
    // the kernel before has finished: its records and count are final, and the write kernel of an earlier pass on
    // this slot has read blk
    pdl_wait();
    const unsigned long long n = ps.p.result->error_flag ? 0ull : ps.p.result->count;
    if (blockIdx.x == 0 && threadIdx.x == 0) ps.p.blk[gridDim.x] = n;   // (the write kernel rewrites result->count)
    if (n > ps.in_cap) return;
    unsigned long long lo, hi, c = 0;
    compact_range(n, lo, hi);
    ps.setup(lo, hi);
    __syncthreads();
    for (unsigned long long i = lo + threadIdx.x; i < hi; i += kCompactThreads) c += ps.count(i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kCompactThreads / 32; w++) t += s_sum[w];
        ps.p.blk[blockIdx.x] = t;
    }
}

template <class Pass>
__device__ __forceinline__ void compact_write(Pass ps)
{
    __shared__ unsigned long long s_red[kCompactThreads / 32];
    __shared__ unsigned int s_warp[kCompactThreads / 32];
    __shared__ unsigned long long s_run;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_launch_next();
    pdl_wait();
    const unsigned long long n = ps.p.blk[gridDim.x];
    if (n > ps.in_cap) {   // the input records did not fit: a capacity with which the rescan fits
        if (blockIdx.x == 0 && tid == 0) {
            const unsigned long long c = ps.overflow(n);
            ps.p.result->count = c;
            if (ps.p.count_out) *ps.p.count_out = c;
        }
        return;
    }
    // outputs of the CTAs before this one
    unsigned long long before = 0;
    for (uint32_t i = (uint32_t)tid; i < blockIdx.x; i += kCompactThreads) before += ps.p.blk[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (lane == 0) s_red[warp] = before;
    __syncthreads();
    if (tid == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kCompactThreads / 32; w++) t += s_red[w];
        s_run = t;
    }
    unsigned long long lo, hi;
    compact_range(n, lo, hi);
    ps.setup(lo, hi);
    __syncthreads();   // (publishes s_run and the pass's setup)
    for (unsigned long long c0 = lo; c0 < hi; c0 += kCompactThreads) {
        const unsigned long long i = c0 + (unsigned long long)tid;
        const uint32_t c = i < hi ? ps.count(i) : 0u;
        uint32_t incl = c;   // block scan of the per-record counts
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned long long at = s_run + (incl - c);
        for (int w = 0; w < warp; w++) at += s_warp[w];
        if (c) ps.write(i, at);
        __syncthreads();
        if (tid == 0) {
            unsigned long long t = 0;
            for (int w = 0; w < kCompactThreads / 32; w++) t += s_warp[w];
            s_run += t;
        }
        __syncthreads();
    }
    if (blockIdx.x == gridDim.x - 1 && tid == 0) {   // the last range ends the input records: its end is the total
        ps.p.result->count = s_run;
        if (ps.p.count_out) *ps.p.count_out = s_run;
    }
}

}  // namespace pfac

#endif  // __CUDACC__
