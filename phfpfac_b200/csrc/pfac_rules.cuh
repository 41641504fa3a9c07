// Verify pass of sets with per-pattern case rules (PFAC_PATTERNS_CASE_RULES, include/pfac_b200.h, DESIGN.md §3.11).
//
// A mixed set's automaton is that of its folded patterns: launch_scan folds the text out of place, the unchanged
// detector, dense-match and ordering kernels scan the folded copy, and their records -- (pos, owner id), ordered
// by (pos, pattern length) -- land in the slot's pre-record buffer.  This pass turns each of them into the records
// of the owner's group members that match at pos: a caseless member (and an exact member without letters) always
// does; an exact member with letters does iff the ORIGINAL text at pos equals its bytes.  Members of a group are
// stored in ascending id order and all have the owner's length, so the output is ordered by (pos, length, id).
// Two launches, both over the pre-record count the ordering pass left in Result::count:
//   pfac_rules_count_kernel  passing members of each CTA's contiguous range of pre-records
//   pfac_rules_write_kernel  stable compaction (a block scan: a record expands to 0..G outputs) into the caller's
//                            buffer; the last CTA writes Result::count and the caller's count
// If the pre-records overflowed their buffer, the count passed on is pre_count x (largest group): with that
// capacity a rescan's pre-records fit and so do its expanded records.  Nothing is written past out[cap).
#pragma once
#include "pfac_kernel.cuh"

#if defined(__CUDACC__)

namespace pfac {

constexpr int kRulesThreads = 256;

struct RulesParams {
    const uint2 *pre;              // the detector's records (pos, owner id); their count in result->count
    unsigned long long pre_cap;
    const uint8_t *in_al;          // the original (unfolded) text in aligned-stream coordinates
    uint32_t mis, pos_bias;        // a record at pos starts at in_al[mis + pos - pos_bias]
    const int2 *grp;               // [n_ids] {first member, members} of an owner id
    uint32_t n_ids;
    const int4 *mem;               // {id, length, offset of its bytes in pool (-1: matches wherever its owner does), 0}
    const uint8_t *pool;
    unsigned long long max_group;  // members of the largest group
    unsigned long long *blk;       // [gridDim.x + 1]: expanded records per CTA, then the pre-record count
    uint2 *out;                    // caller's records
    unsigned long long cap;
    Result *result;
    unsigned long long *count_out; // caller's count (may be null)
};

__device__ __forceinline__ bool rules_pass(const RulesParams &p, uint2 r, int4 m)
{
    if (m.z < 0) return true;
    const uint8_t *t = p.in_al + ((unsigned long long)p.mis + r.x - p.pos_bias);
    const uint8_t *q = p.pool + m.z;
    // 16 bytes per step with no exit inside it: the step's loads are independent and in flight together (a
    // byte-by-byte loop with an early exit waits one memory round trip per byte)
    for (int k0 = 0; k0 < m.y; k0 += 16) {
        uint32_t diff = 0;
#pragma unroll
        for (int k = 0; k < 16; k++)
            if (k0 + k < m.y) diff |= (uint32_t)(__ldg(t + k0 + k) ^ __ldg(q + k0 + k));
        if (diff) return false;
    }
    return true;
}

// members of record r's group that pass (owner ids are checked when the tables are built or loaded)
__device__ __forceinline__ uint32_t rules_count(const RulesParams &p, uint2 r)
{
    if (r.y >= p.n_ids) return 0u;
    const int2 g = __ldg(p.grp + r.y);
    uint32_t c = 0;
    for (int j = 0; j < g.y; j++) c += rules_pass(p, r, __ldg(p.mem + g.x + j)) ? 1u : 0u;
    return c;
}

// This CTA's contiguous range [lo, hi) of the n pre-records
__device__ __forceinline__ void rules_range(unsigned long long n, unsigned long long &lo, unsigned long long &hi)
{
    const unsigned long long per = (n + gridDim.x - 1) / gridDim.x;
    lo = min(n, (unsigned long long)blockIdx.x * per);
    hi = min(n, lo + per);
}

__global__ void __launch_bounds__(kRulesThreads) pfac_rules_count_kernel(const RulesParams p)
{
    __shared__ unsigned long long s_sum[kRulesThreads / 32];
    pdl_launch_next();
    pdl_wait();   // the ordering pass (or the dense-match kernel) has finished
    // (a tripped watchdog leaves the records unspecified: nothing is read, the caller gets the error)
    const unsigned long long n = p.result->error_flag ? 0ull : p.result->count;
    if (blockIdx.x == 0 && threadIdx.x == 0) p.blk[gridDim.x] = n;   // (the write kernel rewrites result->count)
    if (n > p.pre_cap) return;
    unsigned long long lo, hi, c = 0;
    rules_range(n, lo, hi);
    for (unsigned long long i = lo + threadIdx.x; i < hi; i += kRulesThreads) c += rules_count(p, p.pre[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kRulesThreads / 32; w++) t += s_sum[w];
        p.blk[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kRulesThreads) pfac_rules_write_kernel(const RulesParams p)
{
    __shared__ unsigned long long s_red[kRulesThreads / 32];
    __shared__ unsigned int s_warp[kRulesThreads / 32];
    __shared__ unsigned long long s_run;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_launch_next();
    pdl_wait();
    const unsigned long long n = p.blk[gridDim.x];
    if (n > p.pre_cap) {   // the pre-records did not fit: a capacity with which the rescan fits
        if (blockIdx.x == 0 && tid == 0) {
            p.result->count = n * p.max_group;
            if (p.count_out) *p.count_out = n * p.max_group;
        }
        return;
    }
    // expanded records of the CTAs before this one
    unsigned long long before = 0;
    for (uint32_t i = (uint32_t)tid; i < blockIdx.x; i += kRulesThreads) before += p.blk[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (lane == 0) s_red[warp] = before;
    __syncthreads();
    if (tid == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kRulesThreads / 32; w++) t += s_red[w];
        s_run = t;
    }
    __syncthreads();
    unsigned long long lo, hi;
    rules_range(n, lo, hi);
    for (unsigned long long c0 = lo; c0 < hi; c0 += kRulesThreads) {
        const unsigned long long i = c0 + (unsigned long long)tid;
        const uint2 r = i < hi ? p.pre[i] : make_uint2(0u, 0xFFFFFFFFu);
        const uint32_t c = i < hi ? rules_count(p, r) : 0u;
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
        if (c) {
            const int2 g = __ldg(p.grp + r.y);
            for (int j = 0; j < g.y && at < p.cap; j++) {
                const int4 m = __ldg(p.mem + g.x + j);
                if (rules_pass(p, r, m)) p.out[at++] = make_uint2(r.x, (uint32_t)m.x);
            }
        }
        __syncthreads();
        if (tid == 0) {
            unsigned long long t = 0;
            for (int w = 0; w < kRulesThreads / 32; w++) t += s_warp[w];
            s_run += t;
        }
        __syncthreads();
    }
    if (blockIdx.x == gridDim.x - 1 && tid == 0) {   // the last range ends the pre-records: its end is the total
        p.result->count = s_run;
        if (p.count_out) *p.count_out = s_run;
    }
}

}  // namespace pfac

#endif  // __CUDACC__
