// Device-side carry of the streaming scan (pfac_scan_flows_device_sync, include/pfac_b200.h).
//
// A flow set keeps, per flow, the last t_f = min(M - 1, P_f) bytes of its stream in a row of the tail store
// (M = max_pat_len, P_f = bytes the flow has consumed).  A call takes n chunks of distinct flows and runs the
// batch path (pfac_batch.cuh) over documents that are each flow's tail followed by its chunk:
//   pfac_flow_pack_kernel  tail_f ++ chunk_i for every chunk, back to back, into the packed buffer
//   (the packed scan: detector, dense-match pass, ordering pass, unchanged)
//   (the split pass with CARRY = true: a record is kept iff its pattern ends in the chunk)
//   pfac_flow_tail_kernel  the last min(M - 1, t_i + c_i) bytes of every document -> its flow's tail row, only
//                          if the call's records fit (result->count <= cap) and the watchdog did not trip
// A match that ends in the chunk starts at or after P_f - (M - 1), i.e. inside the tail or the chunk, so the
// union of a flow's records over its calls is exactly the scan of its whole stream (DESIGN.md §3.9).
#pragma once
#include "pfac_batch.cuh"

#if defined(__CUDACC__)

namespace pfac {

constexpr int kFlowThreads = 256;
constexpr uint32_t kPackWarpBytes = 32u * 16u;   // one 16-byte word per lane and step

struct FlowParams {
    const uint8_t *in;          // the caller's chunks (any alignment)
    const uint32_t *doc;        // n + 1 offsets of the documents in the packed buffer (doc[0] = 0)
    const uint32_t *tail;       // n: carried bytes at the start of every document
    const uint32_t *flow;       // n: flow of every chunk (distinct)
    const uint32_t *src;        // n: offset of every chunk in `in`
    uint32_t n;
    uint32_t total;             // doc[n]: packed bytes
    uint8_t *tails;             // tail store: one row of `stride` bytes per flow
    uint32_t stride;            // round_up(keep, 16)
    uint32_t keep;              // M - 1
    uint8_t *packed;            // total bytes, rounded up to 16, + 32 readable bytes
    const Result *result;       // tail kernel: the call's count and watchdog
    unsigned long long cap;
};

// The 16 bytes at p (any alignment), built from the aligned 16-byte words that hold them (both hold some of
// them: nothing outside the allocation of p[0, 16) is read)
__device__ __forceinline__ uint4 load16(const uint8_t *p)
{
    const uintptr_t a = (uintptr_t)p;
    const uint32_t sh = (uint32_t)(a & 15u);
    const uint4 *w = reinterpret_cast<const uint4 *>(a - sh);
    const uint4 lo = w[0];
    if (sh == 0) return lo;
    const uint4 hi = w[1];
    const uint32_t W[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    const uint32_t q = sh >> 2, b = (sh & 3u) * 8u;
    uint32_t r[5];
#pragma unroll
    for (int k = 0; k < 5; k++) r[k] = q == 0 ? W[k] : q == 1 ? W[k + 1] : q == 2 ? W[k + 2] : W[k + 3];
    return make_uint4(__funnelshift_r(r[0], r[1], b), __funnelshift_r(r[1], r[2], b), __funnelshift_r(r[2], r[3], b),
                      __funnelshift_r(r[3], r[4], b));
}

// Work is balanced over the output bytes: every warp builds 512-byte segments of the packed buffer, one 16-byte
// store per lane.  A word inside one tail or one chunk is two aligned loads and funnel shifts; a word across a
// seam (tail | chunk, document | document) is assembled byte by byte.
__global__ void __launch_bounds__(kFlowThreads) pfac_flow_pack_kernel(const FlowParams f)
{
    pdl_launch_next();
    pdl_wait();   // the previous call's tail kernel has written the tails and its scan has read the packed buffer
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned long long warps = (unsigned long long)gridDim.x * (kFlowThreads / 32);
    for (unsigned long long seg = (unsigned long long)blockIdx.x * (kFlowThreads / 32) + (threadIdx.x >> 5);
         seg * kPackWarpBytes < f.total; seg += warps) {
        const uint32_t s0 = (uint32_t)(seg * kPackWarpBytes);
        const uint32_t s1 = min(f.total, s0 + kPackWarpBytes) - 1u;
        // the documents of the segment's first and last byte bound the search of every word in it
        uint32_t dd = 0;
        if (lane == 0 || lane == 31) dd = batch_doc_of(f.doc, 0u, f.n, lane == 0 ? s0 : s1);
        const uint32_t d_lo = __shfl_sync(0xffffffffu, dd, 0), d_hi = __shfl_sync(0xffffffffu, dd, 31);
        const uint32_t o = s0 + 16u * lane;
        if (o >= f.total) continue;
        uint32_t d = batch_doc_of(f.doc, d_lo, d_hi + 1u, o);
        uint32_t lo = __ldg(f.doc + d), hi = __ldg(f.doc + d + 1), t = __ldg(f.tail + d);
        uint4 v;
        if (o >= lo + t && o + 16u <= hi) {
            v = load16(f.in + __ldg(f.src + d) + (o - lo - t));
        } else if (o + 16u <= lo + t) {
            v = load16(f.tails + (size_t)__ldg(f.flow + d) * f.stride + (o - lo));
        } else {
            uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (uint32_t j = 0; j < 16u; j++) {
                const uint32_t p = o + j;
                if (p >= f.total) break;
                if (p >= hi) {   // (p < total = doc[n]: a later document holds p)
                    d = batch_doc_of(f.doc, d + 1u, f.n, p);
                    lo = __ldg(f.doc + d);
                    hi = __ldg(f.doc + d + 1);
                    t = __ldg(f.tail + d);
                }
                const uint32_t q = p - lo;
                const uint32_t byte = q < t ? f.tails[(size_t)__ldg(f.flow + d) * f.stride + q]
                                            : __ldg(f.in + __ldg(f.src + d) + (q - t));
                w[j >> 2] |= byte << (8u * (j & 3u));
            }
            v = make_uint4(w[0], w[1], w[2], w[3]);
        }
        *reinterpret_cast<uint4 *>(f.packed + o) = v;
    }
}

// One warp per chunk: the last min(keep, t_i + c_i) bytes of document i become its flow's tail, 16 bytes per lane
// (the row is 16-byte aligned and `stride` long; the bytes past the tail are never read).
__global__ void __launch_bounds__(kFlowThreads) pfac_flow_tail_kernel(const FlowParams f)
{
    pdl_launch_next();
    pdl_wait();   // the split pass has finished: result->count is the call's count
    if (f.result->error_flag != 0u || f.result->count > f.cap) return;   // the call does not commit
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = gridDim.x * (kFlowThreads / 32);
    for (uint32_t i = blockIdx.x * (kFlowThreads / 32) + (threadIdx.x >> 5); i < f.n; i += warps) {
        const uint32_t hi = __ldg(f.doc + i + 1);
        const uint32_t k = min(f.keep, hi - __ldg(f.doc + i));
        uint8_t *row = f.tails + (size_t)__ldg(f.flow + i) * f.stride;
        for (uint32_t w = lane; 16u * w < k; w += 32u)
            *reinterpret_cast<uint4 *>(row + 16u * w) = load16(f.packed + (hi - k) + 16u * w);
    }
}

}  // namespace pfac

#endif  // __CUDACC__
