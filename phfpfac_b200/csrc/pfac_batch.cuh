// Split pass of the batch scan (pfac_scan_batch_device, include/pfac_b200.h).
//
// The documents of a batch are packed back to back and scanned ONCE with the ordinary launch sequence
// (detector, dense-match pass, ordering pass), whose records -- ordered by (global position, pattern length)
// -- land in a raw buffer.  This pass turns them into the per-document results:
//   a record at global position p with pattern id belongs to document d = the last one with doc[d] <= p
//   (empty documents never own one) and is kept iff p + len[id] <= doc[d + 1], i.e. the match ends inside
//   its document.  The automaton is a trie, so a walk from p reaches a final state at depth L iff
//   text[p, p + L) is that pattern; for an L that stays inside the document the packed buffer gives the same
//   answer as the document alone, and every match of the document alone starts in it.  Hence the kept
//   records are exactly the per-document results.
// Three launches, all over the raw count the ordering pass left in Result::count:
//   pfac_batch_count_kernel  kept records of each CTA's contiguous range of raw records
//   pfac_batch_split_kernel  stable compaction: {p - doc[d], id} into the caller's buffer, p into kpos
//   pfac_batch_docs_kernel   doc_first[i] = kept records before doc[i] (a binary search of kpos)
// A raw count beyond the raw buffer is passed on as the count (it bounds the kept count: the caller rescans
// with a buffer that size).
// The streaming scan (pfac_flows.cuh) runs the count and split kernels with CARRY = true: its document d is the
// carried tail of a flow (tail[d] bytes) followed by the new chunk, and a record is kept iff its pattern ends in
// the chunk, doc[d] + tail[d] < p + len[id] <= doc[d + 1].  doc_first needs no change: every kept record of
// document d still starts at or after doc[d].
#pragma once
#include "pfac_kernel.cuh"

#if defined(__CUDACC__)

namespace pfac {

constexpr int kBatchThreads = 256;

struct BatchParams {
    const uint2 *raw;           // raw records of the packed scan, count in result->count
    unsigned long long raw_cap;
    const uint32_t *doc;        // n_docs + 1 document offsets (doc[0] = 0, non-decreasing)
    uint32_t n_docs;
    const int32_t *len;         // pattern length of every id
    uint32_t n_ids;
    unsigned long long *blk;    // kept records per CTA of the count / split kernels, then the raw count (gridDim.x + 1)
    uint2 *out;                 // caller's records
    unsigned long long cap;
    uint32_t *kpos;             // global positions of the kept records (raw_cap entries)
    unsigned long long *doc_first;   // caller's n_docs + 1 offsets
    Result *result;
    unsigned long long *count_out;   // caller's count (may be null)
    const uint32_t *tail;       // CARRY: bytes of carried tail at the start of every document (null for batches)
};

// last d in [a, b) with doc[d] <= p (doc[a] <= p)
__device__ __forceinline__ uint32_t batch_doc_of(const uint32_t *doc, uint32_t a, uint32_t b, uint32_t p)
{
    while (b - a > 1u) {
        const uint32_t m = (a + b) >> 1;
        if (__ldg(doc + m) <= p) a = m;
        else b = m;
    }
    return a;
}

// This CTA's contiguous range [lo, hi) of the n raw records, and the documents of its first and last record
// (every record of the range lies in [s_doc[0], s_doc[1]]: the search per record starts from that window).
__device__ __forceinline__ void batch_range(const BatchParams &b, unsigned long long n, unsigned long long &lo,
                                            unsigned long long &hi, uint32_t *s_doc)
{
    const unsigned long long per = (n + gridDim.x - 1) / gridDim.x;
    lo = min(n, (unsigned long long)blockIdx.x * per);
    hi = min(n, lo + per);
    if (lo < hi && (threadIdx.x == 0 || threadIdx.x == 32)) {
        const unsigned long long i = threadIdx.x == 0 ? lo : hi - 1;
        s_doc[threadIdx.x >> 5] = batch_doc_of(b.doc, 0u, b.n_docs, b.raw[i].x);
    }
    __syncthreads();
}

// Is raw record i kept, and in which document does it lie
template <bool CARRY>
__device__ __forceinline__ bool batch_keep(const BatchParams &b, unsigned long long i, uint32_t d_lo, uint32_t d_hi,
                                           uint2 &r, uint32_t &d)
{
    r = b.raw[i];
    d = batch_doc_of(b.doc, d_lo, d_hi + 1u, r.x);
    const uint32_t L = r.y < b.n_ids ? (uint32_t)__ldg(b.len + r.y) : 0u;
    const unsigned long long end = (unsigned long long)r.x + L;
    if (CARRY && end <= (unsigned long long)__ldg(b.doc + d) + __ldg(b.tail + d)) return false;   // ends in the tail
    return end <= (unsigned long long)__ldg(b.doc + d + 1);
}

template <bool CARRY>
__global__ void __launch_bounds__(kBatchThreads) pfac_batch_count_kernel(const BatchParams b)
{
    __shared__ uint32_t s_doc[2];
    pdl_launch_next();
    pdl_wait();   // the ordering pass of the packed scan has finished
    const unsigned long long n = b.result->count;
    if (blockIdx.x == 0 && threadIdx.x == 0) b.blk[gridDim.x] = n;   // (the split kernel rewrites result->count)
    if (n > b.raw_cap) return;   // (the split kernel passes the raw count on)
    unsigned long long lo, hi;
    batch_range(b, n, lo, hi, s_doc);
    unsigned int kept = 0;
    for (unsigned long long i = lo + threadIdx.x; i < hi; i += kBatchThreads) {
        uint2 r;
        uint32_t d;
        kept += batch_keep<CARRY>(b, i, s_doc[0], s_doc[1], r, d) ? 1u : 0u;
    }
    __shared__ unsigned int s_sum[kBatchThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = kept;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kBatchThreads / 32; w++) t += s_sum[w];
        b.blk[blockIdx.x] = t;
    }
}

template <bool CARRY>
__global__ void __launch_bounds__(kBatchThreads) pfac_batch_split_kernel(const BatchParams b)
{
    __shared__ uint32_t s_doc[2];
    __shared__ unsigned long long s_red[kBatchThreads / 32];
    __shared__ unsigned int s_warp[kBatchThreads / 32];
    __shared__ unsigned long long s_run;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_launch_next();
    pdl_wait();
    const unsigned long long n = b.blk[gridDim.x];
    if (n > b.raw_cap) {   // the raw records did not fit: their count is the capacity of the rescan
        if (blockIdx.x == 0 && tid == 0 && b.count_out) *b.count_out = n;
        return;
    }
    // kept records of the CTAs before this one
    unsigned long long before = 0;
    for (uint32_t i = (uint32_t)tid; i < blockIdx.x; i += kBatchThreads) before += b.blk[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    if (lane == 0) s_red[warp] = before;
    __syncthreads();
    if (tid == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kBatchThreads / 32; w++) t += s_red[w];
        s_run = t;
    }
    unsigned long long lo, hi;
    batch_range(b, n, lo, hi, s_doc);   // (its barrier publishes s_run)
    for (unsigned long long c0 = lo; c0 < hi; c0 += kBatchThreads) {
        const unsigned long long i = c0 + (unsigned long long)tid;
        uint2 r = make_uint2(0u, 0u);
        uint32_t d = 0;
        const bool keep = i < hi && batch_keep<CARRY>(b, i, s_doc[0], s_doc[1], r, d);
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = (unsigned int)__popc(bal);
        __syncthreads();
        unsigned long long at = s_run;
        for (int w = 0; w < warp; w++) at += s_warp[w];
        at += (unsigned long long)__popc(bal & ((1u << lane) - 1u));
        if (keep) {
            if (at < b.cap) b.out[at] = make_uint2(r.x - __ldg(b.doc + d), r.y);
            b.kpos[at] = r.x;   // (at < kept <= raw count <= raw_cap)
        }
        __syncthreads();
        if (tid == 0) {
            unsigned long long t = 0;
            for (int w = 0; w < kBatchThreads / 32; w++) t += s_warp[w];
            s_run += t;
        }
        __syncthreads();
    }
    if (blockIdx.x == gridDim.x - 1 && tid == 0) {   // the last range ends the raw records: its end is the total
        b.result->count = s_run;
        if (b.count_out) *b.count_out = s_run;
    }
}

__global__ void __launch_bounds__(kBatchThreads) pfac_batch_docs_kernel(const BatchParams b)
{
    pdl_launch_next();
    pdl_wait();
    const unsigned long long total = b.result->count;
    if (total > b.raw_cap) return;   // (the raw records did not fit: doc_first is unspecified)
    const unsigned long long step = (unsigned long long)gridDim.x * kBatchThreads;
    for (unsigned long long j = (unsigned long long)blockIdx.x * kBatchThreads + threadIdx.x; j <= b.n_docs; j += step) {
        unsigned long long first = total;
        if (j < b.n_docs) {   // kept records before doc[j]: the first kpos >= doc[j]
            const uint32_t p = __ldg(b.doc + j);   // (kpos is ascending)
            unsigned long long a = 0, e = total;
            while (a < e) {
                const unsigned long long m = (a + e) >> 1;
                if (b.kpos[m] < p) a = m + 1;
                else e = m;
            }
            first = a;
        }
        b.doc_first[j] = first;
    }
}

}  // namespace pfac

#endif  // __CUDACC__
