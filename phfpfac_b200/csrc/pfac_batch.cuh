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
//   pfac_batch_count_kernel  \ the stable expansion of pfac_compact.cuh, each raw record yielding itself if it
//   pfac_batch_split_kernel  /  is kept: {p - doc[d], id} into the caller's buffer, p into kpos
//   pfac_batch_docs_kernel   doc_first[i] = kept records before doc[i] (a binary search of kpos)
// A raw count beyond the raw buffer is passed on as the count (it bounds the kept count: the caller rescans
// with a buffer that size).
// The streaming scan (pfac_flows.cuh) runs the count and split kernels with CARRY = true: its document d is the
// carried tail of a flow (tail[d] bytes) followed by the new chunk, and a record is kept iff its pattern ends in
// the chunk, doc[d] + tail[d] < p + len[id] <= doc[d + 1].  doc_first needs no change: every kept record of
// document d still starts at or after doc[d].
#pragma once
#include "pfac_compact.cuh"

#if defined(__CUDACC__)

namespace pfac {

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

// The split pass as a stable expansion (pfac_compact.cuh): a raw record yields itself if it is kept
template <bool CARRY>
struct BatchPass {
    const BatchParams &p;
    unsigned long long in_cap;
    const uint32_t *win;   // documents of the range's first and last record (shared memory)
    uint2 r;               // the last record counted, and its document
    uint32_t d;
    __device__ explicit BatchPass(const BatchParams &b) : p(b), in_cap(b.raw_cap) {}
    // every record of the range lies in [win[0], win[1]]: the search per record starts from that window
    __device__ void setup(unsigned long long lo, unsigned long long hi)
    {
        __shared__ uint32_t s_doc[2];
        if (lo < hi && (threadIdx.x == 0 || threadIdx.x == 32))
            s_doc[threadIdx.x >> 5] = batch_doc_of(p.doc, 0u, p.n_docs, p.raw[threadIdx.x == 0 ? lo : hi - 1].x);
        win = s_doc;
    }
    __device__ uint32_t count(unsigned long long i) { return batch_keep<CARRY>(p, i, win[0], win[1], r, d) ? 1u : 0u; }
    __device__ void write(unsigned long long, unsigned long long at)
    {
        if (at < p.cap) p.out[at] = make_uint2(r.x - __ldg(p.doc + d), r.y);
        p.kpos[at] = r.x;   // (at < kept <= raw count <= raw_cap)
    }
    __device__ unsigned long long overflow(unsigned long long n) const { return n; }
};

template <bool CARRY>
__global__ void __launch_bounds__(kCompactThreads) pfac_batch_count_kernel(const BatchParams b) { compact_count(BatchPass<CARRY>(b)); }

template <bool CARRY>
__global__ void __launch_bounds__(kCompactThreads) pfac_batch_split_kernel(const BatchParams b) { compact_write(BatchPass<CARRY>(b)); }

__global__ void __launch_bounds__(kCompactThreads) pfac_batch_docs_kernel(const BatchParams b)
{
    pdl_launch_next();
    pdl_wait();
    const unsigned long long total = b.result->count;
    if (total > b.raw_cap) return;   // (the raw records did not fit: doc_first is unspecified)
    const unsigned long long step = (unsigned long long)gridDim.x * kCompactThreads;
    for (unsigned long long j = (unsigned long long)blockIdx.x * kCompactThreads + threadIdx.x; j <= b.n_docs; j += step) {
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
