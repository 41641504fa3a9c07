// ASCII case fold of a scan's input for caseless table sets (PFAC_PATTERNS_CASELESS, include/pfac_b200.h).
//
// A caseless set's tables are those of its folded patterns; launch_scan runs this kernel before the detector, on
// the same stream, so that every kernel of the scan reads folded text and none of them changes (DESIGN.md §3.10).
// Bytes 0x41-0x5A become 0x61-0x7A; every other byte, 0x80-0xFF included, is left as it is.  The fold is
// idempotent: bytes folded twice (a flow's carried tail) are unchanged by the second pass.
#pragma once
#include "pfac_kernel.cuh"

#if defined(__CUDACC__)

namespace pfac {

constexpr int kFoldThreads = 256;
constexpr int kFoldUnroll = 4;   // 16-byte words in flight per thread

// Four bytes at once: a byte is an upper-case letter iff its low seven bits are >= 0x41 and < 0x5B and its top
// bit is clear; (t + 0x3f) and (t + 0x25) set bit 7 of a byte at exactly those two bounds, without carries
// between bytes (t <= 0x7f).  Bit 5 of such a byte is then set.
__device__ __forceinline__ uint32_t fold_word(uint32_t w)
{
    const uint32_t t = w & 0x7f7f7f7fu;
    const uint32_t up = (t + 0x3f3f3f3fu) & ~(t + 0x25252525u) & ~w & 0x80808080u;
    return w | (up >> 2);
}

__device__ __forceinline__ uint8_t fold_byte(uint8_t c) { return (c >= 0x41u && c <= 0x5Au) ? (uint8_t)(c | 0x20u) : c; }

// out_al[i] = fold(in_al[i]) for i in [lo, hi), in aligned-stream coordinates: in_al and out_al are 16-byte
// aligned (in_al = out_al folds in place).  The 16-byte words inside [lo, hi) are loaded and stored whole; the
// partial first and last words byte by byte, so nothing outside [in_al + lo, in_al + hi) is read and nothing
// outside [out_al + lo, out_al + hi) is written.
__global__ void __launch_bounds__(kFoldThreads) pfac_fold_kernel(const uint8_t *in_al, uint8_t *out_al,
                                                                 unsigned long long lo, unsigned long long hi)
{
    pdl_launch_next();
    // before the first read AND the first write: the kernels of the previous scan on this stream read out_al
    pdl_wait();
    const unsigned long long w_lo = (lo + 15u) >> 4, w_hi = hi >> 4;   // whole words [w_lo, w_hi)
    const unsigned long long tid = (unsigned long long)blockIdx.x * kFoldThreads + threadIdx.x;
    const unsigned long long nthreads = (unsigned long long)gridDim.x * kFoldThreads;
    if (tid < 32u) {   // the partial words: the head [lo, min(hi, 16 w_lo)), the tail [max(lo, 16 w_hi), hi)
        const unsigned long long head_end = min(hi, w_lo << 4);
        const unsigned long long i = tid < 16u ? lo + tid : max(head_end, w_hi << 4) + (tid - 16u);
        if (tid < 16u ? i < head_end : i < hi) out_al[i] = fold_byte(in_al[i]);
    }
    const uint4 *src = reinterpret_cast<const uint4 *>(in_al);
    uint4 *dst = reinterpret_cast<uint4 *>(out_al);
    for (unsigned long long w = w_lo + tid; w < w_hi; w += kFoldUnroll * nthreads) {
        uint4 v[kFoldUnroll];
#pragma unroll
        for (int k = 0; k < kFoldUnroll; k++) {
            const unsigned long long j = w + (unsigned long long)k * nthreads;
            if (j < w_hi) v[k] = src[j];
        }
#pragma unroll
        for (int k = 0; k < kFoldUnroll; k++) {
            const unsigned long long j = w + (unsigned long long)k * nthreads;
            if (j < w_hi) dst[j] = make_uint4(fold_word(v[k].x), fold_word(v[k].y), fold_word(v[k].z), fold_word(v[k].w));
        }
    }
}

}  // namespace pfac

#endif  // __CUDACC__
