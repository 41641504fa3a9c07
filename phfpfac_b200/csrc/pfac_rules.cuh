// Verify pass of sets with per-pattern case rules (PFAC_PATTERNS_CASE_RULES, include/pfac_b200.h, DESIGN.md §3.11).
//
// A mixed set's automaton is that of its folded patterns: launch_scan folds the text out of place, the unchanged
// detector, dense-match and ordering kernels scan the folded copy, and their records -- (pos, owner id), ordered
// by (pos, pattern length) -- land in the slot's pre-record buffer.  This pass turns each of them into the records
// of the owner's group members that match at pos: a caseless member (and an exact member without letters) always
// does; an exact member with letters does iff the ORIGINAL text at pos equals its bytes.  Members of a group are
// stored in ascending id order and all have the owner's length, so the output is ordered by (pos, length, id).
// Two launches, both over the pre-record count the ordering pass left in Result::count: pfac_rules_count_kernel and
// pfac_rules_write_kernel are the stable expansion of pfac_compact.cuh, each pre-record yielding the records of its
// passing members into the caller's buffer.
// If the pre-records overflowed their buffer, the count passed on is pre_count x (largest group): with that
// capacity a rescan's pre-records fit and so do its expanded records.  Nothing is written past out[cap).
#pragma once
#include "pfac_compact.cuh"

#if defined(__CUDACC__)

namespace pfac {

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

// The verify pass as a stable expansion (pfac_compact.cuh): a pre-record yields one record per passing member
struct RulesPass {
    const RulesParams &p;
    unsigned long long in_cap;
    uint2 r;   // the last pre-record counted
    __device__ explicit RulesPass(const RulesParams &rp) : p(rp), in_cap(rp.pre_cap) {}
    __device__ void setup(unsigned long long, unsigned long long) {}
    __device__ uint32_t count(unsigned long long i)
    {
        r = p.pre[i];
        return rules_count(p, r);
    }
    __device__ void write(unsigned long long, unsigned long long at)
    {
        const int2 g = __ldg(p.grp + r.y);
        for (int j = 0; j < g.y && at < p.cap; j++) {
            const int4 m = __ldg(p.mem + g.x + j);
            if (rules_pass(p, r, m)) p.out[at++] = make_uint2(r.x, (uint32_t)m.x);
        }
    }
    __device__ unsigned long long overflow(unsigned long long n) const { return n * p.max_group; }
};

__global__ void __launch_bounds__(kCompactThreads) pfac_rules_count_kernel(const RulesParams p) { compact_count(RulesPass(p)); }

__global__ void __launch_bounds__(kCompactThreads) pfac_rules_write_kernel(const RulesParams p) { compact_write(RulesPass(p)); }

}  // namespace pfac

#endif  // __CUDACC__
