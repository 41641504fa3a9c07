// PFAC scan kernels for sm_100a (B200).  Replace TraceTable_kernel + SUBSEG_MATCH
// (reference master_kernel.cu:37-180).  Design notes: DESIGN.md section 3.
//
//   pfac_scan2_kernel / pfac_scan_kernel<MODE>   the detector: persistent, one CTA per SM, warp specialised.
//     * producer warp (one lane): streams the CTA's tiles of 16 x 512 bytes (+ halo of max_pat_len-1 bytes)
//       into a shared-memory ring with cp.async.bulk (TMA bulk copy, SASS UBLKCP), full/empty mbarriers per
//       stage, L2 evict-first hint on the streamed input;
//     * 31 consumer warps taking slots (4 consecutive 512-byte slices) of the CTA's tiles from a shared
//       counter.  Per slot
//         stage 1  16 start positions per lane and slice against T1 (64 KiB byte table over 2-byte windows,
//                  probed at even offsets only in mode 0; up to eight bit-planes: root fan-out + depth-1 rows,
//                  bytes 1-2 .. 5-6, short-pattern exceptions) -- or, in global mode, against T2 (a blocked
//                  Bloom filter of the 4-byte prefixes); survivors compacted into the warp's queue;
//         stage 2  survivors against the two-point checks (4-byte prefix -> m1 -> window -> m2 -> window -> T3)
//                  or T2.
//       A start that survives becomes a CANDIDATE of its tile; the detector's filters decide nothing else.
//       All of them are shared-memory (global mode: L2) resident prefix filters derived from the first PHF rows.
//     * the warp that finishes a tile's last slot publishes the tile, hands the stage back and settles the
//       tile's candidates: through the pattern directory (emit_tile_dir: every pattern length probed in
//       parallel, exact compare) or by the plain PFAC walk of SUBSEG_MATCH (emit_tile) straight from the PHF;
//       records go, one (position, pattern length)-ordered run per tile, into the arrival-order scratch.
//   pfac_dense_kernel     tiles with more candidates than the detector keeps (and, DIRECT, whole scans of sets
//                         with patterns of <= 3 bytes): every start walked, level-synchronously.
//   pfac_finalize_kernel  scans the per-tile counts and moves the runs from arrival order to position order --
//                         the order main.cc:341-349 prints.  Output is deterministic run to run.
//   All kernels of a scan are programmatic dependent launches (griddepcontrol).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#ifdef PFAC_TRACE   // development build (make variant NAME=trace EXTRA=-DPFAC_TRACE): device-side timeline of a scan
#include <stdio.h>
#endif

#include "pfac_derive.h"

namespace pfac {

struct Ctrl {   // device-side control block; the finalize kernel resets it for the next launch
    unsigned int ticket;
    unsigned int error_flag;
    unsigned long long alloc;   // records reserved in the arrival-order scratch
    unsigned int n_dense;       // tiles the detector handed over whole (to the dense-match pass)
    unsigned int exited;        // CTAs of a DIRECT dense-match scan that are done (the last one resets this block)
};

struct Result {   // written by the finalize kernel, copied to the host
    unsigned long long count;
    unsigned int error_flag;
    unsigned int pad;
};

// what a walk needs: the input, the canonical PHF arrays, the scratch and the tile directory
struct EmitParams {
    const uint8_t *in_al;
    uint32_t mis, a_start_end, a_valid_end, max_pat_len;
    int32_t use_ref_bound;
    uint64_t base_pos;
    uint32_t pos_bias;
    const int32_t *r;
    const int2 *htval;
    const int32_t *idmap;
    const int32_t *s0;        // root row, s0Table (main.cc:200)
    // The same transition function in the layout of the candidate walks (null when the PHF width is below 256):
    // step[idx] = {HT[idx], val[idx], r[row of val[idx]]}, s0r[b] = {s0Table[b], r[row of it]} -- a walk step is
    // ONE dependent load instead of r[] then {HT,val}
    const int4 *step;
    const int2 *s0r;
    // pattern directory (pfac_derive.h PatDir; null: walk instead): the strings of the final states, hashed
    const uint4 *dir;
    const uint8_t *pool;
    uint32_t dir_slots;
    unsigned long long len_mask;
    int32_t ht_size, width_bit, n_final;
    uint2 *scratch;
    unsigned long long scratch_cap;
    unsigned int *tile_cnt;
    unsigned long long *tile_src;   // [n_tiles] start of the tile's (contiguous, position-ordered) run of records in the scratch
    unsigned int *tile_nc;
    uint32_t n_tiles, tiles_per_part;
    unsigned long long *partial;
    Ctrl *ctrl;
};

struct ScanParams {
    const uint8_t *in_al;     // 16-byte aligned base: caller's pointer rounded down
    uint32_t mis;             // offset of the first start position in the aligned stream (0..15)
    uint32_t a_start_end;     // mis + n_starts   (aligned-stream coordinates, exclusive)
    uint32_t a_valid_end;     // mis + n_valid
    uint32_t n_tiles;
    uint32_t halo;            // staged halo bytes, multiple of 16, >= max_pat_len-1
    uint32_t max_pat_len;
    int32_t use_ref_bound;    // reproduce the 4096+512 walk bound (master_kernel.cu:141-144)
    uint64_t base_pos;        // global position of the first start position
    // shared-memory image (pfac_derive.h)
    const uint4 *image;
    uint32_t image_bytes, off_t2, off_tm, off_tm2, off_t3;
    uint32_t t2_shift, has_short, has_t3, t3_shift, tm_bits, tm2_bits;
    uint32_t off_d1, off_e1, nb1, ns1, off_d2, off_e2, nb2, ns2;   // mode 0: perfect-hash tables (pfac_derive.h)
    const uint8_t *gimage;            // mode 2: T1 | Tm | Tm2 | T3 in global memory (offsets above refer to it)
    uint32_t ticket_batch;            // tiles a producer claims with one atomic (1 for small inputs: balance first)
    uint32_t n_stages, stage_magic;   // depth of the input ring (as many as shared memory holds); floor(2^32 / n_stages) + 1
    // output
    unsigned int *tile_cnt;           // [n_tiles] matches of the tile (0 for the tiles handed to the dense-match kernel, which sets it)
    unsigned int *tile_nc;            // [n_tiles] kCandOverflow: too many candidates, the dense-match kernel walks the whole tile; else 0
    unsigned long long *partial;      // [kMaxParts] matches per tile range (for the ordering pass); zero on entry
    unsigned long long *partial_next; // [kMaxParts] the other of the slot's two buffers: zeroed here for the next scan
    EmitParams emit;                  // the walk parameters (emit_tile)
    Ctrl *ctrl;
    uint32_t debug;           // PFAC_DEBUG bits (timing experiments only): 4 no T1, 8 no stage 2
};

struct FinalizeParams {
    const unsigned int *tile_cnt;
    const unsigned long long *tile_src;   // [n_tiles] where the tile's run of records starts in the scratch
    const uint2 *scratch;
    unsigned long long scratch_cap;
    uint2 *out;
    unsigned long long cap;
    uint32_t n_tiles, tiles_per_part;
    const unsigned long long *partial;
    Ctrl *ctrl;
    Result *result;
    unsigned long long *count_out;    // caller's device counter (may be null)
    uint32_t debug, trace_ctas;       // PFAC_TRACE builds: PFAC_DEBUG bits, CTAs of the detector
};

#ifndef PFAC_CONSUMER_WARPS
#define PFAC_CONSUMER_WARPS 31
#endif
constexpr int kConsumerWarps = PFAC_CONSUMER_WARPS;
constexpr int kThreads = (kConsumerWarps + 1) * 32;   // + the producer warp
constexpr int kSlice = 512;           // start positions per stage-1 step of a warp (32 lanes x 16 B)
#ifndef PFAC_TILE_SLICES
#define PFAC_TILE_SLICES 16
#endif
constexpr int kSlicesPerTile = PFAC_TILE_SLICES;    // (<= 32: one flag bit each in the stage's `done` word)
constexpr int kTile = kSlicesPerTile * kSlice;   // 8,192 start positions per tile
// Slices a warp takes at a time (a slot): stage 2 then runs over the survivors of all of them.
// Shared-memory mode: 2 (more would leave too few slots in flight for the ring to prefetch).  Global
// mode: 4 -- stage 2 waits on L2 there, and a fuller queue means more loads in flight per wait.
#ifndef PFAC_SLOT_SLICES
#define PFAC_SLOT_SLICES 2
#endif
#ifndef PFAC_SLOT_SLICES_GLOBAL
#define PFAC_SLOT_SLICES_GLOBAL 4
#endif
#ifndef PFAC_SLOT_SLICES2
#define PFAC_SLOT_SLICES2 4
#endif
// mode (pfac_derive.h): 0 = pfac_scan2_kernel, 1 = pfac_scan_kernel<1> (T1 + T2), 2 = pfac_scan_kernel<2> (global tables)
__host__ __device__ constexpr int slot_slices(int mode) { return mode == 2 ? PFAC_SLOT_SLICES_GLOBAL : mode == 1 ? PFAC_SLOT_SLICES : PFAC_SLOT_SLICES2; }
__host__ __device__ constexpr int q1_cap(int mode) { return 64 * slot_slices(mode); }   // per consumer warp: starts of one slot that passed stage 1 (u16)
__host__ __device__ constexpr int queue_bytes(int mode) { return q1_cap(mode) * 2; }     // a slot with more survivors is handed over whole
// Ring depth the slot scheme needs.  Each warp holds one slot; when the ring is exhausted (or the
// work has ended) the warps block on slots of the next ceil(31 / slots per tile) tiles.  A blocked
// slot's tile must be the NEXT fill of its stage, not the one after -- an mbarrier phase parity
// cannot tell those apart -- so the ring has to be at least that many stages deep.
__host__ __device__ constexpr int min_stages(int mode)
{
    return (kConsumerWarps + kSlicesPerTile / slot_slices(mode) - 1) / (kSlicesPerTile / slot_slices(mode));
}
static_assert(kSlicesPerTile % PFAC_SLOT_SLICES == 0 && kSlicesPerTile % PFAC_SLOT_SLICES_GLOBAL == 0 && kSlicesPerTile % PFAC_SLOT_SLICES2 == 0, "slots tile the tile");
constexpr int kMaxStages = 16;
constexpr int kCtrlBytes = 1664;          // CtlView below
constexpr int kMaxParts = 1024;           // tile ranges of the ordering pass (one per finalize CTA)
constexpr int kCandPerTile = 32;          // candidate starts the detector hands over per tile (more: whole slices)
constexpr unsigned kCandOverflow = 0xFFFFFFFFu;
// Device-side watchdog of the waits (never expected to trip): a TIME limit on the GPU's global timer, not a
// spin count -- under MPS / time slicing / a profiler's replay a correct scan may poll any number of times.
constexpr unsigned long long kWatchdogNs = 20ull * 1000ull * 1000ull * 1000ull;
__device__ __forceinline__ unsigned long long gtime_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
struct Watchdog {   // checks the clock every 1024 polls only
    unsigned spins = 0;
    unsigned long long t0 = 0;
    __device__ __forceinline__ bool expired()
    {
        if ((++spins & 1023u) != 0u) return false;
        const unsigned long long now = gtime_ns();
        if (!t0) { t0 = now; return false; }
        return now - t0 > kWatchdogNs;
    }
};
#ifndef PFAC_WAIT_NS
#define PFAC_WAIT_NS 1000
#endif
constexpr unsigned kWaitNs = PFAC_WAIT_NS;   // suspend-time hint of the consumers' wait for a tile
#ifndef PFAC_TICKET_BATCH
#define PFAC_TICKET_BATCH 4
#endif
constexpr int kTicketBatch = PFAC_TICKET_BATCH;   // tiles a producer claims with one atomic

__host__ __device__ inline uint32_t scan_buf_stride(uint32_t halo) { return (kTile + halo + 32 + 127) & ~127u; }
__host__ inline size_t scan_smem_bytes(uint32_t image_bytes, uint32_t halo, uint32_t n_stages, int mode)
{
    return (size_t)image_bytes + kCtrlBytes + (size_t)kConsumerWarps * queue_bytes(mode) +
           (size_t)n_stages * scan_buf_stride(halo);
}

#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Programmatic dependent launch: the three kernels of a scan are enqueued back to back; the detector lets the
// next kernel's launch proceed at once (pdl_launch_next), and that kernel's CTAs -- set up while the detector
// still runs -- block in pdl_wait() until the whole grid before them has finished and its writes are visible.
// Without the launch attribute both are no-ops.
__device__ __forceinline__ void pdl_launch_next() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
#ifndef PFAC_WAIT_HINT_NS
#define PFAC_WAIT_HINT_NS 0      // suspend-time hint of mbarrier.try_wait (0: none)
#endif
#ifndef PFAC_CONS_SLEEP_NS
#define PFAC_CONS_SLEEP_NS 32    // consumer back-off between polls of a full barrier
#endif
#ifndef PFAC_PROD_SLEEP_NS
#define PFAC_PROD_SLEEP_NS 64    // producer back-off between polls of an empty barrier
#endif
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
#if PFAC_WAIT_HINT_NS > 0
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"   // %3: suspend-time hint (ns)
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"((unsigned)PFAC_WAIT_HINT_NS) : "memory");
#else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
#endif
    return ok != 0;
}
// The same with a suspend-time hint: the warp sleeps inside the instruction until the phase completes
// or about `ns` nanoseconds have passed -- a waiting warp issues nothing in between (a poll loop with
// nanosleep costs issue slots and, for its exit conditions, shared-memory wavefronts).
__device__ __forceinline__ bool mbar_try_wait_for(uint64_t *bar, uint32_t parity, uint32_t ns)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(ns) : "memory");
    return ok != 0;
}
// returns false if the watchdog tripped (never expected).  SLEEP_NS > 0: back off between polls so
// that a waiting warp does not burn the issue slots of the warps that work.
template <unsigned SLEEP_NS>
__device__ __forceinline__ bool mbar_wait(uint64_t *bar, uint32_t parity, unsigned int *error_flag, unsigned code)
{
    Watchdog wd;
    while (!mbar_try_wait(bar, parity)) {
        if (wd.expired()) {
            atomicExch(error_flag, code);
            return false;
        }
        if (SLEEP_NS) __nanosleep(SLEEP_NS);
    }
    return true;
}
// shared-memory atomic add of ONE lane (the caller has elected it): plain ATOMS, without the
// warp-aggregation preamble the compiler wraps around atomicAdd in possibly divergent code
__device__ __forceinline__ uint32_t atoms_add(uint32_t *addr, uint32_t v)
{
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(addr)), "r"(v) : "memory");
    return old;
}
// TMA bulk copy global -> shared with an L2 evict-first policy: the input is streamed once and
// must not push the PHF tables out of L2.  Completion is counted in bytes on the mbarrier.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

// rotl2 of each of the 4 bytes (pfac_derive.h rot2): bank-spreads the T1 index for ASCII text
__device__ __forceinline__ uint32_t rot2x4(uint32_t w)
{
#ifndef PFAC_NO_ROT2
    uint32_t r;   // one LOP3: bitwise select between the two shifted copies
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(r) : "r"(w << 2), "r"(w >> 6), "r"(0xFCFCFCFCu));
    return r;
#else
    return w;
#endif
}

// The kernel's dynamic shared memory.  T1 sits at offset 0 (pfac_derive.cc) so that its lookups
// are LDS.U8 [index + constant] with no address arithmetic.
extern __shared__ __align__(128) uint8_t smem[];

// 16 start positions per lane.  T1 holds four bit-planes per 2-byte window (pfac_derive.h); the
// result has one nibble per position, bit 0 of nibble j set iff start j passes stage 1:
//     P01(j) and (Short(j) or (P12(j+1) and P23(j+2)))
// lo = positions 0..7, hi = positions 8..15.  18 windows are looked up (16 + the two after them).
// The entries are packed one per nibble, so only those four planes may be kept: T1 also carries P34 and ShortC
// (bits 4 and 5, for stage 2 and mode 0), which would otherwise land in, and carry into, the next nibbles.
__device__ __forceinline__ void filter16(const uint4 v, const uint32_t nx, const int lane, uint32_t &lo, uint32_t &hi)
{
    const uint8_t *t1 = smem;
    const uint32_t w[5] = {rot2x4(v.x), rot2x4(v.y), rot2x4(v.z), rot2x4(v.w), rot2x4(nx)};
    uint32_t acc[2] = {0u, 0u};
    uint32_t first2 = 0;   // T1 of the lane's windows 0 and 1
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const uint32_t i0 = w[k] & 0xffffu;
        const uint32_t i1 = __byte_perm(w[k], 0u, 0x4421);
        const uint32_t i2 = w[k] >> 16;
        const uint32_t i3 = __funnelshift_r(w[k], w[k + 1], 24) & 0xffffu;
        uint32_t &a = acc[k >> 1];
        const int sh = (k & 1) * 16;
        const uint32_t e0 = t1[i0] & 15u, e1 = t1[i1] & 15u;
        if (k == 0) first2 = e0 | (e1 << 4);
        a += e0 << sh;
        a += e1 << (sh + 4);
        a += ((uint32_t)t1[i2] & 15u) << (sh + 8);
        a += ((uint32_t)t1[i3] & 15u) << (sh + 12);
    }
    // windows 16 and 17 (their P12 / P23 planes belong to starts 14..15) are the next lane's windows
    // 0 and 1: one shuffle instead of two more bank-conflicted look-ups; lane 31 has no neighbour
    uint32_t ex = __shfl_down_sync(0xffffffffu, first2, 1);
    if (lane == 31) ex = ((uint32_t)t1[w[4] & 0xffffu] & 15u) | (((uint32_t)t1[__byte_perm(w[4], 0u, 0x4421)] & 15u) << 4);
    // plane bits: 1 = P01, 2 = P12, 4 = P23, 8 = Short.  Align P12 of j+1 (shift 4+1), P23 of j+2
    // (shift 8+2) and Short of j (shift 3) with bit 0 of nibble j.
    const uint32_t y_lo = __funnelshift_r(acc[0], acc[1], 5), y_hi = __funnelshift_r(acc[1], ex, 5);
    const uint32_t z_lo = __funnelshift_r(acc[0], acc[1], 10), z_hi = __funnelshift_r(acc[1], ex, 10);
    lo = acc[0] & ((y_lo & z_lo) | (acc[0] >> 3)) & 0x11111111u;
    hi = acc[1] & ((y_hi & z_hi) | (acc[1] >> 3)) & 0x11111111u;
}

// Stage 1 of the global mode (pattern sets whose prefixes do not fit the shared-memory Tm): the
// hashed 4-byte prefix of each of the 16 starts against T2 (a blocked Bloom filter, pfac_derive.h), which
// fills shared memory -- one LDS.32 and one mask compare per start.  Result: bit j = start j of the lane passes.
__device__ __forceinline__ uint32_t one_hot(uint32_t n) { return __funnelshift_l(0u, 1u, n); }   // 1 << (n & 31): SHF.L.W
__device__ __forceinline__ bool t2_probe(const uint32_t *__restrict__ t2, uint32_t w4, uint32_t shift)
{
    const uint32_t h = w4 * kHash4Mul;
    uint32_t m = one_hot(h >> shift);
#pragma unroll
    for (int i = 1; i < kT2KeyBits; i++) m |= one_hot(h >> (shift - 5u * i));   // (shared-memory tables have at most 2^21 bits: shift >= 11)
    return (t2[h >> (shift + 5u)] & m) == m;
}
__device__ __forceinline__ uint32_t filter16_t2(const uint4 v, const uint32_t nx, const uint32_t *__restrict__ t2, uint32_t shift)
{
    const uint32_t w[5] = {v.x, v.y, v.z, v.w, nx};
    uint32_t acc = 0u;   // bit j: start j passes
#pragma unroll
    for (int k = 0; k < 4; k++) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t w4 = j == 0 ? w[k] : __funnelshift_r(w[k], w[k + 1], 8 * j);
            if (t2_probe(t2, w4, shift)) acc |= 1u << (k * 4 + j);
        }
    }
    return acc;
}
// bit 0 of each of the 8 nibbles -> 8 adjacent bits
__device__ __forceinline__ uint32_t nibble_bits(uint32_t x)
{
    x &= 0x11111111u;
    x = (x | (x >> 3)) & 0x03030303u;
    x = (x | (x >> 6)) & 0x000F000Fu;
    return (x | (x >> 12)) & 0xFFu;
}

// tile-relative bound of what a start at tile-relative tpos may read (master_kernel.cu:141-144 + input end)
__device__ __forceinline__ uint32_t walk_limit(const ScanParams &p, uint32_t a0, uint32_t tpos)
{
    uint32_t lim_a = p.a_valid_end;
    if (p.use_ref_bound) {
        // reference tiles are 4096 bytes of global positions with a 512-byte halo
        const unsigned long long g = p.base_pos + (unsigned long long)(a0 + tpos - p.mis);
        const unsigned long long lim_g = (g & ~4095ull) + 4608ull;
        const unsigned long long lim2 = lim_g - p.base_pos + p.mis;
        if (lim2 < lim_a) lim_a = (uint32_t)lim2;
    }
    uint32_t lim_t = lim_a - a0;
    const uint32_t depth = tpos + p.max_pat_len;   // a walk reads at most max_pat_len bytes
    return lim_t < depth ? lim_t : depth;
}

// A start that survived every filter: remember it as a candidate of its tile (past
// kCandPerTile the counter keeps growing and the tile is handed to the dense-match kernel whole)
__device__ __forceinline__ void add_candidate(uint32_t *n, uint16_t *list, uint32_t tpos)
{
    const uint32_t i = atomicAdd(n, 1u);
    if (i < (uint32_t)kCandPerTile) list[i] = (uint16_t)tpos;
    __threadfence_block();   // rare path: the list entry is visible before this warp reports the slot finished
}

// Read-only loads of the PHF tables with an L2 evict-last policy: the tables are a megabyte or a few
// that every walk chases through dependent loads, next to a gigabyte of input streamed with
// evict-first -- they are to stay in the 126 MB L2.
__device__ __forceinline__ uint64_t policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ int32_t ldg_keep(const int32_t *ptr)
{
    int32_t v;
    asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(ptr), "l"(policy_evict_last()));
    return v;
}
__device__ __forceinline__ int2 ldg_keep(const int2 *ptr)
{
    int2 v;
    asm volatile("ld.global.nc.L2::cache_hint.v2.b32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(ptr), "l"(policy_evict_last()));
    return v;
}

// ---------------------------------------------------------------------------------------------
// The plain PFAC walk of SUBSEG_MATCH (master_kernel.cu:37-74) over the canonical PHF arrays: used
// for the starts that survived every filter of the detector (by the warp that finishes their tile,
// emit_tile below) and, beyond the cached levels, by the dense-match kernel.

// master_kernel.cu:52-64 over the canonical arrays
__device__ __forceinline__ int32_t phf_next(const EmitParams &p, int32_t state, uint32_t byte)
{
    const int32_t key = (state << 8) + (int32_t)byte;                // :52
    const int32_t row = key >> p.width_bit;                          // :53
    const int32_t idx = ldg_keep(&p.r[row]) + (key & ((1 << p.width_bit) - 1));   // :54-55
    if (idx < 0 || idx >= p.ht_size) return -1;                      // :56-57
    const int2 hv = ldg_keep(&p.htval[idx]);                            // :59-61
    return hv.x == row ? hv.y : -1;
}

template <bool WRITE>
__device__ __forceinline__ uint32_t emit_walk(const EmitParams &p, uint32_t a, uint32_t lim_a, unsigned long long o)
{
    int32_t state = ldg_keep(&p.s0[p.in_al[a]]);                        // :41
    if (state < 0) return 0;                                         // :43
    uint32_t n = 0, q = a + 1;
    const uint32_t rec_pos = a - p.mis + p.pos_bias;
    while (true) {
        if (state < p.n_final) {                                     // :44-47, :67-70
            if (WRITE && o + n < p.scratch_cap) p.scratch[o + n] = make_uint2(rec_pos, (uint32_t)ldg_keep(&p.idmap[state]));
            n++;
        }
        if (q >= lim_a) break;                                       // :50
        state = phf_next(p, state, p.in_al[q]);
        if (state < 0) break;                                        // :63-64
        q++;
    }
    return n;
}

__device__ __forceinline__ int4 ldg_keep(const int4 *ptr)
{
    int4 v;
    asm volatile("ld.global.nc.L2::cache_hint.v4.b32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr), "l"(policy_evict_last()));
    return v;
}

// Text bytes of a candidate walk: the input is read in aligned 32-bit words, one word AHEAD of the walk, so that
// the byte a step needs is in a register and the step's only dependent load is the transition entry.  Words
// that would reach past the readable input are not loaded (the last bytes come one by one).
struct TextAhead {
    const uint8_t *in;
    uint32_t end;          // a_valid_end
    uint32_t cur = 0, nxt = 0;
    __device__ __forceinline__ uint32_t word(uint32_t a4) const   // aligned word at a4, bytes past `end` not touched
    {
        if (a4 + 4u <= end) return *reinterpret_cast<const uint32_t *>(in + a4);
        uint32_t w = 0;
        for (uint32_t i = 0; i < 4u && a4 + i < end; i++) w |= (uint32_t)in[a4 + i] << (8u * i);
        return w;
    }
    __device__ __forceinline__ void start(uint32_t a)
    {
        cur = word(a & ~3u);
        nxt = word((a & ~3u) + 4u);
    }
    __device__ __forceinline__ uint32_t at(uint32_t q)   // byte q; q only ever grows by one from start()'s a
    {
        const uint32_t b = (cur >> ((q & 3u) * 8u)) & 255u;
        if ((q & 3u) == 3u) {
            cur = nxt;
            nxt = word((q & ~3u) + 8u);
        }
        return b;
    }
};

// One walk, once, over the one-load layout (EmitParams::step): same states, same order as walk_collect below.
__device__ __forceinline__ uint32_t walk_collect_fast(const EmitParams &p, uint32_t a, uint32_t lim_a, int32_t (&st)[4])
{
    TextAhead tx{p.in_al, p.a_valid_end};
    tx.start(a);
    const int2 s = ldg_keep(&p.s0r[tx.at(a)]);                       // :41
    int32_t state = s.x, rcur = s.y;
    if (state < 0) return 0;                                         // :43
    uint32_t n = 0, q = a + 1;
    const int32_t mask = (1 << p.width_bit) - 1;
    while (true) {
        if (state < p.n_final) {                                     // :44-47, :67-70
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (n == (uint32_t)i) st[i] = state;
            n++;
        }
        if (q >= lim_a) break;                                       // :50
        const int32_t key = (state << 8) + (int32_t)tx.at(q);        // :52
        const int32_t row = key >> p.width_bit;                      // :53
        const int32_t idx = rcur + (key & mask);                     // :54-55
        if (idx < 0 || idx >= p.ht_size) break;                      // :56-57
        const int4 e = ldg_keep(&p.step[idx]);                       // :59-61
        if (e.x != row || e.y < 0) break;                            // :63-64
        state = e.y;
        rcur = e.z;
        q++;
    }
    return n;
}

// The same walk, once: counts the matches of start a and keeps the first kWalkKeep final states in
// registers, so that the records can be written after the scratch space is reserved without walking
// the (latency-bound) chain a second time.  Starts with more matches than that are walked again.
constexpr int kWalkKeep = 4;
__device__ __forceinline__ uint32_t walk_collect(const EmitParams &p, uint32_t a, uint32_t lim_a, int32_t (&st)[kWalkKeep])
{
    int32_t state = ldg_keep(&p.s0[p.in_al[a]]);                        // :41
    if (state < 0) return 0;                                         // :43
    uint32_t n = 0, q = a + 1;
    while (true) {
        if (state < p.n_final) {                                     // :44-47, :67-70
#pragma unroll
            for (int i = 0; i < kWalkKeep; i++)
                if (n == (uint32_t)i) st[i] = state;
            n++;
        }
        if (q >= lim_a) break;                                       // :50
        state = phf_next(p, state, p.in_al[q]);
        if (state < 0) break;                                        // :63-64
        q++;
    }
    return n;
}
__device__ __forceinline__ void write_collected(const EmitParams &p, uint32_t a, uint32_t lim_a, uint32_t n,
                                                const int32_t (&st)[kWalkKeep], unsigned long long o)
{
    if (n > (uint32_t)kWalkKeep) {
        emit_walk<true>(p, a, lim_a, o);
        return;
    }
    const uint32_t rec_pos = a - p.mis + p.pos_bias;
#pragma unroll
    for (int i = 0; i < kWalkKeep; i++)
        if ((uint32_t)i < n && o + i < p.scratch_cap) p.scratch[o + i] = make_uint2(rec_pos, (uint32_t)ldg_keep(&p.idmap[st[i]]));
}


// The walks of one tile: its (at most 32) candidates are sorted by position with a warp-wide bitonic
// network, every lane runs SUBSEG_MATCH for its start once, keeping the first final states in
// registers; the tile's records are reserved as ONE run of the arrival-order scratch (one atomic) and
// written in (position, pattern length) order.  Called by the warp that finished the tile's last slot.
// Not inlined: the detector's hot loop must not pay for its registers.
__device__ __noinline__ void emit_tile(const EmitParams &p, uint32_t tile, uint32_t my_cand, int lane)
{
    const uint32_t a0 = tile * (uint32_t)kTile;
    auto limit = [&](uint32_t a) {
        uint32_t lim_a = p.a_valid_end;
        if (p.use_ref_bound) {   // reference tiles: 4096 bytes of global positions + 512-byte halo
            const unsigned long long g = p.base_pos + (unsigned long long)(a - p.mis);
            const unsigned long long lim2 = ((g & ~4095ull) + 4608ull) - p.base_pos + p.mis;
            if (lim2 < lim_a) lim_a = (uint32_t)lim2;
        }
        const unsigned long long depth = (unsigned long long)a + p.max_pat_len;
        return depth < lim_a ? (uint32_t)depth : lim_a;
    };
    uint32_t key = my_cand;   // tile-relative start of lane's candidate, 0xFFFF = none
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1)
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {   // bitonic sort across the warp
            const uint32_t other = __shfl_xor_sync(0xffffffffu, key, j);
            const bool up = ((lane & k) == 0) == ((lane & j) == 0);
            key = up ? min(key, other) : max(key, other);
        }
    const bool live = key != 0xFFFFu;
    const uint32_t a = a0 + key;
    int32_t st[kWalkKeep];
    const uint32_t cnt = !live ? 0u : p.step ? walk_collect_fast(p, a, limit(a), st) : walk_collect(p, a, limit(a), st);
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    if (total) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&p.ctrl->alloc, (unsigned long long)total);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (cnt) write_collected(p, a, limit(a), cnt, st, base + incl - cnt);
        if (lane == 0) {
            p.tile_src[tile] = base;
            atomicAdd(&p.partial[tile / p.tiles_per_part], (unsigned long long)total);
        }
    }
    if (lane == 0) p.tile_cnt[tile] = total;
}

// The same for tiles with one or two candidates (nearly all of them when matches are sparse), without the
// chain of dependent transitions: for every pattern length d of the set at once -- lane l asks for d = l + 1
// and d = l + 33 -- "is text[start, start + d) a pattern?".  The start's bytes come from the staged tile
// (copied to registers before the stage went back to the producer, lane l holds bytes l and l + 32); the
// polynomial hashes of ALL prefixes come from one warp scan (pfac_derive.h); then one probe of the pattern
// directory per length and, on a hit, an exact compare of the bytes by the whole warp.  Three rounds of
// independent loads instead of up to 64 dependent ones.  The records equal the walk's: the automaton is a
// trie, text[start, start + d) reaches a final state iff it is that state's own string, and the walk's bound
// (end of input, reference tile bound, max_pat_len) caps d.  Returns false (nothing written) if a probe met a
// foreign string with the same 64-bit hash and length -- the caller then walks.
constexpr int kDirCand = 2;
constexpr uint32_t kNoHit = 0xFFFFFFFFu;
// K^e (or K^-e) for e < 64 from compile-time squares: six predicated 64-bit multiplies, no memory
template <bool INV>
__device__ __forceinline__ unsigned long long dir_pow(uint32_t e)
{
    unsigned long long r = 1ull;
#pragma unroll
    for (int i = 0; i < 6; i++)
        if ((e >> i) & 1u) r *= dir_cpow(INV ? kDirMulInv : kDirMul, 1u << i);
    return r;
}
__device__ __noinline__ bool emit_tile_dir(const EmitParams &p, uint32_t tile, uint32_t key0, uint32_t key1, uint32_t b0_lo,
                                           uint32_t b0_hi, uint32_t b1_lo, uint32_t b1_hi, int lane)
{
    const uint32_t a0 = tile * (uint32_t)kTile;
    const uint32_t key[kDirCand] = {key0, key1};   // tile-relative starts in position order, 0xFFFF = none
    const uint32_t blo[kDirCand] = {b0_lo, b1_lo}, bhi[kDirCand] = {b0_hi, b1_hi};
    const unsigned long long kinv_lo = dir_pow<true>((uint32_t)lane), kinv_hi = kinv_lo * dir_cpow(kDirMulInv, 32u);
    const unsigned long long kpow_lo = dir_pow<false>((uint32_t)lane + 1u), kpow_hi = kpow_lo * dir_cpow(kDirMul, 32u);
    // 1. the prefix hashes and the first probe of every (candidate, length): independent loads, all in flight together
    unsigned long long hd[kDirCand][2];
    uint32_t sl[kDirCand][2];
    int4 e[kDirCand][2];
    bool ask[kDirCand][2];
#pragma unroll
    for (int c = 0; c < kDirCand; c++) {
        uint32_t dmax = 0;
        if (key[c] != 0xFFFFu) {   // (uniform)
            const uint32_t a = a0 + key[c];
            uint32_t lim_a = p.a_valid_end;
            if (p.use_ref_bound) {   // reference tiles: 4096 bytes of global positions + 512-byte halo (master_kernel.cu:141-144)
                const unsigned long long g = p.base_pos + (unsigned long long)(a - p.mis);
                const unsigned long long lim2 = ((g & ~4095ull) + 4608ull) - p.base_pos + p.mis;
                if (lim2 < lim_a) lim_a = (uint32_t)lim2;
            }
            dmax = min(lim_a - a, p.max_pat_len);   // the deepest state the walk can reach (:50)
        }
        // prefix sums of (byte_i + 1) K^-i over i = 0..63, two elements per lane
        unsigned long long s_lo = (unsigned long long)(blo[c] + 1u) * kinv_lo, s_hi = (unsigned long long)(bhi[c] + 1u) * kinv_hi;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(0xffffffffu, s_lo, o), v = __shfl_up_sync(0xffffffffu, s_hi, o);
            if (lane >= o) { s_lo += u; s_hi += v; }
        }
        s_hi += __shfl_sync(0xffffffffu, s_lo, 31);
        hd[c][0] = s_lo * kpow_lo;   // hash of text[a, a + d), d = lane + 1
        hd[c][1] = s_hi * kpow_hi;   //                         d = lane + 33
#pragma unroll
        for (int r = 0; r < 2; r++) {
            const uint32_t d = (uint32_t)lane + 1u + 32u * r;
            ask[c][r] = d <= dmax && ((p.len_mask >> (d - 1u)) & 1ull);
            sl[c][r] = dir_slot(hd[c][r], p.dir_slots);
            e[c][r] = make_int4(0, 0, 0, -1);
            if (ask[c][r]) e[c][r] = ldg_keep(reinterpret_cast<const int4 *>(&p.dir[sl[c][r]]));
        }
    }
    // 2. resolve the probes (open addressing: nearly always the first slot decides)
    uint32_t hit[kDirCand][2], ew[kDirCand][2], bal[kDirCand][2], total = 0;
#pragma unroll
    for (int c = 0; c < kDirCand; c++)
#pragma unroll
        for (int r = 0; r < 2; r++) {
            hit[c][r] = kNoHit;
            ew[c][r] = 0xFFFFFFFFu;
            if (ask[c][r]) {
                const uint32_t d = (uint32_t)lane + 1u + 32u * r, lo = (uint32_t)hd[c][r], hi = (uint32_t)(hd[c][r] >> 32);
                int4 x = e[c][r];
                for (uint32_t q = sl[c][r]; (uint32_t)x.w != 0xFFFFFFFFu;) {
                    if ((uint32_t)x.x == lo && (uint32_t)x.y == hi && ((uint32_t)x.w >> 25) == d) { ew[c][r] = (uint32_t)x.w; hit[c][r] = (uint32_t)x.z; break; }
                    q = (q + 1u) & (p.dir_slots - 1u);
                    x = ldg_keep(reinterpret_cast<const int4 *>(&p.dir[q]));
                }
            }
            bal[c][r] = __ballot_sync(0xffffffffu, hit[c][r] != kNoHit);
            total += __popc(bal[c][r]);
        }
    // 3. the records' place in the scratch is reserved while the hits are verified byte by byte by the whole warp
    //    (lane l compares bytes l and l + 32 of the stored string)
    unsigned long long base = 0;
    if (total && lane == 0) base = atomicAdd(&p.ctrl->alloc, (unsigned long long)total);
    bool clean = true;
#pragma unroll
    for (int c = 0; c < kDirCand; c++)
#pragma unroll
        for (int r = 0; r < 2; r++)
            for (uint32_t hits = bal[c][r]; hits; hits &= hits - 1u) {
                const uint32_t w = __shfl_sync(0xffffffffu, ew[c][r], __ffs(hits) - 1);
                const uint32_t d = w >> 25;
                const uint8_t *pat = p.pool + (w & 0x1FFFFFFu);
                bool same = true;
                if ((uint32_t)lane < d) same = (uint32_t)__ldg(&pat[lane]) == blo[c];
                if ((uint32_t)lane + 32u < d) same = same && (uint32_t)__ldg(&pat[lane + 32]) == bhi[c];
                clean = clean && __all_sync(0xffffffffu, same);   // (uniform)
            }
    if (!clean) return false;   // a foreign string with the same hash and length: the caller walks (the reservation stays unused)
    if (total) {
        base = __shfl_sync(0xffffffffu, base, 0);
        uint32_t off = 0;
        const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
        for (int c = 0; c < kDirCand; c++)
#pragma unroll
            for (int r = 0; r < 2; r++) {
                const unsigned long long o = base + off + __popc(bal[c][r] & lt);
                if (hit[c][r] != kNoHit && o < p.scratch_cap) p.scratch[o] = make_uint2(a0 + key[c] - p.mis + p.pos_bias, hit[c][r]);
                off += __popc(bal[c][r]);
            }
        if (lane == 0) {
            p.tile_src[tile] = base;
            atomicAdd(&p.partial[tile / p.tiles_per_part], (unsigned long long)total);
        }
    }
    if (lane == 0) p.tile_cnt[tile] = total;
    return true;
}

// Development timeline (PFAC_TRACE builds, PFAC_DEBUG bit 64): every CTA of the detector stamps %globaltimer at
// its start (0), when the filter image is in (1), when its last tile is done (2), when that tile's candidates
// are settled (3) and when its last warp leaves (4) -- atomicMax into the last words of the record scratch;
// the ordering pass prints the minima / maxima over the CTAs next to its own start, wait and end.
#ifdef PFAC_TRACE
#define PFAC_STAMP(p, k)                                                                                                       \
    do {                                                                                                                       \
        if ((p).debug & 64u)                                                                                                   \
            atomicMax(reinterpret_cast<unsigned long long *>((p).emit.scratch + ((p).emit.scratch_cap - 1ull - blockIdx.x * 8ull - (k)))), \
                      gtime_ns());                                                                                             \
    } while (0)
#else
#define PFAC_STAMP(p, k) do { } while (0)
#endif

// The control block of the detector kernels (kCtrlBytes of shared memory after the image).
struct CtlView {
    uint64_t *full, *empty;     // [kMaxStages] mbarriers of the input ring
    uint32_t *tile;             // [kMaxStages] tile id of the stage
    uint32_t *ncand;            // [kMaxStages] candidates (bit 31: a dense slot, hand the slices over whole)
    uint32_t *done;             // [kMaxStages] low byte: slots of the tile that are finished; bits 8..: flagged slices
    uint32_t *grab;             // next (tile, slice) slot of this CTA
    uint32_t *kend;             // sequence number of the CTA's sentinel tile
    uint64_t *imgbar;           // mbarrier of the image copy
    uint16_t *cand;             // [kMaxStages][kCandPerTile]
};
__device__ __forceinline__ CtlView ctl_view(uint8_t *ctl)
{
    CtlView c;
    c.full = reinterpret_cast<uint64_t *>(ctl);
    c.empty = reinterpret_cast<uint64_t *>(ctl + 128);
    c.tile = reinterpret_cast<uint32_t *>(ctl + 256);
    c.ncand = reinterpret_cast<uint32_t *>(ctl + 384);
    c.done = reinterpret_cast<uint32_t *>(ctl + 448);
    c.grab = reinterpret_cast<uint32_t *>(ctl + 512);
    c.kend = reinterpret_cast<uint32_t *>(ctl + 516);
    c.imgbar = reinterpret_cast<uint64_t *>(ctl + 520);
    c.cand = reinterpret_cast<uint16_t *>(ctl + 640);
    return c;
}
static_assert(640 + kMaxStages * kCandPerTile * 2 <= kCtrlBytes, "control block");

__device__ __forceinline__ void bulk_g2s_plain(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Prologue shared by the detector kernels: barriers, control words, and the filter image, which one
// thread brings in with TMA bulk copies (the other warps meanwhile start on their roles; consumers wait
// for the image in image_wait()).
__device__ __forceinline__ void detector_init(const ScanParams &p, const CtlView &c)
{
    const int tid = threadIdx.x;
    if (tid == 0) PFAC_STAMP(p, 0);
    pdl_launch_next();
    if (tid == 0) {
        for (uint32_t s = 0; s < p.n_stages; s++) {
            mbar_init(&c.full[s], 1);
            mbar_init(&c.empty[s], 1);   // one arrival per tile: the warp that finishes its last slot (finish_slot)
            c.ncand[s] = 0;
            c.done[s] = 0;
        }
        mbar_init(c.imgbar, 1);
        *c.grab = 0;
        *c.kend = 0xFFFFFFFFu;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(c.imgbar, p.image_bytes);
        const uint8_t *src = reinterpret_cast<const uint8_t *>(p.image);
        const uint64_t keep = policy_evict_last();   // every CTA of every scan reads it: it is to stay in L2
        for (uint32_t o = 0; o < p.image_bytes; o += 32768u)
            bulk_g2s(smem + o, src + o, min(32768u, p.image_bytes - o), c.imgbar, keep);
    }
    // up to here nothing was read or written that an earlier kernel on the stream may touch (the image is
    // constant): the kernels before this one -- the previous scan's ordering pass, whoever produced the input --
    // must have finished before the rest
    pdl_wait();
    if (blockIdx.x == 0)
        for (int i = tid; i < kMaxParts; i += kThreads) p.partial_next[i] = 0ull;   // (nobody touches it during this scan)
    __syncthreads();
}
__device__ __forceinline__ void image_wait(const ScanParams &p, const CtlView &c)
{
    mbar_wait<32>(c.imgbar, 0u, &p.ctrl->error_flag, 5u);
}

// The producer role (one lane): streams the CTA's tiles -- blockIdx.x, + gridDim.x, ... : consecutive
// tiles are in flight on different SMs at the same time, a sequential sweep for the DRAM pages, and
// no atomic is needed to hand them out -- into the ring.  Its loop is kept short on purpose: one thread
// runs it, and at 8 KiB per tile every hundred cycles of it cost bandwidth.  A stage is free again when
// the consumer warp that finished the tile's last slot has published the tile's result and arrived on
// its `empty` barrier (finish_slot).
__device__ __forceinline__ void producer_role(const ScanParams &p, const CtlView &c, uint8_t *s_in, uint32_t stride)
{
    const uint32_t n_stages = p.n_stages;
    const uint64_t policy = policy_evict_first();
    const uint32_t want = (uint32_t)kTile + p.halo;
    // interior tiles [t_lo, t_hi): every start of them is a start position and no walk from them can
    // reach the end of the input or a reference walk bound (bit 31 of the tile word: the consumers then
    // skip those checks)
    uint32_t t_lo = 0xFFFFFFFFu, t_hi = 0;
    if (!p.use_ref_bound) {
        t_lo = (p.mis + (uint32_t)kTile - 1u) / (uint32_t)kTile;
        const uint32_t by_valid = p.a_valid_end >= (uint32_t)kTile + p.max_pat_len
                                      ? (p.a_valid_end - (uint32_t)kTile - p.max_pat_len) / (uint32_t)kTile + 1u : 0u;
        t_hi = min(by_valid, p.a_start_end / (uint32_t)kTile);
    }
    uint32_t s = 0, round = 0;
    for (uint32_t t = blockIdx.x;; t += gridDim.x) {
        // the stage's previous tile (one round ago) must be consumed and published
        if (round > 0 && !mbar_wait<PFAC_PROD_SLEEP_NS>(&c.empty[s], (round - 1) & 1u, &p.ctrl->error_flag, 3u)) {
            *reinterpret_cast<volatile uint32_t *>(c.kend) = 0u;   // watchdog tripped: let the consumers go
            return;
        }
        if (t >= p.n_tiles) {
            // sentinel: consumers leave when they see it; kend releases the warps whose slot
            // lies past the sentinel tile (its stage is never filled)
            c.tile[s] = t;
            *reinterpret_cast<volatile uint32_t *>(c.kend) = round * n_stages + s;
            mbar_arrive(&c.full[s]);   // release: orders the stores above
            return;
        }
        c.tile[s] = t | ((t >= t_lo && t < t_hi) ? 0x80000000u : 0u);
        uint8_t *buf = s_in + s * stride;
        const uint32_t a0 = t * (uint32_t)kTile;
        const uint32_t avail = p.a_valid_end - a0;
        const uint32_t nbytes = avail < want ? avail : want;
        const uint32_t nb16 = nbytes & ~15u;
        // last bytes of the input: not a whole 16-byte block, copied by hand and ordered before the
        // barrier's completion with a proxy fence
        if (nb16 < nbytes) {
            for (uint32_t i = nb16; i < nbytes; i++) buf[i] = p.in_al[(size_t)a0 + i];
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        mbar_expect_tx(&c.full[s], nb16);   // release: orders the tile word before the consumers' reads
        if (nb16) bulk_g2s(buf, p.in_al + a0, nb16, &c.full[s], policy);
        if (++s == n_stages) { s = 0; round++; }
    }
}

// End of a slot.  One shared-memory atomic per slot counts the tile's finished slots (low byte) and
// collects the flagged slices (bits 8..): the warp that finishes the tile's last slot publishes the
// tile's result (flag mask, candidate list) to global memory, resets the stage's words and hands the
// stage back to the producer.
template <int SLOTS_PER_TILE>
__device__ __forceinline__ void finish_slot(const ScanParams &p, const CtlView &c, int lane, uint32_t s, uint32_t tile,
                                            uint32_t anym, uint32_t slice0, const uint8_t *buf)
{
    anym = __reduce_or_sync(0xffffffffu, anym);   // (a warp barrier: the lanes' candidate stores precede lane 0's atomic)
    uint32_t old = 0;
    if (lane == 0) old = atoms_add(&c.done[s], 1u + ((anym << slice0) << 8));   // each slot owns its slices' bits
    old = __shfl_sync(0xffffffffu, old, 0);
    if ((old & 255u) != (uint32_t)SLOTS_PER_TILE - 1u) return;
    const uint32_t flags = (old >> 8) | (anym << slice0);
    uint32_t nc = 0, my_cand = 0xFFFFu;
    if (flags) {   // rare: some start of the tile survived every filter
        __threadfence_block();
        nc = *reinterpret_cast<volatile uint32_t *>(&c.ncand[s]);
        if (nc > (uint32_t)kCandPerTile) nc = kCandOverflow;   // too many (or the overflow bit is set)
        if (nc != kCandOverflow && (uint32_t)lane < nc) my_cand = *reinterpret_cast<volatile uint16_t *>(&c.cand[s * kCandPerTile + lane]);
        __syncwarp();
    }
    // one or two candidates and a pattern directory: their bytes are taken along (lane l: bytes l and l + 32)
    const bool by_dir = p.emit.dir != nullptr && nc >= 1u && nc <= (uint32_t)kDirCand;
    uint32_t key0 = 0xFFFFu, key1 = 0xFFFFu, b0_lo = 0, b0_hi = 0, b1_lo = 0, b1_hi = 0;
    if (by_dir) {
        key0 = __shfl_sync(0xffffffffu, my_cand, 0);
        key1 = __shfl_sync(0xffffffffu, my_cand, 1);
        if (key1 < key0) { const uint32_t t = key0; key0 = key1; key1 = t; }
        if ((uint32_t)lane < p.max_pat_len) b0_lo = buf[key0 + lane];
        if ((uint32_t)lane + 32u < p.max_pat_len) b0_hi = buf[key0 + 32u + lane];
        if (key1 != 0xFFFFu) {
            if ((uint32_t)lane < p.max_pat_len) b1_lo = buf[key1 + lane];
            if ((uint32_t)lane + 32u < p.max_pat_len) b1_hi = buf[key1 + 32u + lane];
        }
        __syncwarp();
    }
    if (lane == 0) {
        if (nc == kCandOverflow) {
            p.tile_cnt[tile] = 0u;
            p.tile_nc[tile] = kCandOverflow;
            atomicAdd(&p.ctrl->n_dense, 1u);
        } else {
            if (!flags) p.tile_cnt[tile] = 0u;
            p.tile_nc[tile] = 0u;
        }
        if (flags) c.ncand[s] = 0;
        c.done[s] = 0;
        mbar_arrive(&c.empty[s]);   // release: orders the shared-memory reads and resets above before the refill
    }
    // The walks of the tile's candidates, straight away, by this warp -- AFTER the stage went back to
    // the producer (the walk reads the input and the PHF from global memory: microseconds of dependent
    // loads that must stall one warp, not the ring).
#ifndef PFAC_EXP_NO_EMIT   // (timing experiment: no walks, no records)
    if (lane == 0) PFAC_STAMP(p, 2);
    if (flags && nc != kCandOverflow) {
        if (!by_dir || !emit_tile_dir(p.emit, tile, key0, key1, b0_lo, b0_hi, b1_lo, b1_hi, lane)) emit_tile(p.emit, tile, my_cand, lane);
        if (lane == 0) PFAC_STAMP(p, 3);
    }
#endif
}

// A consumer warp takes the next slot of the CTA's tile sequence and waits for its tile.  Returns
// false when the work has ended.  Slot g belongs to the CTA's k-th tile, k = g / slots per tile:
// stage k % n_stages, phase k / n_stages; a warp leaves on a slot of the sentinel tile or, told by
// kend, on one past it.
template <int SLOTS_PER_TILE>
__device__ __forceinline__ bool take_slot(const ScanParams &p, const CtlView &c, int lane, uint32_t &s, uint32_t &slot_in_tile,
                                          uint32_t &tile)
{
    uint32_t g = 0;
    if (lane == 0) g = atoms_add(c.grab, 1u);
    g = __shfl_sync(0xffffffffu, g, 0);
    const uint32_t k = g / (uint32_t)SLOTS_PER_TILE;
    slot_in_tile = g - k * (uint32_t)SLOTS_PER_TILE;
    const uint32_t round = __umulhi(k, p.stage_magic);   // k / n_stages, exact for k < 2^32 / n_stages
    s = k - round * p.n_stages;
    // the wait suspends the warp in hardware; only when it times out is the end of the work checked
    if (mbar_try_wait(&c.full[s], round & 1u)) goto have_tile;   // the common case: the tile is there already
    for (Watchdog wd;;) {
        if (*reinterpret_cast<volatile uint32_t *>(c.kend) < k) return false;   // a slot past the end of the work
        if (mbar_try_wait_for(&c.full[s], round & 1u, kWaitNs)) break;
        if (wd.expired()) {
            atomicExch(&p.ctrl->error_flag, 2u);
            return false;
        }
    }
have_tile:
    tile = c.tile[s];   // bit 31 = interior flag (producer_role)
    return (tile & 0x7FFFFFFFu) < p.n_tiles;
}

// ---------------------------------------------------------------------------------------------
// Mode 0 detector: all filter tables in shared memory.
//
// Stage 1 probes T1 at EVEN offsets of the input stream only -- 8 LDS.U8 per lane and 16 start
// positions instead of 16.  An even start 2k is judged by the windows at 2k (its bytes 0-1: plane P01)
// and 2k+2 (bytes 2-3: P23); an odd start 2k+1 by the windows at 2k+2 (its bytes 1-2: P12) and 2k+4
// (bytes 3-4: P34).  Patterns too short for the second window pass on the planes Short (<= 3 bytes,
// even starts) and ShortC (<= 4 bytes, odd starts).  The eight T1 bytes of a lane are packed four to
// a register and the two rules evaluated for all of them with funnel shifts.
//
// Stage 2 (per slot, lane-parallel over the compacted survivors): the 4-byte prefix in the
// perfect-hash table of level 1 -> m1; the window that ends the shortest pattern below it keys level 2
// -> m2; the window that ends the shortest pattern of that group in T3.
template <bool HAS_SHORT, bool HAS_SC, bool W3>
__device__ __forceinline__ uint32_t s1_combine(uint32_t X, uint32_t Xn)
{
    if (W3) {
        // with the third-window planes (pfac_derive.h; no Short plane then): an even start 2k also needs P45 of
        // window k+2 unless ShX of window k+1 excuses it, an odd start 2k+1 P56 of window k+3 unless ShX of k+2
        const uint32_t ev = __funnelshift_r(X, Xn, 10) & (__funnelshift_r(X, Xn, 22) | __funnelshift_r(X, Xn, 11));   // -> bit 0
        uint32_t od = __funnelshift_r(X, Xn, 8) & __funnelshift_r(X, Xn, 19) & (__funnelshift_r(X, Xn, 30) | __funnelshift_r(X, Xn, 18));   // -> bit 1
        if (HAS_SC) od |= __funnelshift_r(X, Xn, 12);
        return (X & ev & 0x01010101u) | (od & 0x02020202u);
    }
    // X = T1 bytes of windows k..k+3, Xn = of the four after them.  Result: bit 0 of byte k = even
    // start 2k passes, bit 1 = odd start 2k+1 passes.
    uint32_t b = __funnelshift_r(X, Xn, 10);                       // P23 of window k+1 -> bit 0
    if (HAS_SHORT) b |= X >> 3;                                    // Short of window k -> bit 0
    uint32_t o = __funnelshift_r(X, Xn, 8) & __funnelshift_r(X, Xn, 19);   // P12 of k+1, P34 of k+2 -> bit 1
    if (HAS_SC) o |= __funnelshift_r(X, Xn, 12);                   // ShortC of window k+1 -> bit 1
    return (X & b & 0x01010101u) | (o & 0x02020202u);
}
// the T1 bytes of the 8 even windows of a lane's 16 bytes, four to a register
__device__ __forceinline__ void s1_probe(const uint4 v, uint32_t &X0, uint32_t &X1)
{
    const uint8_t *t1 = smem;
    const uint32_t r0 = rot2x4(v.x), r1 = rot2x4(v.y), r2 = rot2x4(v.z), r3 = rot2x4(v.w);
    const uint32_t e0 = t1[r0 & 0xffffu], e1 = t1[r0 >> 16], e2 = t1[r1 & 0xffffu], e3 = t1[r1 >> 16];
    const uint32_t e4 = t1[r2 & 0xffffu], e5 = t1[r2 >> 16], e6 = t1[r3 & 0xffffu], e7 = t1[r3 >> 16];
    X0 = e0 + (e1 << 8) + (e2 << 16) + (e3 << 24);
    X1 = e4 + (e5 << 8) + (e6 << 16) + (e7 << 24);
}
// unaligned 32-bit read of the staged tile
__device__ __forceinline__ uint32_t load_w4(const uint8_t *buf, uint32_t pos)
{
    const uint32_t *wp = reinterpret_cast<const uint32_t *>(buf + (pos & ~3u));
    return __funnelshift_r(wp[0], wp[1], (pos & 3u) * 8u);
}

// Stage 1 over two consecutive slices (1 KiB, `pair` = tile-relative offset of the lane's 16 bytes in
// the lower one): bit 16 h + j of the result = start j of this lane in slice h passed.  The upper
// slice goes first: the T1 bytes of the two windows after a lane's 16 bytes are the next lane's first
// two -- for lane 31 those of lane 0 in the slice above (lane 31 of the upper slice looks them up itself).
// `above` (HAS_ABOVE): the first T1 register of the slice after the pair, already probed by the caller (the
// slot's pairs go top down), so that only the slot's last slice pays lane 31's own look-ups; x0_out = this
// pair's lower slice's, for the pair below.
template <bool HAS_SHORT, bool HAS_SC, bool W3, bool HAS_ABOVE>
__device__ __forceinline__ uint32_t s1_pair(const uint8_t *buf, uint32_t pair, int lane, uint32_t next_lane, uint32_t above, uint32_t &x0_out)
{
    const uint4 v1 = *reinterpret_cast<const uint4 *>(buf + pair + kSlice);
    const uint4 v0 = *reinterpret_cast<const uint4 *>(buf + pair);
#ifdef PFAC_EXP_NO_S1   // timing experiment: the streaming skeleton alone
    x0_out = above;
    return ((v0.x ^ v1.y) + (v0.z ^ v1.w)) == 0x12345679u ? 1u : 0u;
#endif
    uint32_t X0, X1, Y0, Y1;
    s1_probe(v1, Y0, Y1);
    s1_probe(v0, X0, X1);
    x0_out = X0;
    uint32_t ey = __shfl_sync(0xffffffffu, HAS_ABOVE && lane == 0 ? above : Y0, next_lane);
    if (!HAS_ABOVE && lane == 31) {
        const uint32_t r = rot2x4(*reinterpret_cast<const uint32_t *>(buf + pair + kSlice + 16));
        ey = (uint32_t)smem[r & 0xffffu] | ((uint32_t)smem[r >> 16] << 8);
        if (W3) ey |= (uint32_t)smem[rot2x4(*reinterpret_cast<const uint32_t *>(buf + pair + kSlice + 20)) & 0xffffu] << 16;   // (one window more)
    }
    const uint32_t ex = __shfl_sync(0xffffffffu, lane == 0 ? Y0 : X0, next_lane);
    const uint32_t q0 = s1_combine<HAS_SHORT, HAS_SC, W3>(X0, X1) * 0x01041040u;
    const uint32_t q1 = s1_combine<HAS_SHORT, HAS_SC, W3>(X1, ex) * 0x01041040u;
    const uint32_t q2 = s1_combine<HAS_SHORT, HAS_SC, W3>(Y0, Y1) * 0x01041040u;
    const uint32_t q3 = s1_combine<HAS_SHORT, HAS_SC, W3>(Y1, ey) * 0x01041040u;
    // byte 3 of each product = the 8 results in start order
    return __byte_perm(__byte_perm(q0, q1, 0x0073), __byte_perm(q2, q3, 0x0073), 0x5410);
}

constexpr int kSlotSlices2 = slot_slices(0);   // slices per slot of the mode-0 detector (2 or 4)
static_assert(kSlotSlices2 % 2 == 0 && kSlicesPerTile % kSlotSlices2 == 0, "slots are made of slice pairs");
constexpr int kQ2Cap = q1_cap(0);              // survivors a slot's queue holds; a slot with more is handed over whole

template <bool HAS_SHORT, bool HAS_SC, bool W3>
__global__ void __launch_bounds__(kThreads, 1) pfac_scan2_kernel(const ScanParams p)
{
    constexpr int kSlotSlices = kSlotSlices2, kSlotsPerTile = kSlicesPerTile / kSlotSlices;
    constexpr int kQueueBytes = kQ2Cap * 2;
    uint8_t *ctl = smem + p.image_bytes;
    const CtlView c = ctl_view(ctl);
    uint8_t *qbase = ctl + kCtrlBytes;
    uint8_t *s_in = qbase + kConsumerWarps * kQueueBytes;
    const uint32_t stride = scan_buf_stride(p.halo);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    detector_init(p, c);
    if (warp == kConsumerWarps) {
        if (lane == 0) producer_role(p, c, s_in, stride);
        return;
    }
    image_wait(p, c);
    if (tid == 0) PFAC_STAMP(p, 1);

    const uint16_t *s_d1 = reinterpret_cast<const uint16_t *>(smem + p.off_d1);
    const uint16_t *s_e1 = reinterpret_cast<const uint16_t *>(smem + p.off_e1);
    const uint16_t *s_d2 = reinterpret_cast<const uint16_t *>(smem + p.off_d2);
    const uint16_t *s_e2 = reinterpret_cast<const uint16_t *>(smem + p.off_e2);
    const uint32_t *s_t3 = reinterpret_cast<const uint32_t *>(smem + p.off_t3);
    uint16_t *wq = reinterpret_cast<uint16_t *>(qbase + warp * kQueueBytes);   // stage-1 survivors of the slot
    const uint32_t next_lane = (lane + 1) & 31;

    for (;;) {
        uint32_t s, slot_in_tile, tinfo;
        if (!take_slot<kSlotsPerTile>(p, c, lane, s, slot_in_tile, tinfo)) break;
        const uint32_t tile = tinfo & 0x7FFFFFFFu;
        const bool interior = (tinfo >> 31) != 0;   // every start of the tile counts, no walk reaches the end of the input
        const uint32_t slice0 = slot_in_tile * (uint32_t)kSlotSlices;
        const uint8_t *buf = s_in + s * stride;
        const uint32_t a0 = tile * (uint32_t)kTile;
        const uint32_t valid_t = p.a_valid_end - a0;   // tile-relative end of readable input (may exceed the buffer)
        // ---- stage 1 of all the slot's slice pairs (their T1 probes overlap), then the compaction: the
        // lanes' survivor counts are scanned across the warp and every lane writes its own into the queue
        constexpr int kPairs = kSlotSlices / 2;
        uint32_t m[kPairs];
        const uint32_t base = slice0 * kSlice + lane * 16;   // tile-relative position of the lane's first start
        {
            uint32_t x0 = 0;
            m[kPairs - 1] = s1_pair<HAS_SHORT, HAS_SC, W3, false>(buf, base + (kPairs - 1) * 2 * kSlice, lane, next_lane, 0u, x0);
#pragma unroll
            for (int pr = kPairs - 2; pr >= 0; pr--) m[pr] = s1_pair<HAS_SHORT, HAS_SC, W3, true>(buf, base + pr * 2 * kSlice, lane, next_lane, x0, x0);
        }
        if (!interior) {   // start positions are [mis, a_start_end) in aligned coordinates
#pragma unroll
            for (int h = 0; h < kSlotSlices; h++) {
                const uint32_t a = a0 + base + h * kSlice;
                const uint32_t first = p.mis > a ? p.mis - a : 0u;
                const uint32_t last = p.a_start_end > a ? p.a_start_end - a : 0u;
                uint32_t keep = last >= 16u ? 0xffffu : ((1u << last) - 1u);
                keep &= first >= 16u ? 0u : (0xffffu << first);
                m[h >> 1] &= ~(0xffffu << (16 * (h & 1))) | ((keep & 0xffffu) << (16 * (h & 1)));
            }
        }
        uint32_t cnt = 0;
#pragma unroll
        for (int pr = 0; pr < kPairs; pr++) cnt += __popc(m[pr]);
        uint32_t incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        uint32_t nq = __shfl_sync(0xffffffffu, incl, 31), anym = 0;
        if (nq <= (uint32_t)kQ2Cap) {
            uint16_t *wp = wq + (incl - cnt);
#pragma unroll
            for (int pr = 0; pr < kPairs; pr++) {
                uint32_t mm = m[pr];
                const uint32_t pb = base + pr * 2 * kSlice;
                while (mm) {
                    const uint32_t b = __ffs(mm) - 1;
                    mm &= mm - 1;
                    *wp++ = (uint16_t)(pb + b + (b >> 4) * (kSlice - 16));
                }
            }
        }
        if (nq > (uint32_t)kQ2Cap) {   // dense slot: the dense-match kernel looks at the whole tile
            anym = (1u << kSlotSlices) - 1u;
            if (lane == 0) atomicOr(c.ncand + s, 0x80000000u);
            nq = 0;
        }
        __syncwarp();
#ifdef PFAC_EXP_NO_S2   // timing experiment: stage 1 and the compaction alone
        if (nq < 100000u) nq = 0;
#endif
        // ---- stage 2
        uint32_t e0 = 0;
#ifndef PFAC_S2_BRANCHY
        // The common case -- an interior tile of a set without short patterns and with both key levels --
        // as straight-line, predicated code: a lane whose start is already rejected runs on with harmless
        // addresses instead of branching out (some lane of the warp goes the whole way anyway), and two
        // queue entries per lane are judged at a time, so that the two chains of dependent look-ups
        // (prefix -> m1 -> window -> m2 -> window -> T3) overlap.
        if (!HAS_SHORT && interior && p.ns2) {
            auto judge = [&](const uint32_t (&tp)[2], const bool (&live)[2], int K) {
                uint32_t w4[2], m1[2], w1[2], key2[2], m2[2], w2[2];
                bool ok[2];
#pragma unroll
                for (int k = 0; k < 2; k++) if (k < K) w4[k] = load_w4(buf, tp[k]);
#pragma unroll
                for (int k = 0; k < 2; k++) if (k < K) m1[k] = ph_lookup(s_d1, s_e1, p.nb1, p.ns1, w4[k], ph_mix(w4[k]));
#pragma unroll
                for (int k = 0; k < 2; k++) if (k < K) {
                    ok[k] = live[k] && m1[k] != 0u;          // (interior: tpos + m <= tpos + max_pat_len always holds)
                    w1[k] = load_w4(buf, ok[k] ? tp[k] + m1[k] - 4u : 0u);   // (rejected lanes read one broadcast word: no bank conflicts from them)
                    key2[k] = hash_key2(w4[k], w1[k]);
                }
#pragma unroll
                for (int k = 0; k < 2; k++) if (k < K) m2[k] = ph_lookup(s_d2, s_e2, p.nb2, p.ns2, key2[k], key2[k]);
#pragma unroll
                for (int k = 0; k < 2; k++) if (k < K) {
                    ok[k] = ok[k] && m2[k] != 0u;
                    w2[k] = load_w4(buf, ok[k] ? tp[k] + m2[k] - 4u : 0u);
                    const uint32_t h4 = ok[k] ? hash_t3(key2[k] ^ kT3Seed2, w2[k]) >> p.t3_shift : 0u;
                    ok[k] = ok[k] && ((s_t3[h4 >> 5] >> (h4 & 31u)) & 1u);
                }
#pragma unroll
                for (int k = 0; k < 2; k++)
                    if (k < K && ok[k]) {   // rare
                        anym |= 1u << (tp[k] / (uint32_t)kSlice - slice0);
                        add_candidate(c.ncand + s, c.cand + s * kCandPerTile, tp[k]);
                    }
            };
            for (; e0 < nq; e0 += 64) {
                const uint32_t ea = e0 + lane, eb = e0 + 32 + lane;
                const bool live[2] = {ea < nq, eb < nq};
                const uint32_t tp[2] = {live[0] ? (uint32_t)wq[ea] : 0u, live[1] ? (uint32_t)wq[eb] : 0u};
                if (e0 + 32 < nq) judge(tp, live, 2);
                else judge(tp, live, 1);
            }
        }
#endif
        for (; e0 < nq; e0 += 32) {
            const uint32_t e = e0 + lane;
            if (e >= nq) continue;
            const uint32_t tpos = wq[e];
            bool keep = true;
            if (tpos + 4u <= valid_t) {   // else: settled as a candidate
                const uint32_t w4 = load_w4(buf, tpos);
                bool shortp = false;
                if (HAS_SHORT) {   // starts of patterns that are not in the prefix tables
                    const uint32_t r = rot2x4(w4);
                    shortp = (tpos & 1u) ? (smem[(r >> 8) & 0xffffu] & kT1ShortC) != 0 : (smem[r & 0xffffu] & kT1Short) != 0;
                }
                if (!shortp) {
                    const uint32_t m1 = ph_lookup(s_d1, s_e1, p.nb1, p.ns1, w4, ph_mix(w4));   // 0 = no pattern has this prefix
                    const uint32_t lim = interior ? tpos + p.max_pat_len : walk_limit(p, a0, tpos);   // never past the staged halo
                    keep = m1 != 0 && tpos + m1 <= lim;
                    if (keep) {
                        const uint32_t w1 = load_w4(buf, tpos + m1 - 4u);
                        if (!p.ns2) {
                            const uint32_t h3 = hash_t3(w4, w1) >> p.t3_shift;
                            keep = (s_t3[h3 >> 5] >> (h3 & 31u)) & 1u;
                        } else {
                            const uint32_t key2 = hash_key2(w4, w1);
                            const uint32_t m2 = ph_lookup(s_d2, s_e2, p.nb2, p.ns2, key2, key2);   // 0 = no such group
                            keep = m2 != 0 && tpos + m2 <= lim;
                            if (keep) {
                                const uint32_t w2 = load_w4(buf, tpos + m2 - 4u);
                                const uint32_t h4 = hash_t3(key2 ^ kT3Seed2, w2) >> p.t3_shift;
                                keep = (s_t3[h4 >> 5] >> (h4 & 31u)) & 1u;
                            }
                        }
                    }
                }
            }
            if (keep) {
                anym |= 1u << (tpos / (uint32_t)kSlice - slice0);
                add_candidate(c.ncand + s, c.cand + s * kCandPerTile, tpos);
            }
        }
        finish_slot<kSlotsPerTile>(p, c, lane, s, tile, anym, slice0, buf);
    }
    if (lane == 0) PFAC_STAMP(p, 4);
}

// The detector of the modes without shared-memory two-point tables.  MODE 0 here: stage 1 = T1 (one
// probe per start), stage 2 = T2 (mode 1 of pfac_derive.h: sets whose automaton is not a tree, or
// with short patterns and too many prefixes).  MODE 2: stage 1 = T2 (the whole shared image),
// Tm / Tm2 / T3 in global memory.
template <int MODE>
__global__ void __launch_bounds__(kThreads, 1) pfac_scan_kernel(const ScanParams p)
{
    const uint32_t *s_t2 = reinterpret_cast<const uint32_t *>(smem + p.off_t2);
    const uint8_t *tab = MODE == 2 ? p.gimage : smem;   // where Tm / Tm2 / T3 live
    const uint16_t *s_tm = reinterpret_cast<const uint16_t *>(tab + p.off_tm);
    const uint16_t *s_tm2 = reinterpret_cast<const uint16_t *>(tab + p.off_tm2);
    const uint32_t *s_t3 = reinterpret_cast<const uint32_t *>(tab + p.off_t3);
    uint8_t *ctl = smem + p.image_bytes;
    const CtlView c = ctl_view(ctl);
    uint32_t *s_ncand = c.ncand;
    uint16_t *s_cand = c.cand;
    uint8_t *qbase = ctl + kCtrlBytes;
    constexpr int kSlotSlices = slot_slices(MODE), kSlotsPerTile = kSlicesPerTile / kSlotSlices;
    constexpr int kQ1Cap = q1_cap(MODE), kQueueBytes = queue_bytes(MODE);
    uint8_t *s_in = qbase + kConsumerWarps * kQueueBytes;
    const uint32_t stride = scan_buf_stride(p.halo);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    detector_init(p, c);
    if (warp == kConsumerWarps) {
        if (lane == 0) producer_role(p, c, s_in, stride);
        return;
    }
    image_wait(p, c);

    // ---------------------------------------------------------------------- consumers
    // Slots (kSlotSlices consecutive slices) are not bound to warps: the CTA's tiles form one sequence
    // of slots and a warp that is done takes the next one, so a warp the scheduler favours (or one
    // whose slots have few survivors) simply does more of them instead of spinning on the ring behind
    // the slowest warp.  Slot g belongs to the CTA's k-th tile, k = g / kSlotsPerTile: stage
    // k % n_stages, phase k / n_stages.  A warp leaves on a slot of the sentinel tile or, told by
    // s_kend, on one past it.
    uint16_t *wq = reinterpret_cast<uint16_t *>(qbase + warp * kQueueBytes);   // stage-1 survivors of the slot

    for (;;) {
        uint32_t s, slot_in_tile, tile;
        if (!take_slot<kSlotsPerTile>(p, c, lane, s, slot_in_tile, tile)) break;
        tile &= 0x7FFFFFFFu;
        const uint32_t slice0 = slot_in_tile * (uint32_t)kSlotSlices;   // first slice of the slot
        const uint8_t *buf = s_in + s * stride;
        const uint32_t a0 = tile * (uint32_t)kTile;
        const uint32_t valid_t = p.a_valid_end - a0;   // tile-relative end of readable input (may exceed the buffer)
        // an interior tile: every start of it is a start position and none can reach the end of the
        // input or a reference walk bound
        const bool interior = !p.use_ref_bound && a0 >= p.mis && valid_t >= (uint32_t)kTile + p.max_pat_len &&
                              a0 + (uint32_t)kTile <= p.a_start_end;
        uint32_t anym = 0;   // bit h: slice slice0 + h has a start that survived
        // stage 1 of all the slot's slices: T1 (or, in global mode, T2) over 16 positions per lane and slice ->
        // one 16-bit mask per slice (bit j: start j of the lane's 16 bytes passed)
        uint32_t m16[kSlotSlices];
#pragma unroll
        for (int h = 0; h < kSlotSlices; h++) {
            m16[h] = 0u;
            const uint32_t off = (slice0 + h) * kSlice + lane * 16;
            if (a0 + (slice0 + h) * kSlice >= p.a_start_end) continue;   // (uniform) no start positions from here on
            const uint4 v = *reinterpret_cast<const uint4 *>(buf + off);
            // the 4 bytes after the lane's 16 are the next lane's first word (a strided shared-memory
            // read of them would be a 4-way bank conflict); lane 31 reads its own
            uint32_t nx = __shfl_down_sync(0xffffffffu, v.x, 1);
            if (lane == 31) nx = *reinterpret_cast<const uint32_t *>(buf + off + 16);
            uint32_t m = 0;
            if (!(p.debug & 4u)) {
                if (MODE == 2) {
                    m = filter16_t2(v, nx, s_t2, p.t2_shift);
                } else {
                    uint32_t lo = 0, hi = 0;   // one nibble per start, bit 0 = passes stage 1
                    filter16(v, nx, lane, lo, hi);
                    m = nibble_bits(lo) | (nibble_bits(hi) << 8);
                }
            }
            if (p.debug & 16u) {   // diagnostics: stage 1 alone (its result is consumed, nothing survives)
                if (m == 0x9e37u) anym |= 1u << h;
                m = 0;
            }
            if (!interior) {   // start positions are [mis, a_start_end) in aligned coordinates
                const uint32_t a = a0 + off;
                const uint32_t first = p.mis > a ? p.mis - a : 0u;
                const uint32_t last = p.a_start_end > a ? p.a_start_end - a : 0u;
                uint32_t keep = last >= 16u ? 0xffffu : ((1u << last) - 1u);
                keep &= first >= 16u ? 0u : (0xffffu << first);
                m &= keep;
            }
            m16[h] = m;
        }
        // compaction: the lanes' survivor counts are scanned across the warp and every lane writes its own
        // into the queue (order irrelevant: the candidates are sorted where it matters)
        uint32_t cnt = 0;
#pragma unroll
        for (int h = 0; h < kSlotSlices; h++) cnt += __popc(m16[h]);
        uint32_t incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        uint32_t nq = __shfl_sync(0xffffffffu, incl, 31);
        if (nq <= (uint32_t)kQ1Cap) {
            uint16_t *wp = wq + (incl - cnt);
#pragma unroll
            for (int h = 0; h < kSlotSlices; h++) {
                const uint32_t pb = (slice0 + h) * kSlice + lane * 16;
                for (uint32_t mm = m16[h]; mm; mm &= mm - 1) *wp++ = (uint16_t)(pb + __ffs(mm) - 1);
            }
        }
        if (nq > (uint32_t)kQ1Cap) {   // dense slot: the dense-match kernel looks at the whole tile
            anym = (1u << kSlotSlices) - 1u;
            if (lane == 0) atomicOr(s_ncand + s, 0x80000000u);
            nq = 0;
        }
        __syncwarp();
        // stage 2: the 4-byte prefix (complete Tm, or T2), then the two-point checks -- every pattern
        // under a key is at least m bytes long and has its bytes [m-4, m) in T3.  Starts that cannot
        // be judged here (short patterns, end of the input) are candidates straight away.
        for (uint32_t e0 = 0; e0 < nq; e0 += 32) {
            const uint32_t e = e0 + lane;
            if (e >= nq) continue;
            const uint32_t tpos = wq[e];
            bool keep = true;
            if (!(p.debug & 8u) && tpos + 4u <= valid_t) {
                const uint32_t *wp = reinterpret_cast<const uint32_t *>(buf + (tpos & ~3u));
                const uint32_t w4 = __funnelshift_r(wp[0], wp[1], (tpos & 3u) * 8u);
                bool shortp = false;
                if (MODE != 2 && p.has_short) shortp = (smem[rot2x4(w4) & 0xffffu] & kT1Short) != 0;
                if (!shortp) {
                    if (!p.has_t3) {
                        keep = t2_pass(s_t2, w4, p.t2_shift);
                    } else {
                        const uint32_t m1 = tm_lookup(s_tm, w4, p.tm_bits);   // 0 = no pattern has this prefix
                        const uint32_t lim = interior ? tpos + p.max_pat_len : walk_limit(p, a0, tpos);   // never past the staged halo
                        keep = m1 != 0 && tpos + m1 <= lim;
                        if (keep) {
                            const uint32_t wo = tpos + m1 - 4u;
                            const uint32_t *we = reinterpret_cast<const uint32_t *>(buf + (wo & ~3u));
                            const uint32_t w1 = __funnelshift_r(we[0], we[1], (wo & 3u) * 8u);
                            const uint32_t h3 = hash_t3(w4, w1) >> p.t3_shift;
                            keep = (s_t3[h3 >> 5] >> (h3 & 31u)) & 1u;
                            if (keep && p.tm2_bits) {
                                const uint32_t key2 = hash_key2(w4, w1);
                                const uint32_t m2 = tm_lookup(s_tm2, key2, p.tm2_bits);   // 0 = no such group
                                keep = m2 != 0 && tpos + m2 <= lim;
                                if (keep) {
                                    const uint32_t wo2 = tpos + m2 - 4u;
                                    const uint32_t *wf = reinterpret_cast<const uint32_t *>(buf + (wo2 & ~3u));
                                    const uint32_t w2 = __funnelshift_r(wf[0], wf[1], (wo2 & 3u) * 8u);
                                    const uint32_t h4 = hash_t3(key2 ^ kT3Seed2, w2) >> p.t3_shift;
                                    keep = (s_t3[h4 >> 5] >> (h4 & 31u)) & 1u;
                                }
                            }
                        }
                    }
                }
            }
            if (keep) {
                anym |= 1u << (tpos / (uint32_t)kSlice - slice0);
                add_candidate(s_ncand + s, s_cand + s * kCandPerTile, tpos);
            }
        }
        finish_slot<kSlotsPerTile>(p, c, lane, s, tile, anym, slice0, buf);
    }
}

// ---------------------------------------------------------------------------------------------
// Dense-match pass: the tiles the detector handed over whole (too many candidates: inputs where a
// large share of the start positions match, e.g. a dictionary over English text -- the reference's
// own fixtures).  One CTA per such tile; every start position of the tile is walked as SUBSEG_MATCH
// does (master_kernel.cu:37-74), but
//   * the tile and its halo are staged in shared memory, so the walks read LDS, not global bytes;
//   * the first levels of the trie come from the walk cache (pfac_derive.h: the root row and an exact
//     perfect-hash map of every 2- and 3-byte path) in shared memory; only deeper steps go through
//     r[] / {HT,val} (read-only path, L1/L2);
//   * ONE sweep: each start leaves its match count and its first two final states in shared memory;
//     a block scan over the counts gives every start its place in the tile's record run, which is
//     reserved in the arrival-order scratch with one atomic and written from the stored states
//     (starts with more than two matches are walked again, writing directly).
// Records of a tile come out in (position, pattern length) order; the ordering pass moves the run
// into place like those of the detector.
struct DenseParams {
    EmitParams e;
    const uint8_t *wc_image;    // walk cache image (global); copied to shared memory per CTA
    uint32_t wc_bytes, wc_depth, wc_off_d, wc_off_e, wc_nb, wc_ns;
    uint32_t halo;              // staged halo bytes (multiple of 16, >= max_pat_len - 1)
    const unsigned int *n_dense;   // tiles the detector handed over whole (0: nothing to do)
    // DIRECT mode (no detector ran: pattern sets with patterns of <= 3 bytes match densely) -- the kernel is
    // the whole scan: tiles are taken in ticket order, a chained prefix over the tiles' totals (the
    // scan-then-propagate of a single-pass prefix sum) gives every tile its place in `out`
    uint2 *out;
    unsigned long long cap;
    unsigned long long *prefix;    // [n_tiles] status words of the look-back: epoch << 40 | flag << 38 | records
    uint32_t epoch;                // 1 .. 2^24-1, differs from that of the slot's previous scans
    Result *result;
    unsigned long long *count_out;
};

constexpr int kDenseThreads = 1024;
constexpr int kDensePer = kTile / kDenseThreads;   // consecutive starts a thread owns in the write pass
static_assert(kTile % kDenseThreads == 0 && kSlice % kDensePer == 0 && kSlicesPerTile <= 32, "dense pass ownership");

__host__ inline size_t dense_smem_bytes(uint32_t wc_bytes, uint32_t halo)
{
    // walk cache | text (tile + halo + 16) | cnt u16[kTile] | fin i32[2][kTile] | queues uint2[kTile] | scan scratch | tile list u32[1024]
    return (size_t)((wc_bytes + 127u) & ~127u) + ((kTile + halo + 16 + 127u) & ~127u) + (size_t)kTile * 2 + (size_t)kTile * 8 +
           (size_t)kTile * 8 + 512 + 4 * 1024;
}

template <bool DIRECT>
__global__ void __launch_bounds__(kDenseThreads, 1) pfac_dense_kernel(const DenseParams d)
{
    if (!DIRECT) {
        pdl_launch_next();
        pdl_wait();   // the detector has finished
        if (*reinterpret_cast<const volatile unsigned int *>(d.n_dense) == 0u) return;   // the common case: sparse matches, nothing was handed over
    }
    const EmitParams &p = d.e;
    const uint32_t wcb = (d.wc_bytes + 127u) & ~127u;
    const int32_t *s_s0 = reinterpret_cast<const int32_t *>(smem);
    const uint16_t *s_d = reinterpret_cast<const uint16_t *>(smem + d.wc_off_d);
    const uint2 *s_e = reinterpret_cast<const uint2 *>(smem + d.wc_off_e);
    uint8_t *s_text = smem + wcb;
    const uint32_t text_bytes = (kTile + d.halo + 16 + 127u) & ~127u;
    uint16_t *s_cnt = reinterpret_cast<uint16_t *>(s_text + text_bytes);
    int32_t *s_fin = reinterpret_cast<int32_t *>(s_text + text_bytes + kTile * 2);   // [2][kTile] first final states of a start ...
    uint16_t *s_fin16 = reinterpret_cast<uint16_t *>(s_fin);                          // ... or [4][kTile] when they fit 16 bits
    const bool fin16 = p.n_final <= 65536;
    const uint32_t fin_keep = fin16 ? 4u : 2u;
    uint2 *s_q = reinterpret_cast<uint2 *>(s_text + text_bytes + kTile * 2 + kTile * 8);         // [kTile] the warps' queues of live walks
    uint32_t *s_scan = reinterpret_cast<uint32_t *>(s_text + text_bytes + kTile * 2 + kTile * 16);   // [0..31] warp offsets, [32] total, [33..34] base, [36] ticket
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    // where the records go: the arrival-order scratch (ordered later), or straight to the caller's buffer
    uint2 *const dst = DIRECT ? d.out : p.scratch;
    const unsigned long long dst_cap = DIRECT ? d.cap : p.scratch_cap;

    if (DIRECT) pdl_launch_next();
    for (uint32_t i = tid; i < d.wc_bytes / 16; i += kDenseThreads)
        reinterpret_cast<uint4 *>(smem)[i] = __ldg(reinterpret_cast<const uint4 *>(d.wc_image) + i);
    if (DIRECT) pdl_wait();   // the walk cache (constant) is on its way; everything else waits for the kernels before

    // the cached transition: state after (b0 .. b_{depth-1}) or -1
    auto cached = [&](uint32_t key) -> int32_t {
        const uint32_t dd = s_d[mulhi32(ph_mix(key), d.wc_nb)];
        const uint2 e = s_e[ph_slot(key, dd, d.wc_ns)];
        return e.x == key ? (int32_t)e.y : -1;
    };
    // tile-relative walk bound of the start at aligned coordinate a: end of the input, the reference's
    // 4096+512 tile bound (master_kernel.cu:141-144), max_pat_len bytes
    auto limit_t = [&](uint32_t a, uint32_t a0) -> uint32_t {
        uint32_t lim_a = p.a_valid_end;
        if (p.use_ref_bound) {
            const unsigned long long gpos = p.base_pos + (unsigned long long)(a - p.mis);
            const unsigned long long lim2 = ((gpos & ~4095ull) + 4608ull) - p.base_pos + p.mis;
            if (lim2 < lim_a) lim_a = (uint32_t)lim2;
        }
        const unsigned long long depth = (unsigned long long)a + p.max_pat_len;
        if (depth < lim_a) lim_a = (uint32_t)depth;
        return lim_a - a0;
    };
    // SUBSEG_MATCH for one start, writing its records at dst[o ...] (starts with more than two matches)
    auto walk_write = [&](uint32_t t0, uint32_t a, uint32_t lim_t, unsigned long long o) {
        const uint32_t rec_pos = a - p.mis + p.pos_bias;
        uint32_t n = 0;
        int32_t state = s_s0[s_text[t0]];                             // :41
        for (uint32_t q = t0 + 1; state >= 0; q++) {
            if (state < p.n_final) {                                  // :44-47, :67-70
                if (o + n < dst_cap) dst[o + n] = make_uint2(rec_pos, (uint32_t)ldg_keep(&p.idmap[state]));
                n++;
            }
            if (q >= lim_t) break;                                    // :50
            state = phf_next(p, state, s_text[q]);                    // :52-64
        }
    };

    // Which tiles: DIRECT -- all, in ticket order (a tile only ever waits for tiles that running CTAs
    // hold); otherwise the CTA's share (blockIdx.x, + gridDim.x, ...) of the tiles the detector handed
    // over, found kDenseThreads at a time (one tile_nc word per thread) and listed in shared memory.
    uint32_t *s_list = s_scan + 64;   // [kDenseThreads]
    uint32_t chunk = 0, li = 0, ln = 0;
    for (;;) {
        __syncthreads();   // the previous tile's arrays are free (and, the first time, the walk cache is in place)
        uint32_t tile;
        if (DIRECT) {
            if (tid == 0) s_scan[36] = atomicAdd(&p.ctrl->ticket, 1u);
            __syncthreads();
            tile = s_scan[36];
            if (tile >= p.n_tiles) break;
        } else {
            while (li == ln) {   // (uniform) the list is used up: look at the next kDenseThreads tiles of the share
                const uint64_t first = (uint64_t)blockIdx.x + (uint64_t)chunk * kDenseThreads * gridDim.x;
                if (first >= p.n_tiles) break;
                if (tid == 0) s_scan[37] = 0;
                __syncthreads();
                const uint64_t t = first + (uint64_t)tid * gridDim.x;
                if (t < p.n_tiles && p.tile_nc[t] == kCandOverflow) s_list[atomicAdd(&s_scan[37], 1u)] = (uint32_t)t;
                __syncthreads();
                ln = s_scan[37];
                li = 0;
                chunk++;
                __syncthreads();
            }
            if (li == ln) break;
            tile = s_list[li++];
        }
        const uint32_t a0 = tile * (uint32_t)kTile;
        // ---- stage the tile and its halo (16-byte loads; nothing past the readable input)
        const uint32_t avail = p.a_valid_end - a0;
        const uint32_t nbytes = min(avail, (uint32_t)kTile + d.halo);
        for (uint32_t i = tid; i < (nbytes + 15) / 16; i += kDenseThreads) {
            const uint32_t off = i * 16;
            if (off + 16 <= nbytes) {
                reinterpret_cast<uint4 *>(s_text)[i] = __ldg(reinterpret_cast<const uint4 *>(p.in_al + a0) + i);
            } else {
                for (uint32_t k = off; k < nbytes; k++) s_text[k] = p.in_al[(size_t)a0 + k];
            }
        }
        __syncthreads();
        // ---- the sweep, level by level: a warp owns kTile/32 consecutive starts.  Walking them start by
        // start leaves most lanes idle (walks end at different depths); instead the warp keeps a queue
        // of the walks that are still alive and advances ALL of them one byte per pass -- every pass is
        // dense, 32 walks at a time, and runs the code of one trie level only.  A queue entry is
        // (start | walk bound << 16, state); a final state met bumps the start's count and, for the
        // first two, is kept for the write pass.
        {
            constexpr int kPerWarp = kTile / (kDenseThreads / 32);
            uint2 *q = s_q + warp * kPerWarp;
            const uint32_t w0 = warp * kPerWarp;
            auto record = [&](uint32_t t0, int32_t st) {              // :44-47, :67-70
                if (st < p.n_final) {
                    const uint32_t n = s_cnt[t0];
                    if (fin16) { if (n < 4u) s_fin16[n * kTile + t0] = (uint16_t)st; }
                    else if (n < 2u) s_fin[n * kTile + t0] = st;
                    s_cnt[t0] = (uint16_t)(n + 1u);
                }
            };
            // compaction of a pass's survivors (in place: the write index never passes the batch just read)
            auto push = [&](bool alive, uint32_t &nw, uint2 it) {
                const uint32_t bal = __ballot_sync(0xffffffffu, alive);
                if (alive) q[nw + __popc(bal & lt_mask)] = it;
                nw += __popc(bal);
            };
            uint32_t nq = 0;
            // level 0: the root row (:41-43)
            for (uint32_t e = 0; e < (uint32_t)kPerWarp; e += 32) {
                const uint32_t t0 = w0 + e + lane, a = a0 + t0;
                bool alive = false;
                uint2 it = make_uint2(0u, 0u);
                s_cnt[t0] = 0;
                if (a >= p.mis && a < p.a_start_end) {
                    const int32_t st = s_s0[s_text[t0]];
                    if (st >= 0) {
                        record(t0, st);
                        const uint32_t lim = limit_t(a, a0);
                        alive = t0 + 1u < lim;                        // :50
                        it = make_uint2(t0 | (lim << 16), (uint32_t)st);
                    }
                }
                push(alive, nq, it);
            }
            __syncwarp();
            uint32_t dep = 1;
            if (d.wc_depth >= 2) {   // level 1 from the walk cache
                uint32_t nw = 0;
                for (uint32_t e = 0; e < nq; e += 32) {
                    const bool have = e + lane < nq;
                    uint2 it = have ? q[e + lane] : make_uint2(0u, 0u);
                    __syncwarp();
                    bool alive = false;
                    if (have) {
                        const uint32_t t0 = it.x & 0xffffu;
                        const int32_t st = cached((uint32_t)s_text[t0] | ((uint32_t)s_text[t0 + 1] << 8) | kWalkDepth2);
                        if (st >= 0) {
                            record(t0, st);
                            it.y = (uint32_t)st;
                            alive = t0 + 2u < (it.x >> 16);
                        }
                    }
                    push(alive, nw, it);
                }
                __syncwarp();
                nq = nw;
                dep = 2;
                if (d.wc_depth >= 3) {   // level 2 from the walk cache
                    nw = 0;
                    for (uint32_t e = 0; e < nq; e += 32) {
                        const bool have = e + lane < nq;
                        uint2 it = have ? q[e + lane] : make_uint2(0u, 0u);
                        __syncwarp();
                        bool alive = false;
                        if (have) {
                            const uint32_t t0 = it.x & 0xffffu;
                            const int32_t st = cached((uint32_t)s_text[t0] | ((uint32_t)s_text[t0 + 1] << 8) |
                                                      ((uint32_t)s_text[t0 + 2] << 16) | kWalkDepth3);
                            if (st >= 0) {
                                record(t0, st);
                                it.y = (uint32_t)st;
                                alive = t0 + 3u < (it.x >> 16);
                            }
                        }
                        push(alive, nw, it);
                    }
                    __syncwarp();
                    nq = nw;
                    dep = 3;
                }
            }
            for (; nq; dep++) {   // deeper levels through the PHF (:52-64)
                uint32_t nw = 0;
                for (uint32_t e = 0; e < nq; e += 32) {
                    const bool have = e + lane < nq;
                    uint2 it = have ? q[e + lane] : make_uint2(0u, 0u);
                    __syncwarp();
                    bool alive = false;
                    if (have) {
                        const uint32_t t0 = it.x & 0xffffu;
                        const int32_t st = phf_next(p, (int32_t)it.y, s_text[t0 + dep]);
                        if (st >= 0) {
                            record(t0, st);
                            it.y = (uint32_t)st;
                            alive = t0 + dep + 1u < (it.x >> 16);
                        }
                    }
                    push(alive, nw, it);
                }
                __syncwarp();
                nq = nw;
            }
        }
        __syncthreads();
        // ---- block scan: thread t owns the starts [t * kDensePer, (t + 1) * kDensePer)
        uint32_t mine = 0;
#pragma unroll
        for (int j = 0; j < kDensePer; j++) mine += s_cnt[tid * kDensePer + j];
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_scan[lane], wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += v;
            }
            s_scan[lane] = wi - w;   // exclusive warp offsets
            const uint32_t tot = __shfl_sync(0xffffffffu, wi, 31);   // the tile's total
            unsigned long long base = 0;
            if (DIRECT) {
                // Decoupled look-back over the tiles' status words (epoch << 40 | flag << 38 | value): a tile
                // publishes its own total at once (flag 1 = aggregate), sums the aggregates of the tiles
                // before it back to the nearest one whose inclusive prefix is known (flag 2), 32 status
                // words per step, and then publishes its own inclusive prefix.
                constexpr unsigned long long kVal = (1ull << 38) - 1ull;
                const unsigned long long ep = (unsigned long long)d.epoch << 40;
                volatile unsigned long long *st = d.prefix;
                if (lane == 0) st[tile] = ep | ((tile == 0 ? 2ull : 1ull) << 38) | (unsigned long long)tot;
                for (long long look = (long long)tile - 1; look >= 0; look -= 32) {
                    const long long idx = look - lane;
                    unsigned long long v = ep | (2ull << 38);   // before the first tile: prefix 0
                    if (idx >= 0) {
                        v = st[idx];
                        for (Watchdog wd; (v >> 40) != d.epoch; v = st[idx]) {
                            if (wd.expired()) { atomicExch(&p.ctrl->error_flag, 6u); v = ep | (2ull << 38); break; }
                            __nanosleep(32);
                        }
                    }
                    const uint32_t has_p = __ballot_sync(0xffffffffu, ((v >> 38) & 3ull) == 2ull);
                    const int fp = has_p ? __ffs(has_p) - 1 : 31;   // the nearest tile with an inclusive prefix
                    unsigned long long add = lane <= fp ? (v & kVal) : 0ull;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) add += __shfl_xor_sync(0xffffffffu, add, o);
                    base += add;
                    if (has_p) break;
                }
                const unsigned long long inc = base + tot;
                if (lane == 0) {
                    if (tile > 0) st[tile] = ep | (2ull << 38) | (inc & kVal);
                    if (tile + 1 == p.n_tiles) {   // the last tile owns the total
                        d.result->count = inc;
                        d.result->error_flag = p.ctrl->error_flag;
                        if (d.count_out) *d.count_out = inc;
                    }
                }
            } else if (lane == 31) {
                base = tot ? atomicAdd(&p.ctrl->alloc, (unsigned long long)tot) : 0ull;
                p.tile_cnt[tile] = tot;
                p.tile_src[tile] = base;
                if (tot) atomicAdd(&p.partial[tile / p.tiles_per_part], (unsigned long long)tot);
            }
            if (DIRECT ? lane == 0 : lane == 31) {
                s_scan[32] = tot;
                s_scan[33] = (uint32_t)base;
                s_scan[34] = (uint32_t)(base >> 32);
            }
        }
        __syncthreads();
        const uint32_t total = s_scan[32];
        const unsigned long long base = (unsigned long long)s_scan[33] | ((unsigned long long)s_scan[34] << 32);
        uint32_t off = s_scan[warp] + incl - mine;   // this thread's first record within the tile's run
        // ---- write the records
        if (total) {
#pragma unroll
            for (int j = 0; j < kDensePer; j++) {
                const uint32_t t0 = tid * kDensePer + j, n = s_cnt[t0];
                if (!n) continue;
                const uint32_t a = a0 + t0;
                const unsigned long long o = base + off;
                if (n <= fin_keep) {
                    const uint32_t rec_pos = a - p.mis + p.pos_bias;
                    for (uint32_t k = 0; k < n; k++) {
                        const int32_t st = fin16 ? (int32_t)s_fin16[k * kTile + t0] : s_fin[k * kTile + t0];
                        if (o + k < dst_cap) dst[o + k] = make_uint2(rec_pos, (uint32_t)ldg_keep(&p.idmap[st]));
                    }
                } else {
                    walk_write(t0, a, limit_t(a, a0), o);
                }
                off += n;
            }
        }
    }
    if (DIRECT && tid == 0) {   // the last CTA out resets the control block for the next scan
        __threadfence();
        if (atomicAdd(&p.ctrl->exited, 1u) == gridDim.x - 1u) {
            p.ctrl->ticket = 0;
            p.ctrl->exited = 0;
            p.ctrl->error_flag = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Position-ordering pass.  Every tile's records are one position-ordered run of the arrival-order
// scratch (tile_src, tile_cnt); an exclusive scan of the per-tile counts gives each run its final
// place.  One CTA per tile range; the matches of the ranges before it come from the partial sums the
// emit and dense kernels accumulated.
constexpr int kFinThreads = 256;
constexpr int kFinSmall = 8;   // records a single thread moves by itself

__global__ void __launch_bounds__(kFinThreads) pfac_finalize_kernel(const FinalizeParams f)
{
    __shared__ unsigned long long s_red[kFinThreads / 32];
    __shared__ unsigned long long s_base[kFinThreads];
    __shared__ unsigned int s_cnt[kFinThreads];
    __shared__ unsigned int s_big[kFinThreads / 32];
    __shared__ unsigned long long s_run;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_launch_next();   // (the next scan's detector may set itself up)
#ifdef PFAC_TRACE
    const unsigned long long t_start = gtime_ns();
#endif
    pdl_wait();          // the kernels before this one have finished
#ifdef PFAC_TRACE
    const unsigned long long t_wait = gtime_ns();
#endif
    const uint32_t per = f.tiles_per_part;   // CTA b owns tiles [b*per, (b+1)*per); partial[b] = matches in them
    const uint32_t lo = min(f.n_tiles, blockIdx.x * per), hi = min(f.n_tiles, lo + per);

    unsigned long long sum = 0;
    for (uint32_t i = tid; i < blockIdx.x; i += kFinThreads) sum += f.partial[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) s_red[warp] = sum;
    __syncthreads();
    if (tid == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < kFinThreads / 32; w++) t += s_red[w];
        s_run = t;
    }
    __syncthreads();

    for (uint32_t c0 = lo; c0 < hi; c0 += kFinThreads) {
        const uint32_t i = c0 + tid;
        const unsigned int c = i < hi ? f.tile_cnt[i] : 0u;
        unsigned long long incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        if (lane == 31) s_red[warp] = incl;
        __syncthreads();
        unsigned long long wbase = 0;
        for (int w = 0; w < warp; w++) wbase += s_red[w];
        s_base[tid] = s_run + wbase + incl - c;
        // a tile with a few records (the common case: one match) is moved by the thread that owns it,
        // all tiles of the chunk in parallel -- the dependent loads tile_src -> scratch are latency,
        // not bandwidth; tiles with many records are left to the whole CTA below
        const bool small = c != 0u && c <= (unsigned)kFinSmall;
        if (small) {
            const unsigned long long dst = s_base[tid], src = f.tile_src[i];
            for (uint32_t k = 0; k < c; k++)
                if (src + k < f.scratch_cap && dst + k < f.cap) f.out[dst + k] = f.scratch[src + k];
        }
        s_cnt[tid] = small ? 0u : c;
        const uint32_t big = __ballot_sync(0xffffffffu, !small && c != 0u);
        if (lane == 0) s_big[warp] = big;
        __syncthreads();
        // the remaining matching tiles: all threads move one run at a time (coalesced)
        for (int w = 0; w < kFinThreads / 32; w++)
          for (uint32_t bits = s_big[w]; bits; bits &= bits - 1) {
            const int j = w * 32 + __ffs(bits) - 1;
            const uint32_t n = s_cnt[j];
            const unsigned long long dst = s_base[j], src = f.tile_src[c0 + j];
            // (the run fits both buffers or is cut at the caller's capacity; four loads in flight per thread)
            const uint32_t room = dst < f.cap ? (uint32_t)min((unsigned long long)n, f.cap - dst) : 0u;
            const uint32_t m = src < f.scratch_cap ? (uint32_t)min((unsigned long long)room, f.scratch_cap - src) : 0u;
            for (uint32_t k = tid; k < m; k += 4 * kFinThreads) {
                uint2 r[4];
#pragma unroll
                for (int u = 0; u < 4; u++)
                    if (k + u * kFinThreads < m) r[u] = f.scratch[src + k + u * kFinThreads];
#pragma unroll
                for (int u = 0; u < 4; u++)
                    if (k + u * kFinThreads < m) f.out[dst + k + u * kFinThreads] = r[u];
            }
        }
        __syncthreads();
        if (tid == kFinThreads - 1) s_run = s_base[tid] + c;
        __syncthreads();
    }
#ifdef PFAC_TRACE
    if ((f.debug & 64u) && tid == 0 && blockIdx.x == 0) {
        const unsigned long long t_end = gtime_ns();
        unsigned long long mn[5] = {~0ull, ~0ull, ~0ull, ~0ull, ~0ull}, mx[5] = {0, 0, 0, 0, 0};
        for (uint32_t b = 0; b < f.trace_ctas; b++)
            for (int k = 0; k < 5; k++) {
                unsigned long long *q = const_cast<unsigned long long *>(reinterpret_cast<const unsigned long long *>(f.scratch + (f.scratch_cap - 1ull - b * 8ull - k)));
                const unsigned long long v = *q;
                *q = 0;
                if (v) { mn[k] = v < mn[k] ? v : mn[k]; mx[k] = v > mx[k] ? v : mx[k]; }
            }
        const unsigned long long t0 = mn[0];
        printf("TRACE ns since the first CTA started: CTA starts ..%llu | image in %llu..%llu | last tile done %llu..%llu | its candidates settled %llu..%llu | "
               "last warp out %llu..%llu | ordering pass: CTA 0 starts %lld, passes its wait %llu, ends %llu\n",
               mx[0] - t0, mn[1] - t0, mx[1] - t0, mn[2] - t0, mx[2] - t0, mn[3] - t0, mx[3] - t0, mn[4] - t0, mx[4] - t0,
               (long long)(t_start - t0), t_wait - t0, t_end - t0);
    }
#endif
    if (tid == 0 && lo < hi && hi == f.n_tiles) {   // the CTA whose range ends the input owns the total
        f.result->count = s_run;
        f.result->error_flag = f.ctrl->error_flag;
        if (f.count_out) *f.count_out = s_run;
        f.ctrl->ticket = 0;
        f.ctrl->error_flag = 0;
        f.ctrl->alloc = 0;
        f.ctrl->n_dense = 0;
    }
}

#endif  // __CUDACC__

}  // namespace pfac
