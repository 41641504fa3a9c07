// Device-side derived layouts of one partition's canonical tables (host code, no CUDA).
//
// The canonical PHF arrays r/HT/val (bit-compatible with CreateTable/FFDM, reference phf.c:151)
// stay the authoritative transition function: they are uploaded unchanged (HT and val
// interleaved) and the candidate / dense-match walks follow them exactly as master_kernel.cu:52-64 does.  What is
// derived here is the shared-memory image of the DETECTOR kernel: prefix filters computed from the
// first rows of the PHF.  Every one of them is a superset test -- it may pass a start position
// that cannot match, it never rejects one that can:
//   T1    65,536 x u8 : up to eight bit-planes per 2-byte window (x,y), one LDS.U8 per probe:
//                         P01   a walk starting with (x,y) matches a 1-byte pattern or has a second
//                               edge (root fan-out, s0Table of main.cc:200, folded in) -- exact
//                         P12 / P23 / P34   (x,y) are bytes 1-2 / 2-3 / 3-4 of some path of the automaton
//                         Short / ShortC    (x,y) as bytes 0-1 / 1-2 can complete a pattern of <= 3 / <= 4 bytes
//                         P45 / P56 / ShX   third-window planes (sets without patterns of <= 3 bytes; below)
//                       Mode 0 probes the windows at EVEN offsets only: an even start 2k is judged by the
//                       windows at 2k (P01), 2k+2 (P23) and 2k+4 (P45), an odd start 2k+1 by those at 2k+2
//                       (P12), 2k+4 (P34) and 2k+6 (P56); modes 1 / 2 probe every start (P01, P12, P23).
//                       Indexed with both bytes rotated left by 2 so that the low, high-entropy
//                       bits of ASCII text select the shared-memory bank.
//   level 1 / level 2 (mode 0): perfect-hash tables (hash-and-displace D / E, u16) of every 4-byte prefix -> m1
//                       and of every (prefix, bytes [m1-4, m1)) group -> m2; m = (at most) the shortest pattern
//                       length below the key.  A word that is no key finds m = 0 or, once in 256, another key's m.
//   Tm / Tm2 (mode 2) : the same two levels as COMPLETE cuckoo tables (2 buckets x 2 tagged u16 slots), sized
//                       for the key counts, in global memory
//   T3    2^k3 bits   : hash of (key, pattern bytes [m-4, m)) for every pattern below a key: a start
//                       whose text at offset m-4 is not in T3 cannot complete any pattern under
//                       that key (Wu-Manber style two-point checks; they settle the starts that
//                       share a long prefix with many patterns without walking it)
//   T2    2^k2 bits   : blocked Bloom filter (one word, kT2KeyBits bits) of every 4-byte prefix -- only for pattern sets whose
//                       prefixes do not fit the shared-memory tables.  Such sets (e.g. 100,000 patterns)
//                       get Tm/Tm2/T3 sized for their key counts in GLOBAL memory (a few MB, L2
//                       resident) and T2, filling shared memory, becomes stage 1.
#pragma once
#include <cstdint>
#include <vector>

#include "pfac_internal.h"

namespace pfac {

constexpr uint32_t kHash4Mul = 0x9E3779B1u;
// T2 is a BLOCKED Bloom filter: one multiplicative hash h of the 4-byte prefix selects a 32-bit word (its top
// bits) and kT2KeyBits bit positions inside that word (the 5-bit fields below them) -- one shared-memory load
// and one mask compare per start position decide, instead of one probe per hash function.
#ifndef PFAC_T2_KEY_BITS
#define PFAC_T2_KEY_BITS 2
#endif
constexpr int kT2KeyBits = PFAC_T2_KEY_BITS;
constexpr uint32_t kTmSlotBits = 12;
constexpr uint32_t kTm1Slots = 2u << kTmSlotBits;   // level 1: 4096 buckets x 2 slots (u16: tag << 8 | m, 0 = empty)
constexpr uint32_t kT3Seed2 = 0x5bd1e995u;

#if defined(__CUDACC__)
#define PFAC_HD __host__ __device__
#else
#define PFAC_HD
#endif
// T3 index (before the final shift) of a key and the 4 window bytes (little-endian word)
PFAC_HD inline uint32_t hash_t3(uint32_t key, uint32_t window)
{
    uint32_t x = key * 0x9E3779B1u + window * 0x85EBCA6Bu;
    x ^= x >> 15;
    return x * 0x2C1B3C6Du;
}
// level-2 key of a (4-byte prefix, level-1 window) group
PFAC_HD inline uint32_t hash_key2(uint32_t prefix, uint32_t window)
{
    uint32_t x = prefix * 0xC2B2AE35u ^ window * 0x27D4EB2Fu;
    x ^= x >> 16;
    return x * 0x165667B1u + 0x9E3779B9u;
}
PFAC_HD inline uint32_t tm_slot1(uint32_t key, uint32_t bits) { return (key * 0xC2B2AE35u) >> (32 - bits); }
PFAC_HD inline uint32_t tm_slot2(uint32_t key, uint32_t bits) { return (key * 0x27D4EB2Fu + 0x7F4A7C15u) >> (32 - bits); }
// tags are 1..255 so that an empty slot (0) never matches
PFAC_HD inline uint32_t tm_tag(uint32_t key)
{
    const uint32_t t = (key * 0xFD7046C5u) >> 24;
    return t ? t : 1u;
}
// complete cuckoo table of 2^bits buckets x 2 slots (u16: tag << 8 | m): m of `key`, 0 = not a key.
// Probe order: bucket 1 low, bucket 1 high, bucket 2 low, bucket 2 high.
PFAC_HD inline uint32_t tm_lookup(const uint16_t *tab, uint32_t key, uint32_t bits)
{
    const uint32_t tag = tm_tag(key);
    const uint32_t *t32 = reinterpret_cast<const uint32_t *>(tab);
    const uint32_t a = t32[tm_slot1(key, bits)], b = t32[tm_slot2(key, bits)];
    uint32_t m = 0;
    if ((b >> 24) == tag) m = (b >> 16) & 255u;
    if (((b >> 8) & 255u) == tag) m = b & 255u;
    if ((a >> 24) == tag) m = (a >> 16) & 255u;
    if (((a >> 8) & 255u) == tag) m = a & 255u;
    return m;
}
// T2 of 2^(32 - shift) bits (at least 2^(5 + 5 kT2KeyBits)... the fields may overlap the word index for tiny
// tables, which only weakens the filter): word index and bit mask of the prefix hash h = w4 * kHash4Mul
PFAC_HD inline uint32_t t2_word(uint32_t h, uint32_t shift) { return h >> (shift + 5u); }
PFAC_HD inline uint32_t t2_mask(uint32_t h, uint32_t shift)
{
    uint32_t m = 0;
    for (int i = 0; i < kT2KeyBits; i++) {
        const uint32_t sh = shift >= 5u * (uint32_t)i ? shift - 5u * (uint32_t)i : 0u;
        m |= 1u << ((h >> sh) & 31u);
    }
    return m;
}
PFAC_HD inline bool t2_pass(const uint32_t *t2, uint32_t w4, uint32_t shift)
{
    const uint32_t h = w4 * kHash4Mul, m = t2_mask(h, shift);
    return (t2[t2_word(h, shift)] & m) == m;
}
// rotl2 of a byte; T1 index of the window (c0, c1); T1 bit-planes
#ifndef PFAC_NO_ROT2
PFAC_HD inline uint32_t rot2(uint32_t c) { return ((c << 2) | (c >> 6)) & 0xFFu; }
#else
PFAC_HD inline uint32_t rot2(uint32_t c) { return c; }
#endif
PFAC_HD inline uint32_t t1_index(uint32_t c0, uint32_t c1) { return rot2(c0) | (rot2(c1) << 8); }
constexpr uint8_t kT1P01 = 1, kT1P12 = 2, kT1P23 = 4, kT1Short = 8, kT1P34 = 16, kT1ShortC = 32;
// Third-window planes of the mode-0 detector (Derived::has_w3; only for sets without patterns of <= 3 bytes,
// whose Short plane is empty -- ShX takes its bit): an even start also needs its bytes 4-5 (P45) unless its
// bytes 2-3 end-or-nearly-end a pattern of 4-5 bytes (ShX); an odd start its bytes 5-6 (P56) unless its
// bytes 3-4 belong to a pattern of 5-6 bytes (ShX again: one plane for both exceptions).
constexpr uint8_t kT1P45 = 64, kT1P56 = 128, kT1ShX = 8;

// ---- perfect-hash tables of the mode-0 detector (hash-and-displace, one slot per key).
// bucket = mulhi(x, nb) with x = a mixed hash of the key, d = D[bucket], slot = mulhi(key * c3 + d *
// (key * c4 | 1), ns), entry E[slot] = m << 8 | tag with tag = x & 255.  A key of the set finds its
// own entry; any other word finds m = 0 or, once in 256, some other key's m.
PFAC_HD inline uint32_t mulhi32(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
PFAC_HD inline uint32_t ph_mix(uint32_t key)
{
    uint32_t x = key * 0x9E3779B1u;
    x ^= x >> 15;
    return x * 0x85EBCA77u;
}
PFAC_HD inline uint32_t ph_slot(uint32_t key, uint32_t d, uint32_t ns)
{
    return mulhi32(key * 0xC2B2AE3Du + d * ((key * 0x27D4EB2Fu) | 1u), ns);
}
// x = ph_mix(key) for raw keys (level 1: the 4-byte prefix), x = key for keys that are hashes already (level 2)
PFAC_HD inline uint32_t ph_lookup(const uint16_t *D, const uint16_t *E, uint32_t nb, uint32_t ns, uint32_t key, uint32_t x)
{
    const uint32_t d = D[mulhi32(x, nb)];
    const uint32_t e = E[ph_slot(key, d, ns)];
    return ((e ^ x) & 255u) ? 0u : (e >> 8);   // entry = m << 8 | tag
}

struct Derived {
    // shared-memory image, copied verbatim by the detector kernel (sections 128-byte aligned)
    std::vector<uint8_t> image;
    uint32_t off_t1 = 0, off_t2 = 0, off_tm = 0, off_tm2 = 0, off_t3 = 0;
    uint32_t t2_shift = 32;      // T2 has 2^(32 - t2_shift) bits (t2_word / t2_mask above); 32: no T2
    uint32_t has_short = 0;      // patterns of length <= 3 exist (T1's Short plane is not empty)
    uint32_t has_shortc = 0;     // patterns of length <= 4 exist (T1's ShortC plane is not empty)
    uint32_t has_w3 = 0;         // T1 carries the third-window planes P45 / P56 / ShX (mode 0, no short patterns)
    uint32_t has_t3 = 0;         // Tm + T3 present (then no T2)
    uint32_t t3_shift = 32;
    uint32_t tm_bits = 0, tm2_bits = 0;   // log2 buckets of Tm / Tm2 (0: absent; mode 2 only)
    // mode 0: perfect-hash tables of the 4-byte prefixes (level 1) and the (prefix, window) groups (level 2)
    uint32_t off_d1 = 0, off_e1 = 0, nb1 = 0, ns1 = 0;
    uint32_t off_d2 = 0, off_e2 = 0, nb2 = 0, ns2 = 0;   // ns2 = 0: no level 2
    // mode 0: two-point checks from shared memory; 1: T2 alone; 2: stage 1 = T2 (the whole shared
    // image), Tm/Tm2/T3 sized for the key counts in `gimage` (global memory, L2-resident) -- offsets
    // off_t1/off_tm/off_tm2/off_t3 then refer to gimage, which starts with a copy of T1
    uint32_t mode = 1;
    std::vector<uint8_t> gimage;
    // statistics (pfac_ctx_derived_info)
    uint32_t t1_set = 0, t2_set = 0, t3_set = 0, tm_set = 0, tm2_set = 0, n_prefix4 = 0;
};

// ---- walk cache of the dense-match kernel (pfac_dense_kernel): the first levels of the trie as an
// exact perfect-hash map in shared memory, so that the walks of dense inputs (most starts take a few
// steps) read shared memory instead of chasing r[] / {HT,val} through L1/L2.
//   image = s0Table (256 x i32) | D (nb x u16) | E (ns x {key u32, state i32})
//   key   = b0 | b1 << 8 | kWalkDepth2   or   b0 | b1 << 8 | b2 << 16 | kWalkDepth3
// The map is COMPLETE for every depth it covers: a miss means the automaton has no such path.
constexpr uint32_t kWalkDepth2 = 0x02000000u, kWalkDepth3 = 0x03000000u;
struct WalkCache {
    std::vector<uint8_t> image;
    uint32_t depth = 1;          // 1: root row only, 2: + every 2-byte path, 3: + every 3-byte path
    uint32_t off_d = 0, off_e = 0, nb = 0, ns = 0;
};
void derive_walk_cache(const Partition &P, uint32_t budget_bytes, WalkCache &out);
int32_t walk_cache_lookup(const WalkCache &w, const uint8_t *t, uint32_t depth);

// ---- pattern directory of the candidate walks (emit_tile_dir): every final state's own string, hashed.
// A start that survived the detector's filters is settled by asking, for every pattern length d of the set
// at once (one lane per length, independent loads), "is text[start, start + d) a pattern?" -- a hash probe
// followed by an exact byte compare -- instead of chasing d dependent transitions through the PHF.  The
// answers equal SUBSEG_MATCH's: the automaton is a trie, so text[start, start+d) reaches a final state iff
// it IS that state's string.
//   image = dir (n_slots x {h_lo, h_hi, id, len << 25 | pool offset}; open addressing, linear probing,
//           0xFFFFFFFF in the last word = empty) | pool (the strings)
// Built only for tree-shaped automata with max_len <= 64 and < 32 MiB of strings; otherwise empty and the
// kernels walk.
// Hash of a string b_0..b_{d-1}: the polynomial sum of (b_i + 1) K^(d-i) modulo 2^64 (Horner: h = (h + b + 1) K).
// K is odd, so it has an inverse and the hashes of ALL prefixes of a text follow from one prefix sum:
// h_d = K^d * sum_{i<d} (b_i + 1) K^-i  -- a warp scan on the device (emit_tile_dir).
constexpr uint64_t kDirMul = 0x9E3779B97F4A7C15ull;
PFAC_HD constexpr uint64_t dir_cpow(uint64_t b, uint32_t e)   // b^e modulo 2^64
{
    uint64_t r = 1;
    for (; e; e >>= 1, b *= b)
        if (e & 1u) r *= b;
    return r;
}
PFAC_HD constexpr uint64_t dir_inverse(uint64_t k)   // of an odd k modulo 2^64 (Newton)
{
    uint64_t x = 1;
    for (int i = 0; i < 6; i++) x *= 2 - k * x;
    return x;
}
constexpr uint64_t kDirMulInv = dir_inverse(kDirMul);
static_assert(kDirMul * kDirMulInv == 1ull, "K is invertible");
PFAC_HD inline uint64_t dir_hash_step(uint64_t h, uint32_t byte) { return (h + (uint64_t)byte + 1ull) * kDirMul; }
PFAC_HD inline uint32_t dir_slot(uint64_t h, uint32_t n_slots) { return (uint32_t)(h >> 24) & (n_slots - 1u); }
struct PatDir {
    std::vector<uint8_t> image;
    uint32_t n_slots = 0;        // power of two, 0 = no directory
    uint32_t off_pool = 0;
    uint64_t len_mask = 0;       // bit d-1: some pattern has length d
};
void derive_patdir(const Partition &P, PatDir &out);
int64_t patdir_lookup(const PatDir &pd, const uint8_t *text, uint32_t d);
int patdir_selfcheck(const Partition &P, const PatDir &pd);   // 0 = the directory answers like the walk

// ---- pattern length of every id (batch scans: a record is kept iff its pattern ends inside its document).
// len[id] = depth of the final state that reports id, 0 for ids no reachable final state reports (the earlier
// copies of a duplicated line); len.size() = max id + 1.  The automaton is a trie, so a final state's depth is
// its pattern's length.  PFAC_ERR_ARG (message set) if it is not a tree -- a state reached twice, as in sets
// wrapped from arrays that share states -- or if two final states report one id.
int pattern_lengths(const Partition &P, std::vector<int32_t> &len);

// t2/t3/tm2_bytes: shared-memory budget of the variable sections (rounded down to powers of two)
void derive_tables(const Partition &P, uint32_t t2_bytes, uint32_t t3_bytes, uint32_t tm2_bytes, Derived &out);

// Checks the derived image against the canonical PHF: T1 exact, T1s / Tm / Tm2 / T3 / T2 pass every
// pattern's own bytes.  0 = ok, otherwise the index of the first violated invariant.
int derive_selfcheck(const Partition &P, const Derived &d);

// Diagnostics: survivors per stage of the detector's filter cascade over `text` (counts only).
void derive_profile(const Partition &P, const Derived &d, const uint8_t *text, size_t n, uint64_t out[12]);

}  // namespace pfac
