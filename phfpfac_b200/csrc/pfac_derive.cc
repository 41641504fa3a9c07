// Host-side derivation of the detector kernel's shared-memory filters from one partition's
// canonical PHF arrays (see pfac_derive.h).  Everything here is computed FROM r/HT/val/s0Table,
// i.e. from what CreateTable + FFDM (reference create_table_reorder.c:277, phf.c:151) emit, so
// tables handed in through pfac_tables_from_arrays get the same treatment.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>

#include "pfac_derive.h"

namespace pfac {

namespace {

struct Edge {
    int32_t state, byte, next;
};

// transitions of the automaton, recovered from the PHF slots and grouped by source state
struct Graph {
    std::vector<Edge> edges;
    std::vector<uint32_t> first;
    int32_t n_states = 0, n_final = 0;
    uint32_t begin(int32_t s) const { return s >= 0 && s < n_states ? first[(size_t)s] : 0u; }
    uint32_t end(int32_t s) const { return s >= 0 && s < n_states ? first[(size_t)s + 1] : 0u; }
    bool is_final(int32_t s) const { return s >= 0 && s < n_final; }
};

void build_graph(const Partition &P, Graph &g)
{
    g.n_states = std::max(P.state_num, 0);
    g.n_final = P.n_final;
    const int wb = width_bits(P.width);
    g.edges.reserve((size_t)std::max(P.n_keys, 0));
    // slot idx of row `row` holds the key row*width + (idx - r[row])   (phf.c:197-216)
    for (int32_t idx = 0; idx < P.ht_size; idx++) {
        const int32_t row = P.HT[(size_t)idx];
        if (row < 0 || row >= (int32_t)P.r.size()) continue;
        const int64_t col = (int64_t)idx - P.r[(size_t)row];
        if (col < 0 || col >= P.width) continue;
        const int64_t key = ((int64_t)row << wb) + col;
        const int64_t st = key >> 8;
        const int32_t nx = P.val[(size_t)idx];
        if (st >= g.n_states || nx < 0) continue;   // never produced by a lookup the kernels can make
        g.edges.push_back({(int32_t)st, (int32_t)(key & 255), nx});
    }
    std::sort(g.edges.begin(), g.edges.end(), [](const Edge &a, const Edge &b) {
        return a.state != b.state ? a.state < b.state : a.byte < b.byte;
    });
    g.first.assign((size_t)g.n_states + 2, 0);
    for (const Edge &e : g.edges) g.first[(size_t)e.state + 1]++;
    for (int32_t s = 0; s <= g.n_states; s++) g.first[(size_t)s + 1] += g.first[(size_t)s];
}

inline uint32_t align128(uint32_t x) { return (x + 127u) & ~127u; }
inline uint32_t pow2_bits_for_bytes(uint32_t bytes)   // largest power-of-two bit count <= bytes*8 (0 if < 128 B)
{
    if (bytes < 128) return 0;
    uint32_t bits = 1024;
    while ((uint64_t)bits * 2 <= (uint64_t)bytes * 8) bits *= 2;
    return bits;
}
inline uint32_t log2u(uint32_t x)
{
    uint32_t k = 0;
    while ((1u << k) < x) k++;
    return k;
}

constexpr uint64_t kPathLimit = 1ull << 23;   // general (non-tree) automata may have too many paths

struct Key {
    uint32_t key, m;
};

// Cuckoo placement of every key into 2^bits buckets x 2 slots; false if they do not all fit.
// Keys that share a tag and can see each other's slot take the smaller m, so whichever entry a
// lookup hits first the answer is a valid (not too large) length.
bool place_all(std::vector<Key> &keys, uint32_t bits, std::vector<uint16_t> &tab)
{
    const uint32_t n_slots = 2u << bits;
    if (keys.size() > (size_t)n_slots * 17 / 20) return false;
    std::vector<int32_t> owner(n_slots, -1);
    auto slots_of = [&](uint32_t key, uint32_t sl[4]) {
        const uint32_t b1 = tm_slot1(key, bits), b2 = tm_slot2(key, bits);
        sl[0] = b1 * 2;
        sl[1] = b1 * 2 + 1;
        sl[2] = b2 * 2;
        sl[3] = b2 * 2 + 1;
    };
    uint64_t rng = 0x9E3779B97F4A7C15ull;
    for (size_t i = 0; i < keys.size(); i++) {
        int32_t cur = (int32_t)i;
        bool placed = false;
        for (int kick = 0; kick < 4000 && !placed; kick++) {
            uint32_t sl[4];
            slots_of(keys[(size_t)cur].key, sl);
            for (int c = 0; c < 4 && !placed; c++)
                if (owner[sl[c]] < 0) {
                    owner[sl[c]] = cur;
                    placed = true;
                }
            if (!placed) {
                rng = rng * 6364136223846793005ull + 1442695040888963407ull;
                std::swap(cur, owner[sl[(rng >> 33) & 3]]);
            }
        }
        if (!placed) return false;
    }
    bool changed = true;
    while (changed) {
        changed = false;
        for (size_t i = 0; i < keys.size(); i++) {
            uint32_t sl[4];
            slots_of(keys[i].key, sl);
            for (int c = 0; c < 4; c++) {
                const int32_t o = owner[sl[c]];
                if (o < 0 || (size_t)o == i || tm_tag(keys[(size_t)o].key) != tm_tag(keys[i].key)) continue;
                const uint32_t lo = std::min(keys[i].m, keys[(size_t)o].m);
                if (keys[i].m != lo || keys[(size_t)o].m != lo) {
                    keys[i].m = keys[(size_t)o].m = lo;
                    changed = true;
                }
            }
        }
    }
    tab.assign(n_slots, 0);
    for (uint32_t sl = 0; sl < n_slots; sl++)
        if (owner[sl] >= 0)
            tab[sl] = (uint16_t)((tm_tag(keys[(size_t)owner[sl]].key) << 8) | keys[(size_t)owner[sl]].m);
    return true;
}

// Hash-and-displace placement (pfac_derive.h: ph_lookup) of every key into its own slot: buckets in
// order of decreasing size, each takes the first displacement that puts all its keys on free slots.
// `premixed`: the keys are hashes already (level 2).  false if no 16-bit displacement works.
bool ph_place(const std::vector<uint32_t> &keys, bool premixed, uint32_t nb, uint32_t ns, std::vector<uint16_t> &D,
              std::vector<uint32_t> &slot_of)
{
    D.assign(nb, 0);
    slot_of.assign(keys.size(), 0);
    if (keys.empty()) return true;
    if (keys.size() > ns) return false;
    std::vector<std::vector<uint32_t>> bucket(nb);
    for (uint32_t i = 0; i < keys.size(); i++) {
        const uint32_t x = premixed ? keys[i] : ph_mix(keys[i]);
        bucket[mulhi32(x, nb)].push_back(i);
    }
    std::vector<uint32_t> order(nb);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return bucket[a].size() > bucket[b].size(); });
    std::vector<uint8_t> used(ns, 0);
    std::vector<uint32_t> slots;
    for (uint32_t b : order) {
        const auto &ks = bucket[b];
        if (ks.empty()) break;
        bool placed = false;
        for (uint32_t d = 0; d < 65536 && !placed; d++) {
            slots.clear();
            bool ok = true;
            for (uint32_t i : ks) {
                const uint32_t sl = ph_slot(keys[i], d, ns);
                if (used[sl] || std::find(slots.begin(), slots.end(), sl) != slots.end()) { ok = false; break; }
                slots.push_back(sl);
            }
            if (!ok) continue;
            D[b] = (uint16_t)d;
            for (size_t j = 0; j < ks.size(); j++) {
                used[slots[j]] = 1;
                slot_of[ks[j]] = slots[j];
            }
            placed = true;
        }
        if (!placed) return false;
    }
    return true;
}
// the detector's tables: entry = m << 8 | tag
bool ph_build(const std::vector<Key> &keys, bool premixed, uint32_t nb, uint32_t ns, std::vector<uint16_t> &D,
              std::vector<uint16_t> &E)
{
    std::vector<uint32_t> k(keys.size()), slot_of;
    for (size_t i = 0; i < keys.size(); i++) k[i] = keys[i].key;
    E.assign(ns, 0);
    if (!ph_place(k, premixed, nb, ns, D, slot_of)) return false;
    for (size_t i = 0; i < keys.size(); i++) {
        const uint32_t x = premixed ? k[i] : ph_mix(k[i]);
        E[slot_of[i]] = (uint16_t)((keys[i].m << 8) | (x & 255u));
    }
    return true;
}
// sizes of a perfect-hash table for n keys: about three keys per bucket, slots 80 % full
inline void ph_sizes(size_t n, uint32_t &nb, uint32_t &ns)
{
    nb = (uint32_t)std::max<size_t>(8, (n + 2) / 3);
    ns = (uint32_t)std::max<size_t>(16, n * 5 / 4 + 8);
    nb = (nb + 63u) & ~63u;   // sections stay 128-byte aligned
    ns = (ns + 63u) & ~63u;
}
constexpr uint32_t kPh1MaxBytes = 24576;   // level 1 beyond this: the set goes to global mode

inline uint32_t le32(const uint8_t *q)
{
    return (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
}
inline uint32_t le32(const std::string &s, uint32_t at) { return le32(reinterpret_cast<const uint8_t *>(s.data()) + at); }
inline bool bit(const uint32_t *tab, uint32_t h) { return (tab[h >> 5] >> (h & 31)) & 1u; }

}  // namespace

void derive_tables(const Partition &P, uint32_t t2_bytes, uint32_t t3_bytes, uint32_t tm2_bytes, Derived &out)
{
    out = Derived();
    Graph g;
    build_graph(P, g);
    const int32_t n_states = g.n_states;
    auto s0 = [&](int b) { return P.s0.empty() ? -1 : P.s0[(size_t)b]; };

    // ---- T1 / T1s over the first two bytes, the list of 4-byte prefixes, T2
    std::vector<uint8_t> t1(65536, 0);
    uint32_t t2_bits = pow2_bits_for_bytes(t2_bytes);
    std::vector<uint32_t> t2(t2_bits / 32, 0);
    const uint32_t t2_shift = t2_bits ? 32u - log2u(t2_bits) : 32u;
    std::vector<std::pair<uint32_t, int32_t>> prefix4;   // (4-byte prefix as a little-endian word, state after it)
    bool any_short = false, too_many = false, all_shortc = false;
    for (int b0 = 0; b0 < kCharSet; b0++) {
        const int32_t s1 = s0(b0);
        if (s1 < 0) continue;
        if (g.is_final(s1)) {   // a 1-byte pattern: every pair starting with b0 reports a match
            any_short = true;
            all_shortc = true;   // ... and as bytes 1-2 of a start every window may follow it
            for (int b1 = 0; b1 < kCharSet; b1++) t1[t1_index((uint32_t)b0, (uint32_t)b1)] |= kT1P01 | kT1Short;
        }
        for (uint32_t e1 = g.begin(s1); e1 < g.end(s1); e1++) {
            const int32_t b1 = g.edges[e1].byte, s2 = g.edges[e1].next;
            const uint32_t pair = (uint32_t)b0 | ((uint32_t)b1 << 8);
            t1[t1_index((uint32_t)b0, (uint32_t)b1)] |= kT1P01;
            bool shortp = g.is_final(s2);
            if (shortp)   // a 2-byte pattern (b0, b1): bytes 1-2 of its start are (b1, anything)
                for (int b2 = 0; b2 < kCharSet; b2++) t1[t1_index((uint32_t)b1, (uint32_t)b2)] |= kT1ShortC;
            for (uint32_t e2 = g.begin(s2); e2 < g.end(s2); e2++) {
                const int32_t b2 = g.edges[e2].byte, s3 = g.edges[e2].next;
                if (g.is_final(s3)) {
                    shortp = true;
                    t1[t1_index((uint32_t)b1, (uint32_t)b2)] |= kT1ShortC;
                }
                t1[t1_index((uint32_t)b1, (uint32_t)b2)] |= kT1P12;
                for (uint32_t e3 = g.begin(s3); e3 < g.end(s3); e3++) {
                    t1[t1_index((uint32_t)b2, (uint32_t)g.edges[e3].byte)] |= kT1P23;
                    {   // bytes 3-4 of the paths that go on; a pattern of 4 bytes is settled by its bytes 1-2
                        const int32_t s4 = g.edges[e3].next;
                        if (g.is_final(s4)) t1[t1_index((uint32_t)b1, (uint32_t)b2)] |= kT1ShortC;
                        for (uint32_t e4 = g.begin(s4); e4 < g.end(s4); e4++)
                            t1[t1_index((uint32_t)g.edges[e3].byte, (uint32_t)g.edges[e4].byte)] |= kT1P34;
                    }
                    if (too_many) continue;
                    const uint32_t w = pair | ((uint32_t)b2 << 16) | ((uint32_t)g.edges[e3].byte << 24);
                    if (t2_bits) {
                        const uint32_t h = w * kHash4Mul;
                        t2[t2_word(h, t2_shift)] |= t2_mask(h, t2_shift);
                    }
                    prefix4.push_back({w, g.edges[e3].next});
                    if (prefix4.size() > kPathLimit) too_many = true;
                }
            }
            if (shortp) {
                any_short = true;
                t1[t1_index((uint32_t)b0, (uint32_t)b1)] |= kT1Short;
            }
        }
    }
    if (too_many) std::fill(t2.begin(), t2.end(), 0xFFFFFFFFu);   // not a tree: T2 filters nothing
    if (all_shortc)
        for (auto &b : t1) b |= kT1ShortC;
    out.has_short = any_short ? 1u : 0u;
    for (uint8_t b : t1)
        if (b & kT1ShortC) out.has_shortc = 1;
    out.n_prefix4 = (uint32_t)std::min<size_t>(prefix4.size(), 0xFFFFFFFFu);

    // ---- Tm / Tm2 / T3: two-point checks (pfac_derive.h).  First with the shared-memory sizes; if the
    // 4-byte prefixes do not fit Tm there and the set has no short patterns, once more with tables
    // sized for the key counts, to live in global memory (L2-resident).
    uint32_t t3_bits = too_many ? 0 : pow2_bits_for_bytes(t3_bytes);
    std::vector<uint16_t> tm, tm2;
    std::vector<uint16_t> d1, e1, d2, e2;   // mode 0: perfect-hash tables of the two key levels
    uint32_t nb1 = 0, ns1 = 0, nb2 = 0, ns2 = 0;
    std::vector<uint32_t> t3;
    uint32_t tm2_bits = 0, tm_bits = kTmSlotBits;
    bool global_mode = false;
    for (int attempt = 0; attempt < 2 && t3_bits; attempt++) {
        if (attempt == 1) {
            if (any_short || prefix4.size() > (1u << 22)) { t3_bits = 0; break; }
            global_mode = true;
            tm_bits = 10;
            while ((size_t)(2u << tm_bits) * 7 / 10 < prefix4.size()) tm_bits++;
            t3_bits = 1u << 20;
            while (t3_bits < 64ull * prefix4.size() && t3_bits < (1u << 28)) t3_bits *= 2;
        }
        t3.assign(t3_bits / 32, 0);
        tm.clear();
        tm2.clear();
        tm2_bits = 0;
        nb1 = ns1 = nb2 = ns2 = 0;
        out.t3_shift = 32u - log2u(t3_bits);
        // shortest distance from every state to a final state (reverse breadth-first search)
        const uint32_t kInf = 0xFFFFFFFFu;
        std::vector<uint32_t> rfirst((size_t)n_states + 2, 0), rsrc(g.edges.size());
        for (const Edge &e : g.edges)
            if (e.next < n_states) rfirst[(size_t)e.next + 1]++;
        for (int32_t st = 0; st <= n_states; st++) rfirst[(size_t)st + 1] += rfirst[(size_t)st];
        {
            std::vector<uint32_t> fill(rfirst.begin(), rfirst.end() - 1);
            for (const Edge &e : g.edges)
                if (e.next < n_states) rsrc[fill[(size_t)e.next]++] = (uint32_t)e.state;
        }
        std::vector<uint32_t> mind((size_t)n_states, kInf);
        std::vector<int32_t> bfs;
        for (int32_t st = 0; st < std::min(g.n_final, n_states); st++) {
            mind[(size_t)st] = 0;
            bfs.push_back(st);
        }
        for (size_t i = 0; i < bfs.size(); i++) {
            const int32_t st = bfs[i];
            for (uint32_t e = rfirst[(size_t)st]; e < rfirst[(size_t)st + 1]; e++) {
                const uint32_t src = rsrc[e];
                if (mind[src] == kInf) {
                    mind[src] = mind[(size_t)st] + 1;
                    bfs.push_back((int32_t)src);
                }
            }
        }
        auto dist = [&](int32_t st) { return st >= 0 && st < n_states ? mind[(size_t)st] : kInf; };

        // level 1 keys: one per distinct 4-byte prefix word (a general automaton may reach several states)
        std::sort(prefix4.begin(), prefix4.end());
        std::vector<Key> k1;
        std::vector<std::pair<size_t, size_t>> k1_range;   // prefix4 index range of each key
        for (size_t i = 0; i < prefix4.size();) {
            size_t j = i;
            uint32_t m = kInf;
            while (j < prefix4.size() && prefix4[j].first == prefix4[i].first) {
                const uint32_t d = dist(prefix4[j].second);
                if (d != kInf) m = std::min(m, 4u + d);
                j++;
            }
            if (m != kInf) {
                k1.push_back({prefix4[i].first, std::min(m, 255u)});
                k1_range.push_back({i, j});
            }
            i = j;
        }
        bool ok;
        if (global_mode) {
            ok = place_all(k1, tm_bits, tm);
        } else {
            ph_sizes(k1.size(), nb1, ns1);
            ok = (nb1 + ns1) * 2u <= kPh1MaxBytes && ph_build(k1, false, nb1, ns1, d1, e1);
        }

        // every string of exactly `len` bytes that continues (state, str); str holds the bytes so far
        uint64_t visited = 0;
        typedef std::vector<std::pair<int32_t, std::string>> Level;
        auto descend = [&](Level &level, uint32_t len) {
            Level nxt;
            while (ok && !level.empty() && level[0].second.size() < len) {
                nxt.clear();
                for (const auto &it : level)
                    for (uint32_t e = g.begin(it.first); e < g.end(it.first); e++) {
                        nxt.push_back({g.edges[e].next, it.second + (char)g.edges[e].byte});
                        if (++visited > kPathLimit) ok = false;
                    }
                level.swap(nxt);
            }
        };
        // level 1 windows -> T3; the strings at depth m1 are the members of the level-2 groups
        struct Member {
            uint32_t key2;
            int32_t state;
            std::string str;
        };
        std::vector<Member> members;
        std::vector<uint32_t> l1_bits;   // T3 indices of the level-1 windows
        for (size_t i = 0; i < k1.size() && ok; i++) {
            Level level;
            std::string pre(4, '\0');
            for (int b = 0; b < 4; b++) pre[(size_t)b] = (char)((k1[i].key >> (8 * b)) & 255u);
            for (size_t j = k1_range[i].first; j < k1_range[i].second; j++) level.push_back({prefix4[j].second, pre});
            descend(level, k1[i].m);
            for (auto &it : level) {
                if (dist(it.first) == kInf) continue;   // no pattern below
                const uint32_t w1 = le32(it.second, k1[i].m - 4u);
                l1_bits.push_back(hash_t3(k1[i].key, w1) >> out.t3_shift);
                members.push_back({hash_key2(k1[i].key, w1), it.first, std::move(it.second)});
            }
        }
        // level 2 keys: groups by key2; m2 = the shortest pattern length over the members
        if (ok && (tm2_bytes >= 64 || global_mode)) {
            std::sort(members.begin(), members.end(), [](const Member &x, const Member &y) { return x.key2 < y.key2; });
            std::vector<Key> k2;
            std::vector<std::pair<size_t, size_t>> k2_range;
            for (size_t i = 0; i < members.size();) {
                size_t j = i;
                uint32_t m = kInf;
                while (j < members.size() && members[j].key2 == members[i].key2) {
                    m = std::min<uint32_t>(m, (uint32_t)members[j].str.size() + dist(members[j].state));
                    j++;
                }
                k2.push_back({members[i].key2, std::min(m, 255u)});
                k2_range.push_back({i, j});
                i = j;
            }
            uint32_t bits = 4;
            if (!global_mode)
                while ((4ull << (bits + 1)) <= tm2_bytes) bits++;   // 2^bits buckets x 2 slots x 2 bytes <= tm2_bytes
            else
                while ((size_t)(2u << bits) * 7 / 10 < k2.size()) bits++;
            bool placed2;
            if (global_mode) {
                placed2 = place_all(k2, bits, tm2);
            } else {
                ph_sizes(k2.size(), nb2, ns2);
                placed2 = (uint64_t)(nb2 + ns2) * 2u <= tm2_bytes && ph_build(k2, true, nb2, ns2, d2, e2);
                if (!placed2) nb2 = ns2 = 0;
            }
            if (placed2) {
                tm2_bits = global_mode ? bits : 1u;
                for (size_t i = 0; i < k2.size() && ok; i++)
                    for (size_t j = k2_range[i].first; j < k2_range[i].second; j++) {
                        Level level(1, {members[j].state, members[j].str});
                        descend(level, k2[i].m);   // no-op when the merged m is not beyond the member's depth
                        for (const auto &it : level) {
                            if (dist(it.first) == kInf) continue;
                            const uint32_t h = hash_t3(k2[i].key ^ kT3Seed2, le32(it.second, k2[i].m - 4u)) >> out.t3_shift;
                            t3[h >> 5] |= 1u << (h & 31);
                        }
                    }
            } else {
                tm2.clear();
            }
        }
        // T3 holds the windows of the last level only when the level before it is verified by a
        // tagged perfect-hash look-up (mode 0 with level 2); otherwise the level-1 windows as well
        if (ok && (global_mode || !ns2))
            for (uint32_t h : l1_bits) t3[h >> 5] |= 1u << (h & 31);
        if (ok) {
            out.has_t3 = 1;
            out.tm_bits = tm_bits;
            out.tm2_bits = tm2_bits;
            out.mode = global_mode ? 2u : 0u;
            if (!global_mode) t2_bits = 0;   // the complete shared-memory Tm stands in for T2
            break;
        }
        // too many prefixes for this Tm, or not a tree
        const bool paths_overflow = visited > kPathLimit;
        out.t3_shift = 32;
        if (attempt == 1 || paths_overflow) { t3_bits = 0; tm2_bits = 0; }
    }
    if (!out.has_t3) {   // no two-point checks: T2 alone filters
        t3_bits = 0;
        tm2_bits = 0;
        out.t3_shift = 32;
        out.mode = 1;
        global_mode = false;
        tm.clear();
        tm2.clear();
    }
    if (t2_bits) out.t2_shift = t2_shift;

    // ---- images.  Shared memory: T1 + (Tm, Tm2, T3 | T2) -- or, in global mode, T2 alone; global
    // memory (mode 2): T1, Tm, Tm2, T3.
    const uint32_t tm_bytes = out.has_t3 ? (uint32_t)tm.size() * 2 : 0, tm2_bytes_used = (uint32_t)tm2.size() * 2;
    uint32_t off = 0;
    if (!global_mode) {
        out.off_t1 = off;
        off = align128(off + 65536);
        out.off_t2 = off;
        off = align128(off + t2_bits / 8);
        out.off_tm = out.off_tm2 = off;   // (cuckoo tables exist in global mode only)
        if (out.has_t3) {
            out.nb1 = nb1;
            out.ns1 = ns1;
            out.nb2 = nb2;
            out.ns2 = ns2;
            out.off_d1 = off;
            off = align128(off + nb1 * 2);
            out.off_e1 = off;
            off = align128(off + ns1 * 2);
            out.off_d2 = off;
            off = align128(off + nb2 * 2);
            out.off_e2 = off;
            off = align128(off + ns2 * 2);
        }
        out.off_t3 = off;
        off = align128(off + t3_bits / 8);
        out.image.assign(off, 0);
        if (out.mode == 0 && !any_short && !getenv("PFAC_NO_W3")) {
            // third-window planes: pairs at bytes 4-5 / 5-6 of every path, and the exceptions for the patterns
            // that end before them (depth-first to depth 7; an automaton with too many paths gets planes that
            // pass everything)
            std::vector<uint8_t> w3(65536, 0);
            uint64_t visits = 0;
            bool flood = false;
            struct Node { int32_t state; uint32_t depth; uint8_t byte; };
            std::vector<Node> stack;
            uint8_t path[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            for (int b = kCharSet - 1; b >= 0; b--)
                if (s0(b) >= 0) stack.push_back({s0(b), 1u, (uint8_t)b});
            while (!stack.empty() && !flood) {
                const Node nd = stack.back();
                stack.pop_back();
                if (++visits > kPathLimit) { flood = true; break; }
                path[nd.depth - 1] = nd.byte;
                if (nd.depth == 6) w3[t1_index(path[4], path[5])] |= kT1P45;
                if (nd.depth == 7) w3[t1_index(path[5], path[6])] |= kT1P56;
                if (g.is_final(nd.state)) {
                    if (nd.depth == 4 || nd.depth == 5) w3[t1_index(path[2], path[3])] |= kT1ShX;
                    if (nd.depth == 5 || nd.depth == 6) w3[t1_index(path[3], path[4])] |= kT1ShX;
                }
                if (nd.depth < 7)
                    for (uint32_t e = g.end(nd.state); e > g.begin(nd.state); e--)
                        stack.push_back({g.edges[e - 1].next, nd.depth + 1, (uint8_t)g.edges[e - 1].byte});
            }
            for (size_t i = 0; i < 65536; i++) t1[i] |= flood ? (uint8_t)(kT1P45 | kT1P56) : w3[i];
            out.has_w3 = 1;
        }
        memcpy(out.image.data() + out.off_t1, t1.data(), 65536);
        if (t2_bits) memcpy(out.image.data() + out.off_t2, t2.data(), t2_bits / 8);
        if (out.has_t3) {
            memcpy(out.image.data() + out.off_d1, d1.data(), nb1 * 2);
            memcpy(out.image.data() + out.off_e1, e1.data(), ns1 * 2);
            if (ns2) {
                memcpy(out.image.data() + out.off_d2, d2.data(), nb2 * 2);
                memcpy(out.image.data() + out.off_e2, e2.data(), ns2 * 2);
            }
            memcpy(out.image.data() + out.off_t3, t3.data(), t3_bits / 8);
        }
    } else {
        out.off_t2 = 0;
        out.image.assign(align128(t2_bits / 8), 0);
        if (t2_bits) memcpy(out.image.data(), t2.data(), t2_bits / 8);
        out.off_t1 = 0;   // offsets below are into gimage
        off = 65536;
        out.off_tm = off;
        off = align128(off + tm_bytes);
        out.off_tm2 = off;
        off = align128(off + tm2_bytes_used);
        out.off_t3 = off;
        off = align128(off + t3_bits / 8);
        out.gimage.assign(off, 0);
        memcpy(out.gimage.data(), t1.data(), 65536);
        memcpy(out.gimage.data() + out.off_tm, tm.data(), tm_bytes);
        if (tm2_bits) memcpy(out.gimage.data() + out.off_tm2, tm2.data(), tm2_bytes_used);
        memcpy(out.gimage.data() + out.off_t3, t3.data(), t3_bits / 8);
    }
    if (out.has_t3) {
        for (uint32_t w : t3) out.t3_set += (uint32_t)__builtin_popcount(w);
        for (uint16_t e : tm) out.tm_set += e ? 1u : 0u;
        for (uint16_t e : tm2) out.tm2_set += e ? 1u : 0u;
        if (!global_mode) {
            for (uint16_t e : e1) out.tm_set += (e >> 8) ? 1u : 0u;
            if (ns2)
                for (uint16_t e : e2) out.tm2_set += (e >> 8) ? 1u : 0u;
        }
    }
    for (uint8_t b : t1) out.t1_set += b & kT1P01;
    if (t2_bits)
        for (uint32_t w : t2) out.t2_set += (uint32_t)__builtin_popcount(w);
}

void derive_patdir(const Partition &P, PatDir &out)
{
    out = PatDir();
    if (P.max_len < 1 || P.max_len > 64 || P.n_final < 1 || P.s0.empty()) return;
    Graph g;
    build_graph(P, g);
    // depth-first over the trie; every state must be reached exactly once (a tree) and no deeper than max_len
    struct Item { int32_t state; uint32_t depth; uint8_t byte; };
    std::vector<Item> stack;
    std::vector<uint8_t> path((size_t)P.max_len + 1);
    std::vector<uint8_t> seen((size_t)g.n_states, 0);
    std::vector<uint8_t> pool;
    struct Ent { uint64_t h; uint32_t id, len, off; };
    std::vector<Ent> ents;
    for (int b = kCharSet - 1; b >= 0; b--)
        if (P.s0[(size_t)b] >= 0) stack.push_back({P.s0[(size_t)b], 1u, (uint8_t)b});
    while (!stack.empty()) {
        const Item it = stack.back();
        stack.pop_back();
        if (it.state >= g.n_states || it.depth > (uint32_t)P.max_len || seen[(size_t)it.state]) return;   // not a tree of that depth
        seen[(size_t)it.state] = 1;
        path[it.depth - 1] = it.byte;
        if (g.is_final(it.state)) {
            uint64_t h = 0;
            for (uint32_t i = 0; i < it.depth; i++) h = dir_hash_step(h, path[i]);
            if (pool.size() + it.depth >= (1u << 25)) return;
            ents.push_back({h, (uint32_t)P.idmap[(size_t)it.state], it.depth, (uint32_t)pool.size()});
            pool.insert(pool.end(), path.begin(), path.begin() + it.depth);
            out.len_mask |= 1ull << (it.depth - 1);
        }
        for (uint32_t e = g.end(it.state); e > g.begin(it.state); e--)
            stack.push_back({g.edges[e - 1].next, it.depth + 1, (uint8_t)g.edges[e - 1].byte});
    }
    if ((int32_t)ents.size() != P.n_final) { out = PatDir(); return; }   // a final state nobody reaches: leave it to the walk
    uint32_t n_slots = 64;
    while (n_slots < 2 * ents.size()) n_slots *= 2;
    out.n_slots = n_slots;
    out.off_pool = n_slots * 16u;
    out.image.assign((size_t)out.off_pool + ((pool.size() + 15) & ~(size_t)15), 0);
    uint32_t *dir = reinterpret_cast<uint32_t *>(out.image.data());
    for (uint32_t i = 0; i < n_slots; i++) dir[4 * i + 3] = 0xFFFFFFFFu;
    for (const Ent &e : ents) {
        uint32_t sl = dir_slot(e.h, n_slots);
        while (dir[4 * sl + 3] != 0xFFFFFFFFu) sl = (sl + 1) & (n_slots - 1);
        dir[4 * sl] = (uint32_t)e.h;
        dir[4 * sl + 1] = (uint32_t)(e.h >> 32);
        dir[4 * sl + 2] = e.id;
        dir[4 * sl + 3] = (e.len << 25) | e.off;
    }
    if (!pool.empty()) memcpy(out.image.data() + out.off_pool, pool.data(), pool.size());
}

int pattern_lengths(const Partition &P, std::vector<int32_t> &len)
{
    int32_t max_id = -1;
    for (int32_t id : P.idmap) {
        if (id < 0) return set_error(PFAC_ERR_ARG, "pattern id %d is negative", id);
        max_id = std::max(max_id, id);
    }
    len.assign((size_t)(max_id + 1), 0);
    if (P.n_final < 1 || P.s0.size() != (size_t)kCharSet) return PFAC_OK;
    Graph g;
    build_graph(P, g);
    // depth-first from the root; a state reached twice (shared states or a cycle) has no single depth
    struct Item { int32_t state; int32_t depth; };
    std::vector<Item> stack;
    std::vector<uint8_t> seen((size_t)g.n_states, 0);
    for (int b = 0; b < kCharSet; b++)
        if (P.s0[(size_t)b] >= 0) stack.push_back({P.s0[(size_t)b], 1});
    while (!stack.empty()) {
        const Item it = stack.back();
        stack.pop_back();
        if (it.state >= g.n_states) continue;   // no such state: no lookup reaches it
        if (seen[(size_t)it.state])
            return set_error(PFAC_ERR_ARG, "the automaton is not a tree (state %d is reached twice): pattern lengths are undefined",
                             it.state);
        seen[(size_t)it.state] = 1;
        if (g.is_final(it.state)) {
            const int32_t id = P.idmap[(size_t)it.state];
            if (len[(size_t)id]) return set_error(PFAC_ERR_ARG, "pattern id %d is reported by two final states", id);
            len[(size_t)id] = it.depth;
        }
        for (uint32_t e = g.begin(it.state); e < g.end(it.state); e++) stack.push_back({g.edges[e].next, it.depth + 1});
    }
    // per-pattern case rules: every member of a group reports its owner's length (members never exceed their
    // owner's id, the last line of the group)
    const Partition::CaseGroups &cg = P.groups;
    for (size_t m = 0; m < cg.id.size(); m++)
        if (cg.id[m] >= 0 && (size_t)cg.id[m] < len.size()) len[(size_t)cg.id[m]] = cg.len[m];
    return PFAC_OK;
}

// Host model of the directory look-up (tests): id of the pattern text[0, d), -1 if it is none.
int64_t patdir_lookup(const PatDir &pd, const uint8_t *text, uint32_t d)
{
    if (!pd.n_slots || d < 1 || d > 64) return -1;
    uint64_t h = 0;
    for (uint32_t i = 0; i < d; i++) h = dir_hash_step(h, text[i]);
    const uint32_t *dir = reinterpret_cast<const uint32_t *>(pd.image.data());
    for (uint32_t sl = dir_slot(h, pd.n_slots);; sl = (sl + 1) & (pd.n_slots - 1)) {
        const uint32_t w = dir[4 * sl + 3];
        if (w == 0xFFFFFFFFu) return -1;
        if (dir[4 * sl] == (uint32_t)h && dir[4 * sl + 1] == (uint32_t)(h >> 32) && (w >> 25) == d &&
            !memcmp(pd.image.data() + pd.off_pool + (w & 0x1FFFFFFu), text, d))
            return dir[4 * sl + 2];
    }
}

namespace {

// The detector's stage 1 on the bytes t[0, len) (bytes past len read as 0, like stale shared memory
// may read as anything): P01 of the first pair, and either the short plane or P12 and P23 further on.
bool stage1_pass(const Derived &d, const uint8_t *t, size_t len, bool odd)
{
    if (d.mode == 2) {   // global mode: stage 1 is T2 over the 4-byte prefix (no pattern is shorter than 4)
        if (len < 4) return false;
        const uint32_t *t2 = reinterpret_cast<const uint32_t *>(d.image.data() + d.off_t2);
        return d.t2_shift >= 32 || t2_pass(t2, le32(t), d.t2_shift);
    }
    const uint8_t *t1 = d.image.data() + d.off_t1;
    auto at = [&](size_t i) { return i < len ? (uint32_t)t[i] : 0u; };
    if (d.mode == 0) {
        // mode 0 probes T1 at even offsets of the (16-byte aligned) input stream only.  A start at an
        // even offset sees its bytes 0-1 and 2-3, one at an odd offset its bytes 1-2 and 3-4.
        if (!odd) {
            const uint32_t v0 = t1[t1_index(at(0), at(1))], v2 = t1[t1_index(at(2), at(3))];
            if (d.has_w3)   // (no Short plane: its bit is ShX)
                return (v0 & kT1P01) && (v2 & kT1P23) && ((v2 & kT1ShX) || (t1[t1_index(at(4), at(5))] & kT1P45));
            return (v0 & kT1P01) && ((v0 & kT1Short) || (v2 & kT1P23));
        }
        const uint32_t v1 = t1[t1_index(at(1), at(2))], v3 = t1[t1_index(at(3), at(4))];
        if (d.has_w3)
            return (v1 & kT1ShortC) || ((v1 & kT1P12) && (v3 & kT1P34) && ((v3 & kT1ShX) || (t1[t1_index(at(5), at(6))] & kT1P56)));
        return (v1 & kT1ShortC) || ((v1 & kT1P12) && (v3 & kT1P34));
    }
    const uint32_t v0 = t1[t1_index(at(0), at(1))];
    if (!(v0 & kT1P01)) return false;
    if (v0 & kT1Short) return true;
    return (t1[t1_index(at(1), at(2))] & kT1P12) && (t1[t1_index(at(2), at(3))] & kT1P23);
}

// The detector's stage 2 on the bytes t[0, len): may a pattern start here?  (stage 1 = T1 passed)
// `stage` (optional) receives how far the start got: 1 bypass, 2 T2/Tm pass, 3 level-1 window pass,
// 4 level-2 pass.
bool stage2_pass(const Derived &d, const uint8_t *t, size_t len, bool odd, int *stage)
{
    const uint8_t *img = d.mode == 2 ? d.gimage.data() : d.image.data();   // where T1/Tm/Tm2/T3 live
    const uint8_t *t1 = img + d.off_t1;
    const uint32_t *t2 = reinterpret_cast<const uint32_t *>(d.image.data() + d.off_t2);
    const uint16_t *tm = reinterpret_cast<const uint16_t *>(img + d.off_tm);
    const uint16_t *tm2 = reinterpret_cast<const uint16_t *>(img + d.off_tm2);
    const uint32_t *t3 = reinterpret_cast<const uint32_t *>(img + d.off_t3);
    if (stage) *stage = 1;
    if (len < 4) return true;   // fewer than 4 readable bytes: settled as a candidate
    const uint32_t w4 = le32(t);
    if (d.mode == 0) {
        // short patterns (<= 3 bytes) are not in the prefix tables: their starts become candidates
        if (d.has_short) {
            if (!odd && (t1[t1_index(w4 & 255u, (w4 >> 8) & 255u)] & kT1Short)) return true;
            if (odd && (t1[t1_index((w4 >> 8) & 255u, (w4 >> 16) & 255u)] & kT1ShortC)) return true;
        }
        const uint16_t *D1 = reinterpret_cast<const uint16_t *>(img + d.off_d1), *E1 = reinterpret_cast<const uint16_t *>(img + d.off_e1);
        const uint32_t m1 = ph_lookup(D1, E1, d.nb1, d.ns1, w4, ph_mix(w4));
        if (!m1 || m1 > len) return false;
        if (stage) *stage = 2;
        const uint32_t w1 = le32(t + m1 - 4);
        if (!d.ns2) {
            if (!bit(t3, hash_t3(w4, w1) >> d.t3_shift)) return false;
            if (stage) *stage = 3;
            return true;
        }
        const uint16_t *D2 = reinterpret_cast<const uint16_t *>(img + d.off_d2), *E2 = reinterpret_cast<const uint16_t *>(img + d.off_e2);
        const uint32_t key2 = hash_key2(w4, w1);
        const uint32_t m2 = ph_lookup(D2, E2, d.nb2, d.ns2, key2, key2);
        if (!m2 || m2 > len) return false;
        if (stage) *stage = 3;
        if (!bit(t3, hash_t3(key2 ^ kT3Seed2, le32(t + m2 - 4)) >> d.t3_shift)) return false;
        if (stage) *stage = 4;
        return true;
    }
    if (d.has_short && (t1[t1_index(w4 & 255u, (w4 >> 8) & 255u)] & kT1Short)) return true;
    if (!d.has_t3) {
        if (d.t2_shift < 32 && !t2_pass(t2, w4, d.t2_shift)) return false;
        if (stage) *stage = 2;
        return true;
    }
    const uint32_t m1 = tm_lookup(tm, w4, d.tm_bits);
    if (!m1 || m1 > len) return false;
    if (stage) *stage = 2;
    const uint32_t w1 = le32(t + m1 - 4);
    if (!bit(t3, hash_t3(w4, w1) >> d.t3_shift)) return false;
    if (stage) *stage = 3;
    if (!d.tm2_bits) return true;
    const uint32_t key2 = hash_key2(w4, w1);
    const uint32_t m2 = tm_lookup(tm2, key2, d.tm2_bits);
    if (!m2 || m2 > len) return false;
    if (!bit(t3, hash_t3(key2 ^ kT3Seed2, le32(t + m2 - 4)) >> d.t3_shift)) return false;
    if (stage) *stage = 4;
    return true;
}

}  // namespace

void derive_profile(const Partition &P, const Derived &d, const uint8_t *text, size_t n, uint64_t out[12])
{
    for (int i = 0; i < 12; i++) out[i] = 0;
    const size_t maxlen = (size_t)std::max(P.max_len, 1);
    uint64_t slices = 0;
    size_t last_slice = (size_t)-1;
    for (size_t i = 0; i < n; i++) {
        out[0]++;
        if (!stage1_pass(d, text + i, n - i, (i & 1) != 0)) continue;
        out[1]++;   // stage 1 survivors
        int stage = 0;
        const bool pass = stage2_pass(d, text + i, std::min(n - i, maxlen), (i & 1) != 0, &stage);
        if (stage >= 2) out[2]++;   // T2 / Tm found the prefix
        if (stage >= 3) out[3]++;   // level-1 window passed
        if (stage >= 4) out[4]++;   // level-2 window passed
        if (!pass) continue;
        if (stage == 1) out[5]++;   // bypass (short patterns / end of input)
        out[6]++;   // starts left as candidates
        if (i / 512 != last_slice) {
            last_slice = i / 512;
            slices++;
        }
    }
    out[7] = slices;   // 512-byte slices flagged
    out[8] = (n + 511) / 512;
}

int derive_selfcheck(const Partition &P, const Derived &d)
{
    if (d.image.empty()) return 100;
    const uint8_t *t1 = (d.mode == 2 ? d.gimage.data() : d.image.data()) + d.off_t1;
    auto is_final = [&](int32_t s) { return s >= 0 && s < P.n_final; };
    // T1 is exact over the first two bytes; T1s covers every pair that can end a pattern of <= 3 bytes
    for (int b0 = 0; b0 < kCharSet; b0++) {
        const int32_t s1 = P.s0.empty() ? -1 : P.s0[(size_t)b0];
        for (int b1 = 0; b1 < kCharSet; b1++) {
            const int32_t s2 = s1 < 0 ? -1 : P.lookup(s1, b1);
            const uint32_t v = t1[t1_index((uint32_t)b0, (uint32_t)b1)];
            const bool pass = (v & kT1P01) != 0;
            const bool want = s1 >= 0 && (is_final(s1) || s2 >= 0);
            if (want != pass) return want ? 3 : 4;
            if (!want) continue;
            bool shortp = is_final(s1) || is_final(s2);
            if (s2 >= 0 && !shortp)
                for (int b2 = 0; b2 < kCharSet && !shortp; b2++) shortp = is_final(P.lookup(s2, b2));
            if (shortp && !(d.has_short && (v & kT1Short))) return 7;
        }
    }
    // stage 2 must pass every pattern: run it over each pattern's own bytes (strings of the
    // breadth-first tree from the root row)
    const int32_t n_states = std::max(P.state_num, 0);
    std::vector<int32_t> par((size_t)n_states, -2), order;
    std::vector<uint8_t> pbyte((size_t)n_states, 0);
    for (int b = 0; b < kCharSet; b++) {
        const int32_t s1 = P.s0.empty() ? -1 : P.s0[(size_t)b];
        if (s1 >= 0 && s1 < n_states && par[(size_t)s1] == -2) {
            par[(size_t)s1] = -1;
            pbyte[(size_t)s1] = (uint8_t)b;
            order.push_back(s1);
        }
    }
    for (size_t i = 0; i < order.size(); i++)
        for (int b = 0; b < kCharSet; b++) {
            const int32_t y = P.lookup(order[i], b);
            if (y >= 0 && y < n_states && par[(size_t)y] == -2) {
                par[(size_t)y] = order[i];
                pbyte[(size_t)y] = (uint8_t)b;
                order.push_back(y);
            }
        }
    std::vector<uint8_t> str;
    for (int32_t f = 0; f < std::min(P.n_final, n_states); f++) {
        if (par[(size_t)f] == -2) continue;   // unreachable final (duplicate pattern)
        str.clear();
        for (int32_t x = f; x >= 0; x = par[(size_t)x]) str.push_back(pbyte[(size_t)x]);
        std::reverse(str.begin(), str.end());
        // at either alignment, and whatever follows the pattern in the input
        for (int odd = 0; odd < 2; odd++)
            for (uint8_t fill : {(uint8_t)0x00, (uint8_t)0xFF, (uint8_t)0x5A}) {
                std::vector<uint8_t> padded(str);
                padded.resize(str.size() + 8, fill);
                int stage = 0;
                if (!stage1_pass(d, padded.data(), padded.size(), odd != 0)) return 8;
                if (!stage2_pass(d, padded.data(), str.size(), odd != 0, &stage)) return 10 + stage;
            }
    }
    return 0;
}

// The directory must answer like the walk: for every final state's own string, and for variations of it
// (a byte changed, a byte dropped), "id of the pattern text[0, d)" equals what SUBSEG_MATCH's transitions say.
int patdir_selfcheck(const Partition &P, const PatDir &pd)
{
    if (!pd.n_slots) return 0;
    const int32_t n_states = std::max(P.state_num, 0);
    auto walk_id = [&](const uint8_t *t, uint32_t d) -> int64_t {   // master_kernel.cu:41-70 over t[0, d)
        int32_t st = P.s0.empty() ? -1 : P.s0[t[0]];
        for (uint32_t i = 1; i < d && st >= 0; i++) st = P.lookup(st, t[i]);
        return st >= 0 && st < P.n_final ? (int64_t)(uint32_t)P.idmap[(size_t)st] : -1;
    };
    std::vector<int32_t> par((size_t)n_states, -2), order;
    std::vector<uint8_t> pbyte((size_t)n_states, 0);
    for (int b = 0; b < kCharSet; b++) {
        const int32_t s1 = P.s0.empty() ? -1 : P.s0[(size_t)b];
        if (s1 >= 0 && s1 < n_states && par[(size_t)s1] == -2) {
            par[(size_t)s1] = -1;
            pbyte[(size_t)s1] = (uint8_t)b;
            order.push_back(s1);
        }
    }
    Graph g;
    build_graph(P, g);
    for (size_t i = 0; i < order.size(); i++)
        for (uint32_t e = g.begin(order[i]); e < g.end(order[i]); e++) {
            const int32_t y = g.edges[e].next;
            if (y >= 0 && y < n_states && par[(size_t)y] == -2) {
                par[(size_t)y] = order[i];
                pbyte[(size_t)y] = (uint8_t)g.edges[e].byte;
                order.push_back(y);
            }
        }
    std::vector<uint8_t> str;
    uint32_t k = 0;
    for (int32_t f = 0; f < std::min(P.n_final, n_states); f++, k++) {
        if (par[(size_t)f] == -2) return 1;   // the directory exists only when every final state is reachable
        str.clear();
        for (int32_t x = f; x >= 0; x = par[(size_t)x]) str.push_back(pbyte[(size_t)x]);
        std::reverse(str.begin(), str.end());
        const uint32_t d = (uint32_t)str.size();
        if (d > 64) return 2;
        if (patdir_lookup(pd, str.data(), d) != walk_id(str.data(), d)) return 3;
        if (!((pd.len_mask >> (d - 1)) & 1ull)) return 4;
        for (uint32_t dd = 1; dd < d; dd++)   // its proper prefixes (patterns themselves or not)
            if (((pd.len_mask >> (dd - 1)) & 1ull) && patdir_lookup(pd, str.data(), dd) != walk_id(str.data(), dd)) return 5;
        std::vector<uint8_t> v(str);
        v[k % d] ^= (uint8_t)(1u << (k % 7));   // one byte changed
        if (patdir_lookup(pd, v.data(), d) != walk_id(v.data(), d)) return 6;
    }
    return 0;
}

void derive_walk_cache(const Partition &P, uint32_t budget_bytes, WalkCache &out)
{
    out = WalkCache();
    Graph g;
    build_graph(P, g);
    std::vector<uint32_t> keys2, keys3;
    std::vector<int32_t> st2, st3;
    bool too_many = false;
    for (int b0 = 0; b0 < kCharSet && !too_many; b0++) {
        const int32_t s1 = P.s0.empty() ? -1 : P.s0[(size_t)b0];
        if (s1 < 0) continue;
        for (uint32_t e1 = g.begin(s1); e1 < g.end(s1); e1++) {
            const uint32_t pair = (uint32_t)b0 | ((uint32_t)g.edges[e1].byte << 8);
            keys2.push_back(pair | kWalkDepth2);
            st2.push_back(g.edges[e1].next);
            const int32_t s2 = g.edges[e1].next;
            for (uint32_t e2 = g.begin(s2); e2 < g.end(s2); e2++) {
                keys3.push_back(pair | ((uint32_t)g.edges[e2].byte << 16) | kWalkDepth3);
                st3.push_back(g.edges[e2].next);
            }
            if (keys2.size() + keys3.size() > (1u << 20)) { too_many = true; break; }
        }
    }
    // the root row is always there; depth 2 and then depth 3 as long as they fit the budget
    for (int depth = too_many ? 1 : 3; depth >= 1; depth--) {
        std::vector<uint32_t> keys;
        std::vector<int32_t> states;
        if (depth >= 2) { keys = keys2; states = st2; }
        if (depth >= 3) { keys.insert(keys.end(), keys3.begin(), keys3.end()); states.insert(states.end(), st3.begin(), st3.end()); }
        uint32_t nb = 0, ns = 0;
        std::vector<uint16_t> D;
        std::vector<uint32_t> slot_of;
        if (!keys.empty()) {
            ph_sizes(keys.size(), nb, ns);
            if (1024u + nb * 2u + (uint64_t)ns * 8u > budget_bytes) continue;
            if (!ph_place(keys, false, nb, ns, D, slot_of)) continue;
        }
        out.depth = keys.empty() ? 1u : (uint32_t)depth;
        out.nb = nb;
        out.ns = ns;
        out.off_d = 1024;
        out.off_e = (1024u + nb * 2u + 127u) & ~127u;
        out.image.assign(out.off_e + (size_t)ns * 8u, 0);
        int32_t *s0 = reinterpret_cast<int32_t *>(out.image.data());
        for (int b = 0; b < kCharSet; b++) s0[b] = P.s0.empty() ? -1 : P.s0[(size_t)b];
        if (!keys.empty()) {
            memcpy(out.image.data() + out.off_d, D.data(), nb * 2u);
            uint32_t *E = reinterpret_cast<uint32_t *>(out.image.data() + out.off_e);
            for (uint32_t i = 0; i < ns; i++) { E[2 * i] = 0xFFFFFFFFu; E[2 * i + 1] = 0xFFFFFFFFu; }   // no key has depth byte 0xFF
            for (size_t i = 0; i < keys.size(); i++) {
                E[2 * slot_of[i]] = keys[i];
                E[2 * slot_of[i] + 1] = (uint32_t)states[i];
            }
        }
        return;
    }
}

// host model of the dense kernel's cached walk: the state after the first `depth` bytes of t (depth <= cache depth), -1 = none
int32_t walk_cache_lookup(const WalkCache &w, const uint8_t *t, uint32_t depth)
{
    const int32_t *s0 = reinterpret_cast<const int32_t *>(w.image.data());
    if (depth == 1) return s0[t[0]];
    const uint32_t key = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | (depth == 3 ? ((uint32_t)t[2] << 16) | kWalkDepth3 : kWalkDepth2);
    const uint16_t *D = reinterpret_cast<const uint16_t *>(w.image.data() + w.off_d);
    const uint32_t *E = reinterpret_cast<const uint32_t *>(w.image.data() + w.off_e);
    const uint32_t slot = ph_slot(key, D[mulhi32(ph_mix(key), w.nb)], w.ns);
    return E[2 * slot] == key ? (int32_t)E[2 * slot + 1] : -1;
}

}  // namespace pfac
