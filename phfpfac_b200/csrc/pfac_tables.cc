// Host-side table construction: pattern file -> sorted patterns -> PFAC trie -> PHF arrays.
//
// Produces, bit for bit, what the reference's create_PFAC_table_reorder()
// (CreateTable/create_table_reorder.c:201-378) and FFDM() (PHF/phf.c:151-291) produce, but
// with dynamic limits and near-linear time:
//   * the trie is built from the sorted list with a longest-common-prefix walk instead of a
//     dense state x 256 array (the reference pre-allocates 4,000,000 x 1 KiB rows,
//     create_table_reorder.c:10,306-311);
//   * SortRows' O(R^2) exchange sort (phf.c:126-139), whose tie order decides the packing, is
//     reproduced exactly by moving elements along the chain of strict running maxima with a
//     max-segment-tree (O(R log R));
//   * the first-fit search (phf.c:188-195) tests 64 candidate slots per step against the row's
//     columns with word-wide occupancy masks, and skips full regions through a hierarchical bitmap,
//     instead of trying every offset (100,000 patterns: 1.7 s at width 256, 9 s at width 4096
//     where one offset at a time took 20 minutes).
// tests/test_tables_*.py pin this against the reference's own code (oracle/_ref) and the
// plain-C restatement (oracle/pfac_oracle.c).
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "pfac_derive.h"
#include "pfac_internal.h"

namespace pfac {

static thread_local std::string g_last_error;

int set_error(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

int width_bits(int width)
{
    if (width < 1 || width > 4096 || (width & (width - 1))) return -1;   // phf.c:161
    int b = 0;
    while ((width >> b) != 1) b++;                                        // master_kernel.cu:398
    return b;
}

// master_kernel.cu:52-64
int32_t Partition::lookup(int32_t state, int32_t byte) const
{
    int wb = width_bits(width);
    int32_t key = (int32_t)(((uint32_t)state << 8) + (uint32_t)byte);
    int32_t row = key >> wb;
    int32_t col = key & ((1 << wb) - 1);
    if (row < 0 || row >= (int32_t)r.size()) return -1;
    int32_t index = r[row] + col;
    if (index < 0 || index >= ht_size) return -1;
    return HT[index] == row ? val[index] : -1;
}

namespace {

struct Pattern {
    const unsigned char *p;
    int len;
    int id;   // 1-based line number, create_table_reorder.c:100
};

// create_table_reorder.c:21-45 (comp_pat): memcmp over the common length, then shorter first.
inline int comp_pat(const Pattern &a, const Pattern &b)
{
    int m = a.len < b.len ? a.len : b.len;
    int res = memcmp(a.p, b.p, (size_t)m);
    if (res) return res;
    return a.len < b.len ? -1 : (a.len > b.len ? 1 : 0);
}

// create_table_reorder.c:53-122 (read_pattern) over a memory image of the file.
int read_patterns(const unsigned char *buf, size_t len, std::vector<Pattern> &out)
{
    if (len == 0) return set_error(PFAC_ERR_PATTERN_TOO_LONG, "pattern file is empty");
    size_t i = 0;
    while (i < len) {
        const unsigned char *nl = (const unsigned char *)memchr(buf + i, '\n', len - i);
        if (!nl)   // the reference spins on EOF until the 1024 limit trips (:71-77)
            return set_error(PFAC_ERR_PATTERN_TOO_LONG,
                             "pattern %zu: file does not end with a newline", out.size() + 1);
        size_t plen = (size_t)(nl - (buf + i));
        if (plen > (size_t)kMaxPatternBytes)
            return set_error(PFAC_ERR_PATTERN_TOO_LONG, "Pattern %zu length over 1024.", out.size() + 1);
        if (plen == 0)
            return set_error(PFAC_ERR_EMPTY_PATTERN, "pattern %zu is empty", out.size() + 1);
        out.push_back(Pattern{buf + i, (int)plen, (int)out.size() + 1});
        i += plen + 1;
    }
    return PFAC_OK;
}

// ctdef.h:37-99 (fgetc_ext): a backslash and what follows merge into one byte.  Returns the byte
// (0..255), kEol for a raw newline, -1 at the end of the buffer.  "%3o" / "%2x" = up to 3 octal /
// 2 hex digits (scanf's white-space skip before %x is kept, its sign / 0x prefix handling is not).
constexpr int kEol = 0x10A;   // ctdef.h:13
int next_escaped(const unsigned char *buf, size_t len, size_t &i)
{
    const int ch0 = i < len ? buf[i] : -1;
    i++;
    if (ch0 == '\\') {
        const int ch1 = i < len ? buf[i] : -1;
        i++;
        if (ch1 < 0) return ch0;                                  // :50-52
        if (ch1 >= '0' && ch1 <= '9') {                           // :55-59
            int value = 0, nd = 0;
            i--;
            while (nd < 3 && i < len && buf[i] >= '0' && buf[i] <= '7') { value = value * 8 + (buf[i] - '0'); i++; nd++; }
            return value & 255;
        }
        switch (ch1) {                                            // :61-91
        case 'a': return '\a';
        case 'b': return '\b';
        case 't': return '\t';
        case 'n': return '\n';
        case 'v': return '\v';
        case 'f': return '\f';
        case 'r': return '\r';
        case '\'': case '\"': case '\\': return ch1;
        case 'x': {
            int value = 0, nd = 0;
            while (i < len && (buf[i] == ' ' || (buf[i] >= 9 && buf[i] <= 13))) i++;
            while (nd < 2 && i < len) {
                const int c = buf[i];
                int d;
                if (c >= '0' && c <= '9') d = c - '0';
                else if (c >= 'a' && c <= 'f') d = c - 'a' + 10;
                else if (c >= 'A' && c <= 'F') d = c - 'A' + 10;
                else break;
                value = value * 16 + d;
                i++;
                nd++;
            }
            return value & 255;
        }
        default:                                                  // :87-90: not an escape
            i--;
            return ch0;
        }
    }
    if (ch0 == '\n') return kEol;                                 // :94-96
    return ch0;
}

// create_table_reorder.c:131-185 (read_pattern_ext): read_pattern through fgetc_ext.  The decoded
// bytes live in `arena` (never reallocated: a decoded pattern is not longer than its source).
int read_patterns_ext(const unsigned char *buf, size_t len, std::vector<unsigned char> &arena, std::vector<Pattern> &out)
{
    if (len == 0) return set_error(PFAC_ERR_PATTERN_TOO_LONG, "pattern file is empty");
    arena.clear();
    arena.reserve(len + 1);
    size_t i = 0;
    while (true) {
        const size_t start = arena.size();
        while (true) {
            if (i >= len)   // the reference spins on EOF until the 1024 limit trips (:155-158)
                return set_error(PFAC_ERR_PATTERN_TOO_LONG, "pattern %zu: file does not end with a newline", out.size() + 1);
            const int ch = next_escaped(buf, len, i);
            if (ch == kEol) break;
            if (arena.size() - start >= (size_t)kMaxPatternBytes)
                return set_error(PFAC_ERR_PATTERN_TOO_LONG, "Pattern %zu length over 1024.", out.size() + 1);
            arena.push_back((unsigned char)(ch & 255));
        }
        const size_t plen = arena.size() - start;
        if (plen == 0) return set_error(PFAC_ERR_EMPTY_PATTERN, "pattern %zu is empty", out.size() + 1);
        out.push_back(Pattern{arena.data() + start, (int)plen, (int)out.size() + 1});
        if (i >= len) break;
    }
    return PFAC_OK;
}

// PFAC_PATTERNS_CASELESS: ASCII 'A'-'Z' -> 'a'-'z', every other byte (0x80-0xFF included) unchanged
inline unsigned char ascii_fold(unsigned char c) { return (c >= 'A' && c <= 'Z') ? (unsigned char)(c | 0x20) : c; }

// create_table_reorder.c:277-378 (patternsToPFAC) for an already sorted slice.
// State numbering: finals 0..n-1 = index in the slice (:366), n unused, initial n+1 (:288),
// interior states from n+2 in creation order (:292,331-333).
// Because the slice is sorted (prefix before extension), the edges pattern i can follow are
// exactly those on the path of pattern i-1 up to their common prefix.
void build_trie(const Pattern *pats, int n, Partition &P)
{
    const int initial = n + 1;
    int state_count = n + 2;
    P.n_final = n;
    P.max_len = 0;
    P.min_len = 0;
    P.idmap.resize((size_t)n);
    std::vector<int32_t> &keys = P.keys, &next = P.next;
    std::vector<int32_t> path(1, initial);   // path[d] = state after d bytes of the previous pattern
    std::vector<size_t> edge;                // edge[d] = index of the transition path[d] -> path[d+1]
    const Pattern *prev = nullptr;
    for (int i = 0; i < n; i++) {
        const Pattern &cur = pats[i];
        P.idmap[(size_t)i] = cur.id;                                  // :318
        if (cur.len > P.max_len) P.max_len = cur.len;                 // :319-321
        if (P.min_len == 0 || cur.len < P.min_len) P.min_len = cur.len;
        int l = 0;
        if (prev) {
            int m = prev->len < cur.len ? prev->len : cur.len;
            while (l < m && prev->p[l] == cur.p[l]) l++;
        }
        path.resize((size_t)cur.len + 1);
        edge.resize((size_t)cur.len);
        for (int j = (l < cur.len - 1 ? l : cur.len - 1); j < cur.len - 1; j++) {   // :325-359
            int s = state_count++;
            keys.push_back(path[(size_t)j] * kCharSet + cur.p[j]);
            next.push_back(s);
            edge[(size_t)j] = keys.size() - 1;
            path[(size_t)j + 1] = s;
        }
        const int last = cur.len - 1;                                 // :362-366
        if (l == cur.len) {
            next[edge[(size_t)last]] = i;   // duplicate pattern: PFAC[state][ch] is overwritten
        } else {
            keys.push_back(path[(size_t)last] * kCharSet + cur.p[last]);
            next.push_back(i);
            edge[(size_t)last] = keys.size() - 1;
        }
        path[(size_t)cur.len] = i;
        prev = &cur;
    }
    P.state_num = state_count;                                        // :376
    // ReadKey (phf.c:98) visits keys in ascending order
    std::vector<size_t> order(keys.size());
    for (size_t k = 0; k < order.size(); k++) order[k] = k;
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return keys[a] < keys[b]; });
    std::vector<int32_t> k2(keys.size()), n2(keys.size());
    for (size_t k = 0; k < order.size(); k++) { k2[k] = keys[order[k]]; n2[k] = next[order[k]]; }
    keys.swap(k2);
    next.swap(n2);
    P.s0.assign(kCharSet, -1);                                        // main.cc:200
    for (size_t k = 0; k < keys.size(); k++)
        if (keys[k] / kCharSet == initial) P.s0[(size_t)(keys[k] % kCharSet)] = next[k];
}

// max-segment-tree over positions: first index >= from whose value is > thr
struct MaxTree {
    int N = 1;
    std::vector<int32_t> t;
    explicit MaxTree(const std::vector<int32_t> &leaf)
    {
        while (N < (int)leaf.size()) N <<= 1;
        t.assign((size_t)2 * N, -1);
        for (size_t i = 0; i < leaf.size(); i++) t[(size_t)N + i] = leaf[i];
        for (int i = N - 1; i >= 1; i--) t[(size_t)i] = std::max(t[(size_t)2 * i], t[(size_t)2 * i + 1]);
    }
    void set(int pos, int32_t v)
    {
        int i = pos + N;
        t[(size_t)i] = v;
        for (i >>= 1; i >= 1; i >>= 1) {
            int32_t m = std::max(t[(size_t)2 * i], t[(size_t)2 * i + 1]);
            if (t[(size_t)i] == m) break;
            t[(size_t)i] = m;
        }
    }
    int32_t top() const { return t[1]; }
    int first_greater(int from, int32_t thr) const
    {
        if (from >= N) return -1;
        int i = from + N;
        while (true) {
            if (t[(size_t)i] > thr) {
                while (i < N) {
                    i <<= 1;
                    if (t[(size_t)i] <= thr) i++;
                }
                return i - N;
            }
            while (i & 1) i >>= 1;
            i++;
            if ((i & (i - 1)) == 0) return -1;
        }
    }
};

// occupancy bitmap with two summary levels: next free slot >= s, growable
struct SlotMap {
    std::vector<uint64_t> l0, l1, l2;   // l1 bit = l0 word full, l2 bit = l1 word full
    void ensure(size_t slot)
    {
        size_t w0 = slot / 64 + 1;
        if (w0 <= l0.size()) return;
        w0 = std::max(w0, l0.size() * 2);
        l0.resize(w0, 0);
        l1.resize(w0 / 64 + 1, 0);
        l2.resize(l1.size() / 64 + 1, 0);
    }
    bool used(size_t s)
    {
        ensure(s);
        return (l0[s >> 6] >> (s & 63)) & 1;
    }
    void mark(size_t s)
    {
        ensure(s);
        size_t w = s >> 6;
        l0[w] |= 1ULL << (s & 63);
        if (l0[w] == ~0ULL) {
            size_t w1 = w >> 6;
            l1[w1] |= 1ULL << (w & 63);
            if (l1[w1] == ~0ULL) l2[w1 >> 6] |= 1ULL << (w1 & 63);
        }
    }
    // 64 occupancy bits starting at an arbitrary slot
    uint64_t bits_at(size_t pos) const
    {
        const size_t w = pos >> 6, b = pos & 63;
        uint64_t v = l0[w] >> b;
        if (b) v |= l0[w + 1] << (64 - b);
        return v;
    }
    // phf.c:188-195 for a whole row at once: the first free slot s >= start such that s + d[i] is
    // free for every i (d = the row's other columns relative to its first).  Same answer as trying
    // the free slots one by one; here kFitWords x 64 candidate slots are tested per pass, one
    // column at a time over consecutive occupancy words.
    // (compiled three times; the loader picks the widest vector unit the host has: the word loops below are
    // the whole cost of wide tables -- 100,000 patterns at width 4096: 17 s -> 9 s with AVX-512)
    static constexpr int kFitWords = 32;
#if defined(__x86_64__) && defined(__GNUC__) && !defined(__clang__) && !defined(__SANITIZE_THREAD__)   // (ifunc resolvers run before TSan is up)
    __attribute__((target_clones("avx512f", "avx2", "default")))
#endif
    size_t first_fit(size_t start, const uint32_t *d, int nd)
    {
        size_t s = next_free(start);
        const size_t reach = (nd ? (size_t)d[nd - 1] : 0) + 64 * (kFitWords + 2);
        while (true) {
            const size_t w = s >> 6;
            ensure((w << 6) + reach);
            uint64_t cand[kFitWords], any = 0;
            for (int j = 0; j < kFitWords; j++) cand[j] = ~l0[w + (size_t)j];
            cand[0] &= ~0ULL << (s & 63);
            for (int j = 0; j < kFitWords; j++) any |= cand[j];
            for (int i = 0; i < nd && any; i++) {
                const size_t pos = (w << 6) + d[i], pw = pos >> 6, b = pos & 63;
                any = 0;
                if (b) {
                    uint64_t lo = l0[pw];
                    for (int j = 0; j < kFitWords; j++) {
                        const uint64_t hi = l0[pw + (size_t)j + 1];
                        cand[j] &= ~((lo >> b) | (hi << (64 - b)));
                        any |= cand[j];
                        lo = hi;
                    }
                } else {
                    for (int j = 0; j < kFitWords; j++) {
                        cand[j] &= ~l0[pw + (size_t)j];
                        any |= cand[j];
                    }
                }
            }
            if (any)
                for (int j = 0; j < kFitWords; j++)
                    if (cand[j]) return ((w + (size_t)j) << 6) + (size_t)__builtin_ctzll(cand[j]);
            s = next_free((w + kFitWords) << 6);
        }
    }
    size_t next_free(size_t s)
    {
        ensure(s);
        size_t w = s >> 6;
        uint64_t freebits = ~l0[w] & (~0ULL << (s & 63));
        if (freebits) return (w << 6) + (size_t)__builtin_ctzll(freebits);
        w++;
        while (true) {   // skip full words, 64 or 4096 at a time through the summaries
            ensure(w << 6);
            if ((w & 63) == 0) {
                size_t w1 = w >> 6;
                if ((w1 & 63) == 0 && l2[w1 >> 6] == ~0ULL) { w += 64 * 64; continue; }
                if (l1[w1] == ~0ULL) { w += 64; continue; }
            }
            if (l0[w] == ~0ULL) { w++; continue; }
            return (w << 6) + (size_t)__builtin_ctzll(~l0[w]);
        }
    }
};

// phf.c:151-291 (FFDM) on the sorted key list.
int ffdm(Partition &P, int width)
{
    P.width = width;
    const size_t nk = P.keys.size();
    const int64_t n_r = ((int64_t)P.state_num * kCharSet) / width + 1;   // master_kernel.cu:221
    P.r.assign((size_t)n_r, -1);                                          // phf.c:67
    P.n_keys = (int32_t)nk;
    P.max_key = nk ? P.keys[nk - 1] : 0;                                  // phf.c:111-113
    const int MaxRow = P.max_key / width + 1;                             // phf.c:174
    P.max_row = MaxRow;
    // ReadKey (phf.c:90-117): per row, its columns in ascending order
    std::vector<int32_t> cnt((size_t)MaxRow, 0);
    std::vector<size_t> row_begin((size_t)MaxRow + 1, 0);
    for (size_t k = 0; k < nk; k++) cnt[(size_t)(P.keys[k] / width)]++;
    for (int rr = 0; rr < MaxRow; rr++) row_begin[(size_t)rr + 1] = row_begin[(size_t)rr] + (size_t)cnt[(size_t)rr];

    // SortRows (phf.c:126-139): for i ascending, a[i] is exchanged with every later element that
    // is strictly fuller than what a[i] currently holds.  Equivalent: carry a[i] to the nearest
    // later position q holding a strictly greater count, drop it there, pick up a[q], repeat;
    // what is carried at the end lands in a[i].
    std::vector<int32_t> a((size_t)MaxRow);
    for (int i = 0; i < MaxRow; i++) a[(size_t)i] = i;
    {
        MaxTree tree(cnt);
        for (int i = 0; i < MaxRow - 1; i++) {
            int32_t carry = a[(size_t)i];
            int32_t cc = cnt[(size_t)carry];
            tree.set(i, -1);
            if (tree.top() <= cc) continue;
            int p = i, q;
            while ((q = tree.first_greater(p + 1, cc)) != -1) {
                int32_t picked = a[(size_t)q];
                a[(size_t)q] = carry;
                tree.set(q, cc);
                carry = picked;
                cc = cnt[(size_t)carry];
                p = q;
            }
            a[(size_t)i] = carry;
        }
    }

    // first fit, fullest rows first (phf.c:184-229)
    SlotMap slots;
    std::vector<uint32_t> delta;
    std::vector<int32_t> HT, val;
    int32_t MaxOffset = 0;
    for (int ndx = 0; ndx < MaxRow; ndx++) {
        const int32_t row = a[(size_t)ndx];
        const int32_t c = cnt[(size_t)row];
        if (c <= 0) break;                                                // phf.c:184
        const size_t kb = row_begin[(size_t)row];
        const int32_t col0 = P.keys[kb] % width;
        delta.resize((size_t)c - 1);
        for (int i = 1; i < c; i++) delta[(size_t)i - 1] = (uint32_t)(P.keys[kb + (size_t)i] % width - col0);
        const size_t s = slots.first_fit(0, delta.data(), c - 1);         // phf.c:188-195
        const int64_t offset = (int64_t)s - col0;
        if (offset > INT32_MAX - width)
            return set_error(PFAC_ERR_LIMIT, "hash table offset exceeds 32 bits");
        P.r[(size_t)row] = (int32_t)offset;                               // phf.c:197
        if (offset > MaxOffset) MaxOffset = (int32_t)offset;
        const size_t hi = (size_t)(offset + P.keys[kb + (size_t)c - 1] % width);
        if (hi >= HT.size()) {
            size_t ns = std::max(hi + 1, HT.size() * 2);
            HT.resize(ns, -1);
            val.resize(ns, -1);
        }
        for (int i = 0; i < c; i++) {
            const size_t slot = (size_t)(offset + P.keys[kb + (size_t)i] % width);
            HT[slot] = row;                                               // phf.c:211
            val[slot] = P.next[kb + (size_t)i];                           // phf.c:216
            slots.mark(slot);
        }
    }
    int32_t HTSize = 0;                                                   // phf.c:232-236
    for (int64_t i = MaxOffset; i < (int64_t)MaxOffset + width && i < (int64_t)HT.size(); i++)
        if (HT[(size_t)i] >= 0 || val[(size_t)i] >= 0) HTSize = (int32_t)i + 1;
    HT.resize((size_t)HTSize, -1);
    val.resize((size_t)HTSize, -1);
    P.HT.swap(HT);
    P.val.swap(val);
    P.max_offset = MaxOffset;
    P.ht_size = HTSize;
    return PFAC_OK;
}

// Per-pattern case rules: the groups of one partition's sorted slice.  Lines equal after folding are adjacent (the
// sort is stable, so in file order); the automaton reports the last of each run.  A caseless line is live if no
// later caseless line of the run exists (they are all fold-equal), an exact line if no later exact line of the run
// is byte-equal to it.  orig[id - 1]: the line's bytes before the fold.
void case_groups(const Pattern *pats, int n, const std::vector<const unsigned char *> &orig, const uint8_t *rules,
                 Partition::CaseGroups &G)
{
    G = Partition::CaseGroups();
    G.first.push_back(0);
    for (int a = 0; a < n;) {
        int b = a + 1;
        while (b < n && comp_pat(pats[a], pats[b]) == 0) b++;
        G.owner.push_back(pats[b - 1].id);
        const int L = pats[a].len;
        for (int i = a; i < b; i++) {
            const int id = pats[i].id;
            const bool caseless = rules[id - 1] != 0;
            bool live = true;
            for (int j = i + 1; j < b && live; j++) {
                const int jd = pats[j].id;
                if (caseless) live = rules[jd - 1] == 0;
                else live = rules[jd - 1] != 0 || memcmp(orig[(size_t)id - 1], orig[(size_t)jd - 1], (size_t)L) != 0;
            }
            if (!live) continue;
            int32_t off = -1;
            if (!caseless) {
                const unsigned char *o = orig[(size_t)id - 1];
                if (std::any_of(o, o + L, [](unsigned char c) { return (c | 0x20) >= 'a' && (c | 0x20) <= 'z'; })) {
                    off = (int32_t)G.pool.size();
                    G.pool.insert(G.pool.end(), o, o + L);
                }
            }
            G.id.push_back(id);
            G.len.push_back(L);
            G.off.push_back(off);
        }
        G.first.push_back((int32_t)G.id.size());
        a = b;
    }
}

// rules: null, or (PFAC_PATTERNS_CASE_RULES) caseless[i] of every pattern the reader returns, not all equal
int build(const unsigned char *buf, size_t len, int n_parts, int width, unsigned flags, const uint8_t *rules,
          pfac_tables **out)
{
    if (!out || n_parts < 1) return set_error(PFAC_ERR_ARG, "bad arguments");
    if (width_bits(width) < 0)
        return set_error(PFAC_ERR_WIDTH, "width must be a power of two in [1,4096], got %d", width);
    std::vector<Pattern> pats;
    std::vector<unsigned char> arena;
    const bool caseless = (flags & PFAC_PATTERNS_CASELESS) != 0 || rules;
    int e;
    if (flags & PFAC_PATTERNS_ESCAPES) {
        e = read_patterns_ext(buf, len, arena, pats);
    } else if (caseless) {   // the plain reader's patterns point into the image: fold a copy of it
        arena.assign(buf, buf + len);
        e = read_patterns(arena.data(), len, pats);
    } else {
        e = read_patterns(buf, len, pats);
    }
    if (e) return e;
    // mixed rules: the exact lines are checked against their bytes before the fold
    std::vector<unsigned char> orig_arena;
    std::vector<const unsigned char *> orig;
    if (rules) {
        orig_arena = arena;
        orig.resize(pats.size());
        for (const Pattern &p : pats) orig[(size_t)p.id - 1] = orig_arena.data() + (p.p - arena.data());
    }
    // the fold comes after the reader (an escaped \x41 is 'A', then 'a') and before the sort, so that lines equal
    // after folding are duplicates like any other
    if (caseless)
        for (unsigned char &c : arena) c = ascii_fold(c);
    // qsort(&all_pattern[1], ...) (create_table_reorder.c:116).  glibc's qsort is a stable merge sort, so equal
    // patterns keep file order and the LAST duplicate wins its final state (:366).
    std::stable_sort(pats.begin(), pats.end(), [](const Pattern &a, const Pattern &b) { return comp_pat(a, b) < 0; });
    std::unique_ptr<pfac_tables> t(new pfac_tables);
    t->n_patterns = (int)pats.size();
    t->width = width;
    t->flags = rules ? PFAC_PATTERNS_CASE_RULES : (flags & PFAC_PATTERNS_CASELESS);
    if (rules) t->rules.assign(rules, rules + pats.size());
    t->parts.resize((size_t)n_parts);
    const int n = (int)pats.size();
    const int k = n / n_parts;            // create_table_reorder.c:220
    const int l = k + n % n_parts;        // create_table_reorder.c:222
    // The partitions are independent: trie + FFDM of each on its own thread (the reference runs FFDM per
    // partition under `omp parallel for`, main.cc:123-126).  Errors are thread-local: the first failing
    // partition's code and message are handed back to the caller's thread.
    std::vector<int> rcs((size_t)n_parts, PFAC_OK);
    std::vector<std::string> errs((size_t)n_parts);
    auto one = [&](int g) {
        const int cnt = (g == n_parts - 1) ? l : k;   // divide_patterns, :260-272
        Partition &P = t->parts[(size_t)g];
        if ((int64_t)cnt + 2 + (int64_t)len > (int64_t)(INT32_MAX / kCharSet)) {
            rcs[(size_t)g] = PFAC_ERR_LIMIT;
            errs[(size_t)g] = "automaton too large for 32-bit keys";
            return;
        }
        build_trie(pats.data() + (size_t)g * (size_t)k, cnt, P);
        if (rules) case_groups(pats.data() + (size_t)g * (size_t)k, cnt, orig, rules, P.groups);
        const int rc = ffdm(P, width);
        if (rc) {
            rcs[(size_t)g] = rc;
            errs[(size_t)g] = g_last_error;
        }
    };
    const int n_threads = std::max(1, std::min<int>(n_parts, (int)std::thread::hardware_concurrency()));
    if (n_threads == 1) {
        for (int g = 0; g < n_parts; g++) one(g);
    } else {
        std::atomic<int> next{0};
        auto worker = [&] {
            for (int g; (g = next.fetch_add(1)) < n_parts;) one(g);
        };
        std::vector<std::thread> th;
        for (int i = 1; i < n_threads; i++) th.emplace_back(worker);
        worker();
        for (auto &x : th) x.join();
    }
    for (int g = 0; g < n_parts; g++) {
        if (rcs[(size_t)g]) return set_error(rcs[(size_t)g], "%s", errs[(size_t)g].c_str());
        if (t->parts[(size_t)g].max_len > t->max_pat_len) t->max_pat_len = t->parts[(size_t)g].max_len;   // :238
    }
    *out = t.release();
    return PFAC_OK;
}

}  // namespace
}  // namespace pfac

using namespace pfac;

extern "C" {

const char *pfac_last_error(void) { return g_last_error.c_str(); }
int pfac_abi_version(void) { return PFAC_B200_ABI_VERSION; }

}  // extern "C"  (helpers)

namespace {
// FNV-1a 64 of the pattern file image and the front-end flags: identifies what a table set was built from
// (mixed case rules: and the rule bytes after the flags)
uint64_t source_hash_of(const void *bytes, size_t len, unsigned flags, const uint8_t *rules = nullptr, size_t n_rules = 0)
{
    uint64_t h = 1469598103934665603ull;
    const unsigned char *b = (const unsigned char *)bytes;
    for (size_t i = 0; i < len; i++) h = (h ^ b[i]) * 1099511628211ull;
    for (int i = 0; i < 4; i++) h = (h ^ ((flags >> (8 * i)) & 255u)) * 1099511628211ull;
    for (size_t i = 0; i < n_rules; i++) h = (h ^ rules[i]) * 1099511628211ull;
    return h ? h : 1;   // 0 = unknown (tables wrapped from arrays)
}

// Per-pattern case rules: the refusals of the _rules calls, then the rule class.  Returns 1 (all caseless: the
// PFAC_PATTERNS_CASELESS set), 0 (all exact: the plain set) or 2 (mixed) in *kind.
int check_rules(const unsigned char *buf, size_t len, unsigned flags, const uint8_t *rules, uint32_t n, int *kind)
{
    if (flags & PFAC_PATTERNS_CASELESS)
        return set_error(PFAC_ERR_ARG, "flags %#x: PFAC_PATTERNS_CASELESS (%#x) is not taken with per-pattern rules "
                         "(caseless[i] = 1 for all %u patterns gives that set)", flags, PFAC_PATTERNS_CASELESS, n);
    if (flags & ~PFAC_PATTERNS_ESCAPES)
        return set_error(PFAC_ERR_ARG, "flags %#x: per-pattern rules take PFAC_PATTERNS_ESCAPES (%#x) only", flags,
                         PFAC_PATTERNS_ESCAPES);
    if (!rules) return set_error(PFAC_ERR_ARG, "the rules of %u patterns are NULL", n);
    uint32_t ones = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (rules[i] > 1) return set_error(PFAC_ERR_ARG, "caseless[%u] = %u: a rule is 0 (exact) or 1 (caseless)", i, rules[i]);
        ones += rules[i];
    }
    std::vector<pfac::Pattern> pats;
    std::vector<unsigned char> arena;
    const int e = (flags & PFAC_PATTERNS_ESCAPES) ? pfac::read_patterns_ext(buf, len, arena, pats) : pfac::read_patterns(buf, len, pats);
    if (e) return e;
    if (pats.size() != n)
        return set_error(PFAC_ERR_ARG, "%u rules for %zu patterns: one rule per pattern the reader returns", n, pats.size());
    *kind = ones == n ? 1 : ones == 0 ? 0 : 2;
    return PFAC_OK;
}

// The source hash of a set built with these rules: that of the uniform set for uniform rules
uint64_t rules_hash(const unsigned char *buf, size_t len, unsigned flags, const uint8_t *rules, uint32_t n, int kind)
{
    if (kind != 2) return source_hash_of(buf, len, flags | (kind ? PFAC_PATTERNS_CASELESS : 0u));
    return source_hash_of(buf, len, flags | PFAC_PATTERNS_CASE_RULES, rules, n);
}

// the image of a pattern file; *e = PFAC_ERR_IO if it cannot be opened
std::vector<unsigned char> read_file(const char *path, int *e)
{
    std::vector<unsigned char> buf;
    FILE *f = path ? fopen(path, "rb") : nullptr;
    if (!f) {
        *e = set_error(PFAC_ERR_IO, "Open input file failed: %s", path ? path : "(null)");
        return buf;
    }
    unsigned char tmp[1 << 16];
    size_t got;
    while ((got = fread(tmp, 1, sizeof tmp, f)) > 0) buf.insert(buf.end(), tmp, tmp + got);
    fclose(f);
    *e = PFAC_OK;
    return buf;
}
// The verify pass indexes its tables with the owner ids and offsets these arrays hold
const char *validate_groups(const pfac::Partition::CaseGroups &G, int32_t n_patterns)
{
    if (G.first.size() != G.owner.size() + 1 || G.first[0] != 0 || G.first.back() != (int32_t)G.id.size())
        return "case group ranges";
    for (size_t g = 0; g < G.owner.size(); g++)
        if (G.first[g + 1] < G.first[g] || G.owner[g] < 1 || G.owner[g] > n_patterns) return "case group";
    for (size_t m = 0; m < G.id.size(); m++)
        if (G.id[m] < 1 || G.id[m] > n_patterns || G.len[m] < 1 || G.len[m] > pfac::kMaxPatternBytes || G.off[m] < -1 ||
            (G.off[m] >= 0 && (size_t)G.off[m] + (size_t)G.len[m] > G.pool.size()))
            return "case group member";
    return nullptr;
}
// The kernels index r[] / {HT,val} / s0 / idmap with what these arrays hold, unchecked (as the
// reference does): a table set that did not come out of the builder is checked once, here.
const char *validate_partition(const pfac::Partition &P)
{
    using pfac::kCharSet;
    if (P.state_num < 0 || P.n_final < 0 || P.max_len < 0 || P.ht_size < 0) return "negative size";
    if (pfac::width_bits(P.width) < 0) return "width";
    if ((int64_t)P.r.size() != ((int64_t)P.state_num * kCharSet) / P.width + 1) return "r[] size is not state_num*256/width + 1";
    if ((int64_t)P.HT.size() != P.ht_size || (int64_t)P.val.size() != P.ht_size) return "HT/val size";
    if ((int64_t)P.idmap.size() != P.n_final || P.s0.size() != (size_t)kCharSet) return "idmap/s0 size";
    if (P.n_final > P.state_num + 1) return "more final states than states";
    for (int32_t v : P.s0)
        if (v < -1 || v >= P.state_num) return "s0Table entry out of range";
    for (int32_t v : P.val)
        if (v < -1 || v >= P.state_num) return "val entry out of range";
    for (int32_t v : P.HT)
        if (v < -1 || v >= (int32_t)P.r.size()) return "HT entry out of range";
    return nullptr;
}
}  // namespace

extern "C" {

int pfac_tables_build_mem(const void *pattern_bytes, size_t len, int n_parts, int width, pfac_tables **out)
{
    return pfac_tables_build_mem_ext(pattern_bytes, len, n_parts, width, 0u, out);
}

int pfac_tables_build_mem_ext(const void *pattern_bytes, size_t len, int n_parts, int width, unsigned flags,
                              pfac_tables **out)
{
    if (!pattern_bytes && len) return set_error(PFAC_ERR_ARG, "null pattern buffer");
    try {
        const int rc = build((const unsigned char *)pattern_bytes, len, n_parts, width, flags, nullptr, out);
        if (rc == PFAC_OK && out && *out) (*out)->source_hash = source_hash_of(pattern_bytes, len, flags);
        return rc;
    } catch (const std::bad_alloc &) {
        return set_error(PFAC_ERR_NOMEM, "out of memory building tables");
    }
}

uint64_t pfac_tables_source_hash(const pfac_tables *t) { return t ? t->source_hash : 0; }

int pfac_pattern_file_hash(const char *pattern_file, unsigned flags, uint64_t *hash)
{
    if (!hash) return set_error(PFAC_ERR_ARG, "null hash");
    int e;
    std::vector<unsigned char> buf = read_file(pattern_file, &e);
    if (e) return e;
    *hash = source_hash_of(buf.data(), buf.size(), flags);
    return PFAC_OK;
}

int pfac_tables_build_file(const char *pattern_file, int n_parts, int width, pfac_tables **out)
{
    return pfac_tables_build_file_ext(pattern_file, n_parts, width, 0u, out);
}

int pfac_tables_build_file_ext(const char *pattern_file, int n_parts, int width, unsigned flags, pfac_tables **out)
{
    int e;
    std::vector<unsigned char> buf = read_file(pattern_file, &e);
    if (e) return e;
    return pfac_tables_build_mem_ext(buf.data(), buf.size(), n_parts, width, flags, out);
}

int pfac_tables_build_mem_rules(const void *pattern_bytes, size_t len, int n_parts, int width, unsigned flags,
                                const uint8_t *caseless, uint32_t n_patterns, pfac_tables **out)
{
    if (!pattern_bytes && len) return set_error(PFAC_ERR_ARG, "null pattern buffer");
    const unsigned char *buf = (const unsigned char *)pattern_bytes;
    try {
        int kind = 0;
        int rc = check_rules(buf, len, flags, caseless, n_patterns, &kind);
        if (rc) return rc;
        rc = build(buf, len, n_parts, width, flags | (kind == 1 ? PFAC_PATTERNS_CASELESS : 0u), kind == 2 ? caseless : nullptr, out);
        if (rc == PFAC_OK && out && *out) (*out)->source_hash = rules_hash(buf, len, flags, caseless, n_patterns, kind);
        return rc;
    } catch (const std::bad_alloc &) {
        return set_error(PFAC_ERR_NOMEM, "out of memory building tables");
    }
}

int pfac_tables_build_file_rules(const char *pattern_file, int n_parts, int width, unsigned flags, const uint8_t *caseless,
                                 uint32_t n_patterns, pfac_tables **out)
{
    int e;
    std::vector<unsigned char> buf = read_file(pattern_file, &e);
    if (e) return e;
    return pfac_tables_build_mem_rules(buf.data(), buf.size(), n_parts, width, flags, caseless, n_patterns, out);
}

int pfac_pattern_file_hash_rules(const char *pattern_file, unsigned flags, const uint8_t *caseless, uint32_t n_patterns,
                                 uint64_t *hash)
{
    if (!hash) return set_error(PFAC_ERR_ARG, "null hash");
    try {
        int e, kind = 0;
        std::vector<unsigned char> buf = read_file(pattern_file, &e);
        if (e || (e = check_rules(buf.data(), buf.size(), flags, caseless, n_patterns, &kind))) return e;
        *hash = rules_hash(buf.data(), buf.size(), flags, caseless, n_patterns, kind);
        return PFAC_OK;
    } catch (const std::bad_alloc &) {
        return set_error(PFAC_ERR_NOMEM, "out of memory");
    }
}

int pfac_tables_case_rules(const pfac_tables *t, uint8_t *caseless, uint32_t n)
{
    if (!t || !caseless || n != (uint32_t)t->n_patterns)
        return set_error(PFAC_ERR_ARG, "pfac_tables_case_rules takes one rule per pattern: %u for %d patterns", n,
                         t ? t->n_patterns : 0);
    if (t->flags & PFAC_PATTERNS_CASE_RULES) memcpy(caseless, t->rules.data(), n);
    else memset(caseless, (t->flags & PFAC_PATTERNS_CASELESS) ? 1 : 0, n);
    return PFAC_OK;
}

int pfac_tables_from_arrays(const int32_t *s0, const int32_t *r, int32_t n_r, const int32_t *HT,
                            const int32_t *val, int32_t ht_size, int32_t width, int32_t state_num,
                            int32_t n_final, const int32_t *idmap, int32_t max_pat_len, pfac_tables **out)
{
    if (!out || !s0 || !r || n_r < 1 || ht_size < 0 || (ht_size && (!HT || !val)) || n_final < 0 ||
        (n_final && !idmap) || max_pat_len < 0)
        return set_error(PFAC_ERR_ARG, "bad arguments");
    if (width_bits(width) < 0) return set_error(PFAC_ERR_WIDTH, "width must be a power of two in [1,4096]");
    try {
        std::unique_ptr<pfac_tables> t(new pfac_tables);
        t->n_patterns = n_final;
        t->max_pat_len = max_pat_len;
        t->width = width;
        t->parts.resize(1);
        Partition &P = t->parts[0];
        P.state_num = state_num;
        P.n_final = n_final;
        P.max_len = max_pat_len;
        P.min_len = 1;
        P.width = width;
        P.ht_size = ht_size;
        P.s0.assign(s0, s0 + kCharSet);
        P.r.assign(r, r + n_r);
        P.HT.assign(HT, HT + ht_size);
        P.val.assign(val, val + ht_size);
        P.idmap.assign(idmap, idmap + n_final);
        for (int32_t i = 0; i < ht_size; i++)
            if (P.HT[(size_t)i] >= 0) P.n_keys++;
        if (const char *why = validate_partition(P)) return set_error(PFAC_ERR_ARG, "inconsistent tables: %s", why);
        *out = t.release();
        return PFAC_OK;
    } catch (const std::bad_alloc &) {
        return set_error(PFAC_ERR_NOMEM, "out of memory");
    }
}

// ---- on-disk cache of the canonical arrays (the reference serialises nothing: it rebuilds the trie
// and the PHF on every run, main.cc:100-126).  Little-endian int32 fields:
//   "PFACTBL2", n_parts, n_patterns, max_pat_len, width, source hash (u64: pattern file image + flags),
//   ["PFACTBL3" only: u32 flags (PFAC_PATTERNS_CASELESS or PFAC_PATTERNS_CASE_RULES): written for those sets alone,
//    so that a case-sensitive set writes the same file as before and a library that does not know the flag refuses
//    the cache by its magic (and a library that knows PFAC_PATTERNS_CASELESS only, by the flags value)],
//   [PFAC_PATTERNS_CASE_RULES only: u8 rules[n_patterns]],
//   per partition: state_num, n_final, max_len, min_len, width, n_keys, max_key, max_row, max_offset,
//                  ht_size, n_r, then s0[256], r[n_r], HT[ht_size], val[ht_size], idmap[n_final],
//                  [PFAC_PATTERNS_CASE_RULES only: n_groups, n_members, pool bytes, owner[n_groups],
//                   first[n_groups + 1], id[n_members], len[n_members], off[n_members], u8 pool[]],
//   FNV-1a 64 of everything before it.
namespace {
struct Fnv {
    uint64_t h = 1469598103934665603ull;
    void add(const void *p, size_t n)
    {
        const unsigned char *b = (const unsigned char *)p;
        for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 1099511628211ull;
    }
};
bool put(FILE *f, Fnv &h, const void *p, size_t n)
{
    h.add(p, n);
    return n == 0 || fwrite(p, 1, n, f) == n;
}
bool get(FILE *f, Fnv &h, void *p, size_t n)
{
    if (n && fread(p, 1, n, f) != n) return false;
    h.add(p, n);
    return true;
}
}  // namespace

int pfac_tables_save(const pfac_tables *t, const char *path)
{
    if (!t || !path) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_tables_save");
    FILE *f = fopen(path, "wb");
    if (!f) return set_error(PFAC_ERR_IO, "cannot create %s", path);
    Fnv h;
    const uint32_t flags = t->flags;
    bool ok = put(f, h, flags ? "PFACTBL3" : "PFACTBL2", 8);
    const int32_t head[4] = {(int32_t)t->parts.size(), t->n_patterns, t->max_pat_len, t->width};
    const bool mixed = (flags & PFAC_PATTERNS_CASE_RULES) != 0;
    ok = ok && put(f, h, head, sizeof head) && put(f, h, &t->source_hash, 8) && (!flags || put(f, h, &flags, 4)) &&
         (!mixed || put(f, h, t->rules.data(), t->rules.size()));
    for (const Partition &P : t->parts) {
        const int32_t ph[11] = {P.state_num, P.n_final, P.max_len, P.min_len, P.width, P.n_keys, P.max_key, P.max_row,
                                P.max_offset, P.ht_size, (int32_t)P.r.size()};
        std::vector<int32_t> s0 = P.s0;
        s0.resize(kCharSet, -1);
        ok = ok && put(f, h, ph, sizeof ph) && put(f, h, s0.data(), kCharSet * 4) && put(f, h, P.r.data(), P.r.size() * 4) &&
             put(f, h, P.HT.data(), (size_t)P.ht_size * 4) && put(f, h, P.val.data(), (size_t)P.ht_size * 4) &&
             put(f, h, P.idmap.data(), (size_t)P.n_final * 4);
        if (mixed) {
            const Partition::CaseGroups &G = P.groups;
            const int32_t gh[3] = {(int32_t)G.owner.size(), (int32_t)G.id.size(), (int32_t)G.pool.size()};
            ok = ok && put(f, h, gh, sizeof gh) && put(f, h, G.owner.data(), G.owner.size() * 4) &&
                 put(f, h, G.first.data(), G.first.size() * 4) && put(f, h, G.id.data(), G.id.size() * 4) &&
                 put(f, h, G.len.data(), G.len.size() * 4) && put(f, h, G.off.data(), G.off.size() * 4) &&
                 put(f, h, G.pool.data(), G.pool.size());
        }
    }
    const uint64_t sum = h.h;
    ok = ok && fwrite(&sum, 1, 8, f) == 8;
    ok = (fclose(f) == 0) && ok;
    return ok ? PFAC_OK : set_error(PFAC_ERR_IO, "short write to %s", path);
}

int pfac_tables_load(const char *path, pfac_tables **out)
{
    if (!path || !out) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_tables_load");
    FILE *f = fopen(path, "rb");
    if (!f) return set_error(PFAC_ERR_IO, "Open input file failed: %s", path);
    auto bad = [&](const char *why) {
        fclose(f);
        return set_error(PFAC_ERR_IO, "%s is not a table cache this library wrote (%s)", path, why);
    };
    try {
        Fnv h;
        char magic[8];
        int32_t head[4];
        if (!get(f, h, magic, 8) || (memcmp(magic, "PFACTBL2", 8) != 0 && memcmp(magic, "PFACTBL3", 8) != 0)) return bad("magic");
        const bool v3 = magic[7] == '3';
        uint64_t src_hash = 0;
        uint32_t flags = 0;
        if (!get(f, h, head, sizeof head) || !get(f, h, &src_hash, 8) || head[0] < 1 || head[0] > (1 << 20) || head[1] < 0 ||
            head[2] < 0 || width_bits(head[3]) < 0)
            return bad("header");
        if (v3 && (!get(f, h, &flags, 4) || (flags != PFAC_PATTERNS_CASELESS && flags != PFAC_PATTERNS_CASE_RULES)))
            return bad("flags");
        const bool mixed = flags == PFAC_PATTERNS_CASE_RULES;
        std::vector<uint8_t> rules(mixed ? (size_t)head[1] : 0);
        if (mixed && !get(f, h, rules.data(), rules.size())) return bad("truncated");
        std::unique_ptr<pfac_tables> t(new pfac_tables);
        t->source_hash = src_hash;
        t->flags = flags;
        t->rules.swap(rules);
        t->n_patterns = head[1];
        t->max_pat_len = head[2];
        t->width = head[3];
        t->parts.resize((size_t)head[0]);
        for (Partition &P : t->parts) {
            int32_t ph[11];
            if (!get(f, h, ph, sizeof ph)) return bad("truncated");
            if (ph[0] < 0 || ph[1] < 0 || ph[1] > ph[0] + 1 || ph[9] < 0 || ph[10] < 1 || ph[4] != head[3] ||
                (int64_t)ph[10] != ((int64_t)ph[0] * kCharSet) / ph[4] + 1)
                return bad("partition header");
            P.state_num = ph[0];
            P.n_final = ph[1];
            P.max_len = ph[2];
            P.min_len = ph[3];
            P.width = ph[4];
            P.n_keys = ph[5];
            P.max_key = ph[6];
            P.max_row = ph[7];
            P.max_offset = ph[8];
            P.ht_size = ph[9];
            P.s0.resize(kCharSet);
            P.r.resize((size_t)ph[10]);
            P.HT.resize((size_t)ph[9]);
            P.val.resize((size_t)ph[9]);
            P.idmap.resize((size_t)ph[1]);
            if (!get(f, h, P.s0.data(), kCharSet * 4) || !get(f, h, P.r.data(), P.r.size() * 4) ||
                !get(f, h, P.HT.data(), P.HT.size() * 4) || !get(f, h, P.val.data(), P.val.size() * 4) ||
                !get(f, h, P.idmap.data(), P.idmap.size() * 4))
                return bad("truncated");
            if (mixed) {   // (the sizes are bounded before anything is allocated for them)
                Partition::CaseGroups &G = P.groups;
                int32_t gh[3];
                if (!get(f, h, gh, sizeof gh)) return bad("truncated");
                if (gh[0] < 0 || gh[1] < 0 || gh[2] < 0 || gh[0] > head[1] || gh[1] > head[1] ||
                    (int64_t)gh[2] > (int64_t)gh[1] * kMaxPatternBytes)
                    return bad("case groups header");
                G.owner.resize((size_t)gh[0]);
                G.first.resize((size_t)gh[0] + 1);
                G.id.resize((size_t)gh[1]);
                G.len.resize((size_t)gh[1]);
                G.off.resize((size_t)gh[1]);
                G.pool.resize((size_t)gh[2]);
                if (!get(f, h, G.owner.data(), G.owner.size() * 4) || !get(f, h, G.first.data(), G.first.size() * 4) ||
                    !get(f, h, G.id.data(), G.id.size() * 4) || !get(f, h, G.len.data(), G.len.size() * 4) ||
                    !get(f, h, G.off.data(), G.off.size() * 4) || !get(f, h, G.pool.data(), G.pool.size()))
                    return bad("truncated");
            }
        }
        uint64_t sum = 0;
        if (fread(&sum, 1, 8, f) != 8 || sum != h.h) return bad("checksum");
        for (const Partition &P : t->parts)
            if (const char *why = validate_partition(P)) return bad(why);
        for (uint8_t r : t->rules)
            if (r > 1) return bad("case rule");
        if (mixed)
            for (const Partition &P : t->parts)
                if (const char *why = validate_groups(P.groups, t->n_patterns)) return bad(why);
        fclose(f);
        *out = t.release();
        return PFAC_OK;
    } catch (const std::bad_alloc &) {
        fclose(f);
        return set_error(PFAC_ERR_NOMEM, "out of memory loading %s", path);
    }
}

void pfac_tables_destroy(pfac_tables *t) { delete t; }
int pfac_tables_n_parts(const pfac_tables *t) { return t ? (int)t->parts.size() : 0; }
int pfac_tables_n_patterns(const pfac_tables *t) { return t ? t->n_patterns : 0; }
int pfac_tables_max_pat_len(const pfac_tables *t) { return t ? t->max_pat_len : 0; }
int pfac_tables_width(const pfac_tables *t) { return t ? t->width : 0; }
unsigned pfac_tables_flags(const pfac_tables *t) { return t ? t->flags : 0u; }

static const Partition *part_of(const pfac_tables *t, int part)
{
    if (!t || part < 0 || part >= (int)t->parts.size()) return nullptr;
    return &t->parts[(size_t)part];
}

int pfac_tables_part_info(const pfac_tables *t, int part, int32_t info[9])
{
    const Partition *P = part_of(t, part);
    if (!P || !info) return set_error(PFAC_ERR_ARG, "bad partition index");
    info[0] = P->state_num; info[1] = P->n_final; info[2] = P->max_len; info[3] = P->ht_size;
    info[4] = (int32_t)P->r.size(); info[5] = P->n_keys; info[6] = P->max_key; info[7] = P->max_offset;
    info[8] = P->min_len;
    return PFAC_OK;
}

const int32_t *pfac_tables_s0(const pfac_tables *t, int part) { const Partition *P = part_of(t, part); return P ? P->s0.data() : nullptr; }
const int32_t *pfac_tables_r(const pfac_tables *t, int part) { const Partition *P = part_of(t, part); return P ? P->r.data() : nullptr; }
const int32_t *pfac_tables_HT(const pfac_tables *t, int part) { const Partition *P = part_of(t, part); return P ? P->HT.data() : nullptr; }
const int32_t *pfac_tables_val(const pfac_tables *t, int part) { const Partition *P = part_of(t, part); return P ? P->val.data() : nullptr; }
const int32_t *pfac_tables_idmap(const pfac_tables *t, int part) { const Partition *P = part_of(t, part); return P ? P->idmap.data() : nullptr; }

int pfac_tables_pattern_lengths(const pfac_tables *t, int part, int32_t *lengths, int32_t n, int32_t *n_ids)
{
    const Partition *P = part_of(t, part);
    if (!P || !n_ids || n < 0) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_tables_pattern_lengths");
    try {
        std::vector<int32_t> len;
        const int e = pattern_lengths(*P, len);
        if (e) return e;
        *n_ids = (int32_t)len.size();
        if (!lengths) return PFAC_OK;
        if (n < *n_ids)
            return set_error(PFAC_ERR_OUTPUT_FULL, "%d pattern ids need an array of %d entries, not %d", *n_ids, *n_ids, n);
        if (!len.empty()) memcpy(lengths, len.data(), len.size() * sizeof(int32_t));
        std::fill(lengths + len.size(), lengths + n, 0);
        return PFAC_OK;
    } catch (const std::bad_alloc &) {
        return set_error(PFAC_ERR_NOMEM, "out of memory");
    }
}

int pfac_tables_derive_check(const pfac_tables *t, int part, uint32_t t2_bytes, uint32_t t3_bytes, uint32_t tm2_bytes,
                             uint64_t stats[10])
{
    const Partition *P = part_of(t, part);
    if (!P) return set_error(PFAC_ERR_ARG, "bad partition index");
    try {
        Derived d;
        derive_tables(*P, t2_bytes, t3_bytes, tm2_bytes, d);
        if (stats) {
            const uint64_t v[10] = {d.image.size(), d.t1_set, d.t2_set, d.n_prefix4, d.has_short, d.has_t3,
                                    d.tm_set, d.tm2_set, d.t3_set, d.tm2_bits};
            memcpy(stats, v, sizeof v);
        }
        const int bad = derive_selfcheck(*P, d);
        if (bad) return set_error(PFAC_ERR_INTERNAL, "derived tables violate invariant %d", bad);
        {   // the pattern directory of the candidate walks must answer like the walk
            PatDir pd;
            derive_patdir(*P, pd);
            const int pbad = patdir_selfcheck(*P, pd);
            if (pbad) return set_error(PFAC_ERR_INTERNAL, "pattern directory violates invariant %d", pbad);
        }
        // the dense-match kernel's walk cache must be the PHF's transition function on the levels it covers
        for (uint32_t budget : {131072u, 16384u, 2048u}) {
            WalkCache w;
            derive_walk_cache(*P, budget, w);
            if (w.image.size() < 1024) return set_error(PFAC_ERR_INTERNAL, "walk cache has no root row");
            for (int b0 = 0; b0 < 256; b0++) {
                uint8_t t[3] = {(uint8_t)b0, 0, 0};
                const int32_t s1 = P->s0.empty() ? -1 : P->s0[(size_t)b0];
                if (walk_cache_lookup(w, t, 1) != s1) return set_error(PFAC_ERR_INTERNAL, "walk cache: root row differs");
                if (w.depth < 2) continue;
                for (int b1 = 0; b1 < 256; b1++) {
                    t[1] = (uint8_t)b1;
                    const int32_t s2 = s1 < 0 ? -1 : P->lookup(s1, b1);
                    if (walk_cache_lookup(w, t, 2) != s2) return set_error(PFAC_ERR_INTERNAL, "walk cache: depth 2 differs");
                    if (w.depth < 3 || s2 < 0) continue;
                    for (int b2 = 0; b2 < 256; b2++) {
                        t[2] = (uint8_t)b2;
                        if (walk_cache_lookup(w, t, 3) != P->lookup(s2, b2)) return set_error(PFAC_ERR_INTERNAL, "walk cache: depth 3 differs");
                    }
                }
            }
        }
        return PFAC_OK;
    } catch (const std::bad_alloc &) {
        return set_error(PFAC_ERR_NOMEM, "out of memory");
    }
}

int pfac_tables_filter_profile(const pfac_tables *t, int part, uint32_t t2_bytes, uint32_t t3_bytes, uint32_t tm2_bytes,
                               const void *text, uint64_t n, uint64_t counts[12])
{
    const Partition *P = part_of(t, part);
    if (!P || (!text && n) || !counts) return set_error(PFAC_ERR_ARG, "bad arguments");
    try {
        Derived d;
        derive_tables(*P, t2_bytes, t3_bytes, tm2_bytes, d);
        std::vector<uint8_t> folded;   // a caseless or mixed set counts the text its detector sees
        if (t->flags & (PFAC_PATTERNS_CASELESS | PFAC_PATTERNS_CASE_RULES)) {
            folded.assign((const uint8_t *)text, (const uint8_t *)text + n);
            for (uint8_t &c : folded) c = ascii_fold(c);
            text = folded.data();
        }
        derive_profile(*P, d, (const uint8_t *)text, (size_t)n, counts);
        return PFAC_OK;
    } catch (const std::bad_alloc &) {
        return set_error(PFAC_ERR_NOMEM, "out of memory");
    }
}

int32_t pfac_tables_lookup(const pfac_tables *t, int part, int32_t state, int32_t byte)
{
    const Partition *P = part_of(t, part);
    if (!P || state < 0 || byte < 0 || byte > 255) return -1;
    return P->lookup(state, byte);
}

}  // extern "C"
