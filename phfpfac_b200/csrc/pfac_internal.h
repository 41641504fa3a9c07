// Internal declarations shared by the host-side translation units of libpfac_b200.
#pragma once
#include <cstdarg>
#include <cstdint>
#include <string>
#include <vector>

#include "pfac_b200.h"

namespace pfac {

constexpr int kCharSet = 256;            // ctdef.h:12
constexpr int kRefTile = 4096;           // master_kernel.cu:9-10 (PAGE_SIZE_C)
constexpr int kRefHalo = 512;            // master_kernel.cu:11 (EXTRA_SIZE_PER_TB ints)
constexpr int kMaxPatternBytes = 1022;   // create_table_reorder.c:55,74: buffer of 1024 incl. '\n'

// One partition's canonical tables: the thread_data fields of main.cc:19-32.
struct Partition {
    int32_t state_num = 0;    // create_table_reorder.c:376
    int32_t n_final = 0;      // create_table_reorder.c:239
    int32_t max_len = 0;      // create_table_reorder.c:319-321
    int32_t min_len = 0;
    int32_t width = 256;
    int32_t n_keys = 0, max_key = 0, max_row = 0, max_offset = 0, ht_size = 0;  // phf.c:151-236
    std::vector<int32_t> s0;     // 256 entries = PFAC[n_final+1][.] (main.cc:200)
    std::vector<int32_t> r;      // state_num*256/width + 1 entries (master_kernel.cu:221)
    std::vector<int32_t> HT;     // ht_size entries: row id per slot, -1 empty (phf.c:211)
    std::vector<int32_t> val;    // ht_size entries: next state (phf.c:216)
    std::vector<int32_t> idmap;  // n_final entries (create_table_reorder.c:318)
    // transitions sorted by key = state*256 + byte (the non-negative cells of PFAC[][])
    std::vector<int32_t> keys;
    std::vector<int32_t> next;
    // Sets with per-pattern case rules (PFAC_PATTERNS_CASE_RULES) only: the verify tables.  The automaton is that
    // of the folded patterns, so its final state of a folded string reports one owner id (the last fold-equal line
    // of the partition); group g lists the live lines that fold to that string, ascending by id.  A member with
    // off >= 0 is an exact line with at least one letter: it matches only where the original text equals
    // pool[off, off + len).  Every other member matches wherever its owner does.
    struct CaseGroups {
        std::vector<int32_t> owner;    // [n_groups]
        std::vector<int32_t> first;    // [n_groups + 1]: members first[g] .. first[g + 1] - 1
        std::vector<int32_t> id, len, off;   // [n_members]
        std::vector<uint8_t> pool;
    } groups;

    // master_kernel.cu:52-64
    int32_t lookup(int32_t state, int32_t byte) const;
};

int set_error(int code, const char *fmt, ...);
int width_bits(int width);   // log2 of a power-of-two width, -1 otherwise (master_kernel.cu:397-398)

}  // namespace pfac

struct pfac_tables {
    int n_patterns = 0;
    int max_pat_len = 0;
    int width = 256;
    std::vector<pfac::Partition> parts;
    uint64_t source_hash = 0;   // FNV-1a of the pattern file image + flags the set was built from (0: unknown)
    unsigned flags = 0;         // PFAC_PATTERNS_CASELESS or PFAC_PATTERNS_CASE_RULES (include/pfac_b200.h)
    std::vector<uint8_t> rules; // PFAC_PATTERNS_CASE_RULES: caseless[i] of pattern id i + 1 (n_patterns entries)
};
