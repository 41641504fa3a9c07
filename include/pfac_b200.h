/*
 * pfac_b200.h -- C ABI of the B200-native PFAC (Parallel Failureless Aho-Corasick) matcher.
 *
 * Drop-in boundary for the scan path of mickeyjoe666/PHFPFAC.  Every entry point names the
 * reference interface it replaces (paths relative to the reference's regex_GPU_PHF/).
 * Plain C types only: no CUDA or torch types.  A `void *stream` is a cudaStream_t passed
 * opaquely (NULL = the library's own stream).  All functions return 0 on success or a
 * negative pfac_status; the message is available from pfac_last_error() (thread-local).
 * The library never calls exit() (the reference does, master_kernel.cu:240-244).
 *
 * Layers
 *   pfac_tables_*  : pattern file -> PFAC trie -> PHF (r/HT/val) arrays, bit-compatible with
 *                    create_PFAC_table_reorder() + FFDM()  (create_PFAC_table_reorder.c:6, phf.c:151)
 *   pfac_ctx_*     : one device: table upload + scan of device-resident or host buffers, and of
 *                    batches of independent device-resident documents (pfac_scan_batch_device)
 *                    (GPU_Malloc_Memory / GPU_TraceTable / GPU_Free_memory, main.cc:35-37)
 *   pfac_flows_*   : streaming scan of many flows on one context: chunk by chunk, matches that
 *                    straddle chunk boundaries included, the carried bytes kept on the device
 *                    (pfac_scan_flows_device_sync)
 *   pfac_job_*     : all GPUs of the box: contiguous input chunk + halo per GPU, stream pipeline
 *                    per GPU (the scan loop of main.cc:171-272)
 *   pfac_write_*   : GPU_match_result.txt writer (main.cc:335-350)
 */
#ifndef PFAC_B200_H
#define PFAC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFAC_B200_ABI_VERSION 1

typedef enum pfac_status {
    PFAC_OK = 0,
    PFAC_ERR_IO = -1,               /* cannot open/read a file (main.cc:131-135 perror+exit) */
    PFAC_ERR_PATTERN_TOO_LONG = -2, /* >1022 bytes or no trailing '\n' (create_table_reorder.c:74-77) */
    PFAC_ERR_EMPTY_PATTERN = -3,    /* empty line: undefined in the reference (create_table_reorder.c:362) */
    PFAC_ERR_WIDTH = -4,            /* width not a power of two in [1,4096] (phf.c:161, master_kernel.cu:398) */
    PFAC_ERR_ARG = -5,
    PFAC_ERR_NOMEM = -6,
    PFAC_ERR_CUDA = -7,             /* any CUDA runtime error; never a CPU fallback */
    PFAC_ERR_OUTPUT_FULL = -8,      /* more matches than the caller's capacity; *count = required */
    PFAC_ERR_NO_DEVICE = -9,
    PFAC_ERR_LIMIT = -10,           /* size beyond what the 32-bit record format carries per call */
    PFAC_ERR_INTERNAL = -11         /* device-side watchdog tripped (never expected) */
} pfac_status;

/* One match: `pos` is the start position of the match relative to the first start position of
 * the call, `id` is the 1-based line number of the pattern (create_table_reorder.c:100).
 * Records are ordered by (pos, pattern length) -- the order main.cc:341-349 prints. */
typedef struct pfac_match {
    uint32_t pos;
    uint32_t id;
} pfac_match;

typedef struct pfac_tables pfac_tables; /* host-side table set: n_parts x {s0,r,HT,val,idmap,...} */
typedef struct pfac_ctx pfac_ctx;       /* one device */
typedef struct pfac_job pfac_job;       /* multi-GPU job */
typedef struct pfac_flows pfac_flows;   /* streaming state of many flows on one context */

const char *pfac_last_error(void);
int pfac_abi_version(void);

/* ------------------------------------------------------------------------------ tables
 * Replaces create_PFAC_table_reorder(argv[1], ...) (main.cc:108) and the FFDM loop
 * (main.cc:122-126).  `n_parts` contiguous slices of the sorted pattern list
 * (create_table_reorder.c:253-274; the reference always uses 4*streamnum), each with its
 * own trie and PHF.  The scanner uses n_parts = 1 (results are independent of the
 * partition count).  `width` is the PHF key-table width, argv[3]. */
int pfac_tables_build_file(const char *pattern_file, int n_parts, int width, pfac_tables **out);
int pfac_tables_build_mem(const void *pattern_bytes, size_t len, int n_parts, int width, pfac_tables **out);
/* The same with front-end flags.  PFAC_PATTERNS_ESCAPES reads the pattern file through the
 * reference's escape-processing reader, read_pattern_ext / fgetc_ext (create_table_reorder.c:131-185,
 * ctdef.h:37-99: \ooo, \xhh, \a \b \t \n \v \f \r \' \" \\) -- code the reference ships but its
 * main() never calls, hence behind a flag. */
#define PFAC_PATTERNS_ESCAPES 1u
/* PFAC_PATTERNS_CASELESS (this project's flag; the reference has no case-insensitive mode) builds a set that
 * matches ASCII letters in either case.  The fold maps bytes 0x41-0x5A ('A'-'Z') to 0x61-0x7A and leaves every
 * other byte as it is (no locale, no Unicode: 0xC1-0xDA do not fold).  The patterns are folded after the reader
 * (so with PFAC_PATTERNS_ESCAPES, \x41 is 'a') and before the sort, so the tables are bit-identical to those of
 * the folded pattern file, and every scan of such a set folds its text on the device first:
 *   scan(set of P with PFAC_PATTERNS_CASELESS, T) == scan(set of fold(P), fold(T)), record for record.
 * Lines equal after folding are duplicates: the last such line owns the match ("GET" then "get": only the
 * second line's id is reported; pfac_tables_pattern_lengths reports 0 for the first).  This flag gives the whole
 * set one case rule; the _rules calls below give one rule per pattern. */
#define PFAC_PATTERNS_CASELESS 2u
int pfac_tables_build_file_ext(const char *pattern_file, int n_parts, int width, unsigned flags,
                               pfac_tables **out);
int pfac_tables_build_mem_ext(const void *pattern_bytes, size_t len, int n_parts, int width,
                              unsigned flags, pfac_tables **out);
/* Per-pattern case rules (DESIGN.md section 3.11).  caseless[i] is the rule of pattern id i + 1 (one per pattern
 * the reader returns, so with PFAC_PATTERNS_ESCAPES one per decoded pattern): 1 matches ASCII letters in either
 * case, fold(T[pos, pos+L)) == fold(p); 0 matches byte for byte, T[pos, pos+L) == p.  Two lines are duplicates
 * (the last one owns the match) iff they have the same rule and are equal under it; an exact and a caseless line
 * never are, so several ids can report at one (pos, length): records are ordered by (pos, length, id).  flags may
 * be PFAC_PATTERNS_ESCAPES or 0.  PFAC_ERR_ARG for PFAC_PATTERNS_CASELESS in flags, a NULL rules pointer, a rule
 * other than 0 or 1, and n_patterns != the number of patterns the reader returns.
 * All 1 builds exactly the PFAC_PATTERNS_CASELESS set of the file, all 0 exactly the plain set (same tables,
 * flags, source hash and cache file).  Mixed rules build the automaton of the folded patterns -- bit-identical to
 * the caseless build -- plus verify tables: every scan folds its text out of place, the unchanged detector reports
 * owner ids, and a verify pass expands each record to the members of its owner that pass (exact members are
 * compared with the original bytes).  pfac_tables_flags reports PFAC_PATTERNS_CASE_RULES for such a set; the
 * flag is never passed in. */
#define PFAC_PATTERNS_CASE_RULES 4u
int pfac_tables_build_file_rules(const char *pattern_file, int n_parts, int width, unsigned flags,
                                 const uint8_t *caseless, uint32_t n_patterns, pfac_tables **out);
int pfac_tables_build_mem_rules(const void *pattern_bytes, size_t len, int n_parts, int width, unsigned flags,
                                const uint8_t *caseless, uint32_t n_patterns, pfac_tables **out);
/* The rules of any set, one per pattern (n = pfac_tables_n_patterns, PFAC_ERR_ARG otherwise): all 1 for caseless
 * sets, all 0 for plain sets and sets wrapped from arrays. */
int pfac_tables_case_rules(const pfac_tables *t, uint8_t *caseless, uint32_t n);
/* Wrap caller-built canonical arrays (the thread_data fields of main.cc:19-32) as a
 * one-partition table set; arrays are copied.  n_r = state_num*256/width + 1
 * (master_kernel.cu:221). */
int pfac_tables_from_arrays(const int32_t *s0, const int32_t *r, int32_t n_r, const int32_t *HT,
                            const int32_t *val, int32_t ht_size, int32_t width, int32_t state_num,
                            int32_t n_final, const int32_t *idmap, int32_t max_pat_len,
                            pfac_tables **out);
/* On-disk cache of the canonical arrays of every partition (checksummed; the reference rebuilds its
 * tables on every run, main.cc:100-126).  A loaded set scans exactly like the set that was saved,
 * caseless and mixed sets included: they are written as PFACTBL3 files (PFACTBL2 plus the flags; a mixed set
 * adds its rules and verify tables under the checksum), which older libraries refuse, and case-sensitive sets as
 * PFACTBL2 files.  pfac_tables_load reads both. */
/* What a table set was built from: a 64-bit hash of the pattern file image and the front-end flags
 * (0 for sets wrapped from arrays).  It travels with pfac_tables_save/_load, so that a cache can be
 * checked against the pattern file it is about to stand in for (pfac_pattern_file_hash). */
uint64_t pfac_tables_source_hash(const pfac_tables *t);
int pfac_pattern_file_hash(const char *pattern_file, unsigned flags, uint64_t *hash);
/* The source hash of the set pfac_tables_build_file_rules builds: FNV over the image, the flags and the rule
 * bytes for mixed rules, the uniform set's hash for uniform ones.  The refusals of the builder apply. */
int pfac_pattern_file_hash_rules(const char *pattern_file, unsigned flags, const uint8_t *caseless,
                                 uint32_t n_patterns, uint64_t *hash);
int pfac_tables_save(const pfac_tables *t, const char *path);
int pfac_tables_load(const char *path, pfac_tables **out);
void pfac_tables_destroy(pfac_tables *t);

int pfac_tables_n_parts(const pfac_tables *t);
int pfac_tables_n_patterns(const pfac_tables *t);
int pfac_tables_max_pat_len(const pfac_tables *t); /* over all partitions, main.cc:59 */
int pfac_tables_width(const pfac_tables *t);
/* The front-end flags that change what a set matches: PFAC_PATTERNS_CASELESS, PFAC_PATTERNS_CASE_RULES (mixed
 * per-pattern rules) or 0 (sets wrapped from arrays are case-sensitive). */
unsigned pfac_tables_flags(const pfac_tables *t);
/* info[0..8] = state_num, n_final, max_len, ht_size, n_r, n_keys, max_key, max_offset, min_len */
int pfac_tables_part_info(const pfac_tables *t, int part, int32_t info[9]);
const int32_t *pfac_tables_s0(const pfac_tables *t, int part);    /* 256 entries, main.cc:200 */
const int32_t *pfac_tables_r(const pfac_tables *t, int part);     /* n_r entries */
const int32_t *pfac_tables_HT(const pfac_tables *t, int part);    /* ht_size entries */
const int32_t *pfac_tables_val(const pfac_tables *t, int part);   /* ht_size entries */
const int32_t *pfac_tables_idmap(const pfac_tables *t, int part); /* n_final entries */
/* Builds the detector kernel's shared-memory filters for this partition on the host (the same
 * code pfac_ctx_create runs) and verifies them against the canonical PHF: T1 is exact over the
 * first two bytes, every pattern's own bytes pass T1s / T2 / Tm / Tm2 / T3.  stats[0..9] = image
 * bytes, T1 pairs, T2 bits set, 4-byte prefixes, short patterns present, Tm/T3 present, Tm keys,
 * Tm2 keys, T3 bits set, log2 Tm2 buckets.  t2/t3/tm2_bytes = shared-memory budget.  Needs no GPU. */
int pfac_tables_derive_check(const pfac_tables *t, int part, uint32_t t2_bytes, uint32_t t3_bytes,
                             uint32_t tm2_bytes, uint64_t stats[10]);
/* Diagnostics: how many start positions of `text` survive each stage of the detector's filter
 * cascade (a host model that COUNTS; it reports no matches).  counts[0..8] = positions, T1 pass,
 * prefix found (T2 / level 1), level-1 window pass, level-2 window pass, bypass, starts left as
 * candidates, 512-byte slices flagged, slices.  A caseless or mixed set counts its folded text, as the detector
 * sees it. */
int pfac_tables_filter_profile(const pfac_tables *t, int part, uint32_t t2_bytes, uint32_t t3_bytes,
                               uint32_t tm2_bytes, const void *text, uint64_t n, uint64_t counts[12]);
/* One transition through the PHF exactly as master_kernel.cu:52-64 does it; -1 = none. */
int32_t pfac_tables_lookup(const pfac_tables *t, int part, int32_t state, int32_t byte);
/* Pattern length of every id: lengths[id] = depth of the final state that reports id, 0 for ids no final
 * state reports (earlier duplicates, which caseless sets make common: with "GET" and "get" in one file
 * only the later line's id is ever reported).  A mixed set (PFAC_PATTERNS_CASE_RULES) reports the length of every
 * member of its verify tables, so 0 only for lines shadowed within their rule class.
 * lengths may be NULL: *n_ids receives max id + 1 (size of the array).
 * PFAC_ERR_ARG if the automaton is not a tree, PFAC_ERR_OUTPUT_FULL if n < max id + 1. */
int pfac_tables_pattern_lengths(const pfac_tables *t, int part, int32_t *lengths, int32_t n, int32_t *n_ids);

/* ------------------------------------------------------------------------------ device
 * pfac_ctx_create replaces GPU_Malloc_Memory (master_kernel.cu:188-257) and the table half
 * of GPU_TraceTable's H2D copies (master_kernel.cu:365-383): the tables are uploaded once.
 * `n_streams` = pipeline depth of pfac_scan_host (argv[2], "stream number per GPU");
 * `chunk_bytes` = input bytes per pipeline stage (0 = default). */
int pfac_device_count(int *count);
int pfac_ctx_create(int device, const pfac_tables *t, int part, int n_streams, size_t chunk_bytes,
                    pfac_ctx **out);
void pfac_ctx_destroy(pfac_ctx *ctx); /* GPU_Free_memory, master_kernel.cu:457-524 */
int pfac_ctx_device(const pfac_ctx *ctx);

/* Kernel half of GPU_TraceTable (master_kernel.cu:400-418) on DEVICE-RESIDENT input.
 * Start positions are bytes [0, n_starts) of d_in; bytes [0, n_valid) are readable input
 * (n_valid >= n_starts; the extra bytes are the halo, at most max_pat_len-1 are used).
 * `base_pos` = global position of d_in[0] (only used to reproduce the reference's 4096+512
 * tile walk bound for patterns longer than 513 bytes, master_kernel.cu:141-144).
 * d_out: device array of `cap` pfac_match; d_count: device uint64 receiving the number of
 * matches found.  If it exceeds cap nothing is written past d_out[cap) and the contents
 * of d_out are unspecified: size the buffer from the count and scan again.
 * Size bound per call: min(n_valid, n_starts + max_pat_len - 1) + (d_in & 15) + 12,288 < 2^32
 * (PFAC_ERR_LIMIT otherwise), i.e. up to 2^32 - 12,289 - (d_in & 15) bytes.
 * Asynchronous on `stream`.  Scans of one context share one working set: a call on another
 * stream than the previous one is ordered after it on the device (use one context per stream
 * for scans that should overlap).
 * Caseless sets (PFAC_PATTERNS_CASELESS): the caller's bytes are never written; they are folded into a
 * buffer of the context at the same 16-byte phase, which grows to the largest input scanned so far (up
 * to 4 GiB) and is held until pfac_ctx_destroy.  pfac_scan_batch_device does the same; pfac_scan_host and
 * the flow calls fold the library's own copy of the input in place.
 * Mixed sets (PFAC_PATTERNS_CASE_RULES) fold every input out of place, the library's own buffers included (the
 * exact patterns are checked against the original bytes, and a flow's carried tails stay unfolded): one folded
 * buffer per pipeline stage of pfac_scan_host, one of the packed-buffer size for flow calls, and one for the
 * caller's input, each held until pfac_ctx_destroy.  The detector's records (owner ids) go to a buffer of
 * max(cap, 4096) records; the verify pass expands them into d_out.  If the detector's records overflow that
 * buffer, the count returned is their count times the largest group (a capacity with which a rescan fits);
 * if only the expanded records overflow, the count is exact.  Either way nothing is written past d_out[cap). */
int pfac_scan_device(pfac_ctx *ctx, const void *d_in, uint64_t n_starts, uint64_t n_valid,
                     uint64_t base_pos, void *d_out, uint64_t cap, void *d_count, void *stream);
/* Same, synchronous; *count receives the device count.  PFAC_ERR_OUTPUT_FULL if *count > cap. */
int pfac_scan_device_sync(pfac_ctx *ctx, const void *d_in, uint64_t n_starts, uint64_t n_valid,
                          uint64_t base_pos, void *d_out, uint64_t cap, uint64_t *count, void *stream);

/* Batch of independent documents (packets, log lines, requests) in ONE launch sequence; the reference has
 * no counterpart.  The result of document i is exactly what pfac_scan_device returns for it alone
 * (n_starts = n_valid = its length, base_pos = 0): a match never crosses from one document into the next.
 * The packed buffer is scanned once; a split pass then drops the records whose pattern runs past the end
 * of their document and makes positions relative to it.  Supported by contexts whose automaton is a tree
 * (PFAC_ERR_ARG otherwise: sets wrapped from arrays may share states) and whose patterns are at most 513
 * bytes long (PFAC_ERR_LIMIT otherwise: beyond that the reference's 4096+512 tile bound makes results
 * depend on where a document lies in the buffer).
 *
 * n_docs independent documents packed back to back in d_in: document i = d_in[doc_offsets[i], doc_offsets[i+1]).
 * doc_offsets is a HOST array of n_docs + 1 entries, doc_offsets[0] = 0, non-decreasing; the total
 * doc_offsets[n_docs] + (d_in & 15) + 12,288 < 2^32 as for pfac_scan_device (PFAC_ERR_LIMIT otherwise).  The array
 * is read before the call returns.
 * d_out: device array of `cap` pfac_match, pos relative to the record's document; records ordered by
 * (document, pos, pattern length).  d_doc_first: device uint64[n_docs + 1], the records of document i are
 * d_out[d_doc_first[i], d_doc_first[i+1]).  d_count: device uint64.  If the count exceeds cap, nothing is
 * written past d_out[cap), d_out and d_doc_first are unspecified, and the count is a capacity that suffices
 * for a rescan (it may exceed the records the rescan returns by the matches straddling document boundaries).
 * Same stream and ordering rules as pfac_scan_device (shares its working set). */
int pfac_scan_batch_device(pfac_ctx *ctx, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                           void *d_out, uint64_t cap, void *d_doc_first, void *d_count, void *stream);
/* Same, synchronous; *count receives the device count.  PFAC_ERR_OUTPUT_FULL if *count > cap. */
int pfac_scan_batch_device_sync(pfac_ctx *ctx, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                                void *d_out, uint64_t cap, void *d_doc_first, uint64_t *count, void *stream);

/* Streaming scan of many flows (packets or reads of many connections, one chunk at a time); the reference has
 * no counterpart.  A flow set holds n_flows independent byte streams.  Flow f has consumed P_f bytes so far, and
 * the device keeps its last t_f = min(max_pat_len - 1, P_f) bytes.  One call takes n_chunks chunks for DISTINCT
 * flows; the records of chunk i (flow f) are exactly the matches of flow f's whole stream whose end lies in the
 * chunk, (P_f, P_f + c_i], so the union of a flow's records over its calls equals one pfac_scan_device over its
 * concatenated bytes: nothing missing, nothing twice.  Records of one chunk are ordered by (pos, pattern length);
 * across calls they are NOT globally position-ordered (a long match that ends late is reported after a shorter
 * one that starts after it).  Same preconditions as the batch scan: pfac_flows_create returns PFAC_ERR_ARG for a
 * context whose automaton is not a tree and PFAC_ERR_LIMIT for patterns longer than 513 bytes.
 *
 * A call either commits or leaves every flow unchanged: on PFAC_ERR_OUTPUT_FULL, on refused arguments or when
 * the device watchdog trips no tail and no P_f advances, and a rescan with the returned count as capacity gives
 * exactly the records the call would have given with enough room.  After PFAC_ERR_CUDA the state of the set is
 * unspecified: reset every flow.  Hence the call is synchronous only.  Calls of one set are serialised; the set
 * uses the context's working set like pfac_scan_device (same stream ordering rules).
 *
 * pfac_flows_destroy before its context.  pfac_flows_reset: flow starts a new stream (P_f = 0, empty tail);
 * pfac_flows_position: *bytes = P_f. */
int pfac_flows_create(pfac_ctx *ctx, uint32_t n_flows, pfac_flows **out);
void pfac_flows_destroy(pfac_flows *f);
int pfac_flows_reset(pfac_flows *f, uint32_t flow);
int pfac_flows_position(const pfac_flows *f, uint32_t flow, uint64_t *bytes);
/* Chunk i = d_in[chunk_offsets[i], chunk_offsets[i+1]) (a HOST array of n_chunks + 1 entries, chunk_offsets[0] = 0,
 * non-decreasing) goes to flow flow_ids[i] (a HOST array, distinct ids < n_flows).  d_out, d_chunk_first, *count,
 * cap and PFAC_ERR_OUTPUT_FULL as for pfac_scan_batch_device_sync, with the chunks in place of the documents and
 * pos relative to base[i] (a HOST uint64[n_chunks]: base[i] = P_f - t_f, the stream position of the first carried
 * byte), so a record's stream position is base[i] + pos and flows may run past 4 GiB.  PFAC_ERR_ARG for a flow id
 * out of range or named twice, chunk_offsets[0] != 0 or decreasing offsets; PFAC_ERR_LIMIT when the chunks reach
 * 4 GiB or the packed bytes (chunks plus carried tails) + 12,288 reach 2^32.  All refusals come before anything is
 * enqueued. */
int pfac_scan_flows_device_sync(pfac_flows *f, const void *d_in, const uint64_t *chunk_offsets,
                                const uint32_t *flow_ids, uint32_t n_chunks, void *d_out, uint64_t cap,
                                void *d_chunk_first, uint64_t *base, uint64_t *count, void *stream);

/* Whole GPU_TraceTable (H2D + kernel + D2H, master_kernel.cu:359-428) on HOST input, as a
 * pipeline of chunk_bytes sub-chunks (+halo) over n_streams streams.  h_in[0, n_starts) are
 * start positions, h_in[0, n_valid) readable.  h_out receives up to `cap` records ordered by
 * position (pos relative to h_in[0]); pinned buffers (pfac_host_alloc) copy fastest.
 * n_valid must be < 2^32. */
int pfac_scan_host(pfac_ctx *ctx, const void *h_in, uint64_t n_starts, uint64_t n_valid,
                   uint64_t base_pos, pfac_match *h_out, uint64_t cap, uint64_t *count);

/* Pinned host memory (cudaHostAlloc portable, as main.cc:147,161). */
int pfac_host_alloc(void **ptr, size_t bytes);
void pfac_host_free(void *ptr);
/* Pin memory the caller already has (e.g. an mmap of the input file, read_only = 1) so that H2D
 * copies run at link speed without a staging copy; the reference freads the whole file into a
 * cudaHostAlloc buffer instead (main.cc:147-155).  Failure is not fatal: scan from pageable memory. */
int pfac_host_register(const void *ptr, size_t bytes, int read_only);
void pfac_host_unregister(const void *ptr);

/* Counters of the last scan on this context (for bench.py's gpu_launches / roofline):
 * info[0] = kernel launches, info[1] = tiles, info[2] = CTAs, info[3] = dynamic smem bytes,
 * info[4] = h2d bytes, info[5] = d2h bytes, info[6] = sub-chunks, info[7] = reserved (0).  The launches
 * of a caseless set count the fold kernel of every scan; those of a mixed set (PFAC_PATTERNS_CASE_RULES) count
 * the fold and the two kernels of the verify pass of every scan (caseless launches + 2). */
int pfac_ctx_last_scan_info(const pfac_ctx *ctx, uint64_t info[8]);

/* Optional CUDA-event timing of the detector kernel (pfac_scan_kernel) alone, for roofline
 * reports: after pfac_ctx_set_timing(ctx, 1) every scan records an event pair around that kernel
 * on the scan's stream (ring of 256 launches); pfac_ctx_kernel_time synchronises the device, sums
 * the recorded launches since the last call and resets the ring. */
int pfac_ctx_set_timing(pfac_ctx *ctx, int enable);
int pfac_ctx_kernel_time(pfac_ctx *ctx, double *ms_total, int *n_launches);

/* Derived (shared-memory) table statistics of this context, for DESIGN.md / bench.py:
 * info[0] = image bytes, [1] = T1 pairs set, [2] = T2 bits, [3] = T2 bits set, [4] = 4-byte prefixes,
 * [5] = short patterns (<= 3 bytes) present, [6] = Tm keys, [7] = Tm2 keys, [8] = T3 bits,
 * [9] = T3 bits set, [10] = dynamic smem bytes, [11] = table bytes in HBM, [12] = input ring stages,
 * [13] = log2 Tm2 buckets, [14] = mode (0 two-point checks from shared memory, 1 T2 only,
 * 2 two-point tables in global memory), [15] = log2 Tm buckets */
int pfac_ctx_derived_info(const pfac_ctx *ctx, uint64_t info[16]);

/* ------------------------------------------------------------------------------ multi-GPU job
 * Replaces the GPU x stream loop of main.cc:171-272.  The INPUT is sharded (the reference
 * shards patterns and replicates the input): GPU g scans a contiguous chunk plus a halo of
 * max_pat_len-1 bytes; one host thread per GPU; no inter-GPU traffic.  Results come back as
 * position-ordered segments with 64-bit base positions. */
int pfac_job_create(const pfac_tables *t, const int *devices, int n_devices, int streams_per_gpu,
                    size_t chunk_bytes, pfac_job **out);
void pfac_job_destroy(pfac_job *job);
/* Scan h_in[0, n) (n = file size - 1 for the CLI, main.cc:138).  On return *n_matches is the
 * total.  Records are kept inside the job until the next run. */
int pfac_job_run(pfac_job *job, const void *h_in, uint64_t n, uint64_t *n_matches);
/* The same, reading the input from a file (main.cc:131-155 reads the whole file into pinned memory
 * before anything is scanned): per GPU a reader thread preads its shard in 64 MiB chunks (buffered
 * with sequential read-ahead; O_DIRECT with PFAC_READER_ODIRECT=1) into a ring of pinned buffers
 * while the chunks that are in are scanned; scanning starts with the first chunk.  `n` = bytes of the file to scan (file size - 1
 * for the CLI). */
int pfac_job_run_file(pfac_job *job, const char *path, uint64_t n, uint64_t *n_matches);
int pfac_job_n_segments(const pfac_job *job);
/* Segment i: records[count] with positions relative to *base_pos; segments are in position order. */
int pfac_job_segment(const pfac_job *job, int i, uint64_t *base_pos, const pfac_match **records,
                     uint64_t *count);
/* The sharding rule pfac_job_run applies, as a pure function (also used by bench.py to cut one
 * shard per rank): shard `i` of `n_shards` over an input of `n` bytes owns the start positions
 * [*start, *start + *n_starts) and may read *n_valid >= *n_starts bytes from *start (its halo =
 * the first max_pat_len-1 bytes of the next shard, clipped to n).  Shard sizes are multiples of
 * 64 KiB except the last; trailing shards may be empty. */
int pfac_job_plan(uint64_t n, int n_shards, int max_pat_len, int i, uint64_t *start, uint64_t *n_starts,
                  uint64_t *n_valid);
/* wall-clock seconds of the last run: [0] total scan (H2D+kernel+D2H, all GPUs) */
int pfac_job_last_timing(const pfac_job *job, double secs[4]);

/* ------------------------------------------------------------------------------ writer
 * main.cc:335-350: one line "At position %4d, match pattern %d\n" per record. */
int pfac_write_begin(const char *path, void **writer);
int pfac_write_records(void *writer, uint64_t base_pos, const pfac_match *records, uint64_t count);
int pfac_write_end(void *writer);
/* Format into memory (tests): returns bytes needed; writes at most buf_len. */
size_t pfac_format_records(uint64_t base_pos, const pfac_match *records, uint64_t count, char *buf,
                           size_t buf_len);


/* Optional binary sidecar of the compact records (the reference has none: main.cc:335-350 writes text only).
 * File = 32-byte header {"PFACREC1", u32 version = 1, u32 record bytes = 8, u64 blocks, u64 records}, then per
 * pfac_sidecar_records call with count > 0 one block {u64 base_pos, u64 count, count x pfac_match}; little-endian.
 * The header's totals are written by pfac_sidecar_end.  GPU_match_result.txt is a pure function of the sidecar. */
int pfac_sidecar_begin(const char *path, void **sidecar);
int pfac_sidecar_records(void *sidecar, uint64_t base_pos, const pfac_match *records, uint64_t count);
int pfac_sidecar_end(void *sidecar);
/* Read a sidecar back: *n_records = the total; with pos / id non-NULL (capacity `cap` records each, either may
 * be NULL) the absolute 64-bit positions and pattern ids in file order.  PFAC_ERR_OUTPUT_FULL if cap is too
 * small, PFAC_ERR_IO for a file that is not a complete sidecar. */
int pfac_sidecar_read(const char *path, uint64_t *pos, uint32_t *id, uint64_t cap, uint64_t *n_records);

#ifdef __cplusplus
}
#endif
#endif /* PFAC_B200_H */
