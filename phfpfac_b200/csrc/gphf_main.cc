// gphf -- command-line driver with the reference's surface (regex_GPU_PHF/main.cc:45-352):
//
//     gphf <pattern file name> <stream number per GPU> <Hash table width> <input file name>
//
// writes GPU_match_result.txt in the current directory (main.cc:335), byte-identical to the
// reference.  argv[2] keeps its place but means "pipeline streams per GPU" (input sub-chunks
// in flight); the result does not depend on it.  Exits 1 with a message on any failure, 255
// on a usage error (the reference's exit(-1), main.cc:95).
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "pfac_b200.h"

static double now()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static int fail(const char *what)
{
    fprintf(stderr, "%s: %s\n", what, pfac_last_error());
    return 1;
}

// main.cc:335-350: the job's position-ordered segments -> GPU_match_result.txt; with GPHF_SIDECAR=<file> also the
// binary sidecar of the compact records (pfac_sidecar_*; the reference has no such file)
static int write_results(const pfac_job *job, const char *out_name)
{
    const char *side_name = getenv("GPHF_SIDECAR");
    void *w = nullptr, *sc = nullptr;
    if (pfac_write_begin(out_name, &w)) return fail("open output");
    if (side_name && *side_name && pfac_sidecar_begin(side_name, &sc)) return fail("open sidecar");
    for (int i = 0; i < pfac_job_n_segments(job); i++) {
        uint64_t base, cnt;
        const pfac_match *rec;
        pfac_job_segment(job, i, &base, &rec, &cnt);
        if (pfac_write_records(w, base, rec, cnt)) return fail("write output");
        if (sc && pfac_sidecar_records(sc, base, rec, cnt)) return fail("write sidecar");
    }
    if (pfac_write_end(w)) return fail("close output");
    if (sc && pfac_sidecar_end(sc)) return fail("close sidecar");
    return 0;
}

static bool read_all(const char *path, std::vector<unsigned char> &out)
{
    FILE *f = fopen(path, "rb");
    if (!f) return false;
    unsigned char tmp[1 << 16];
    size_t got;
    while ((got = fread(tmp, 1, sizeof tmp, f)) > 0) out.insert(out.end(), tmp, tmp + got);
    fclose(f);
    return true;
}

// The patterns a well-formed pattern file holds: one per raw newline, except, with the escape reader, a newline
// that "\x" skips as white space before its hex digits (a malformed file is refused by the builder)
static uint32_t count_patterns(const std::vector<unsigned char> &b, bool escapes)
{
    uint32_t n = 0;
    for (size_t i = 0; i < b.size(); i++) {
        if (escapes && b[i] == '\\' && i + 1 < b.size()) {
            const unsigned char c = b[i + 1];
            if (c == 'x') {
                size_t j = i + 2;
                while (j < b.size() && (b[j] == ' ' || (b[j] >= 9 && b[j] <= 13))) j++;
                i = j - 1;
            } else if (c && strchr("abtnvfr'\"\\", c)) {
                i++;   // a two-byte escape
            }          // else octal digits or no escape: the bytes after the backslash are read on their own
            continue;
        }
        n += b[i] == '\n';
    }
    return n;
}

// GPHF_NOCASE_LINES=<file>: the 1-based numbers of the patterns that match in either case, one decimal per line;
// every other pattern of the n matches byte for byte.  false (with a message) for an unparsable line or a number
// out of range.
static bool read_nocase_lines(const char *path, uint32_t n, std::vector<uint8_t> &rules)
{
    std::vector<unsigned char> b;
    if (!read_all(path, b)) {
        fprintf(stderr, "GPHF_NOCASE_LINES: cannot read %s\n", path);
        return false;
    }
    rules.assign(n, 0);
    size_t line = 0;
    for (size_t i = 0; i < b.size();) {
        line++;
        size_t j = i;
        uint64_t v = 0;
        for (; j < b.size() && b[j] >= '0' && b[j] <= '9'; j++)
            if (v <= n) v = v * 10 + (uint64_t)(b[j] - '0');   // (saturates above n: out of range)
        if (j == i || (j < b.size() && b[j] != '\n')) {
            fprintf(stderr, "GPHF_NOCASE_LINES: line %zu of %s is not a pattern number\n", line, path);
            return false;
        }
        if (v < 1 || v > n) {
            fprintf(stderr, "GPHF_NOCASE_LINES: pattern %llu (line %zu of %s) is out of range: the file has %u patterns\n",
                    (unsigned long long)v, line, path, n);
            return false;
        }
        rules[(size_t)v - 1] = 1;
        i = j + 1;
    }
    return true;
}

int main(int argc, char **argv)
{
    if (argc != 5) {   // main.cc:93-96
        fprintf(stderr, "usage: %s <pattern file name> <streamnum> <PHF width> <input file name>\n", argv[0]);
        return 255;
    }
    const int streamnum = atoi(argv[2]);   // main.cc:48
    const int width = atoi(argv[3]);       // main.cc:120
    if (streamnum < 1) {
        fprintf(stderr, "stream number per GPU must be >= 1\n");
        return 1;
    }
    const char *out_name = getenv("GPHF_OUTPUT") ? getenv("GPHF_OUTPUT") : "GPU_match_result.txt";   // main.cc:335

    double t0 = now();
    pfac_tables *tables = nullptr;
    // GPHF_ESCAPES=1: read the patterns through the reference's (unused) escape reader, read_pattern_ext
    // GPHF_CASELESS=1: ASCII letters match in either case (PFAC_PATTERNS_CASELESS)
    const unsigned pflags = (getenv("GPHF_ESCAPES") && atoi(getenv("GPHF_ESCAPES")) ? PFAC_PATTERNS_ESCAPES : 0u) |
                            (getenv("GPHF_CASELESS") && atoi(getenv("GPHF_CASELESS")) ? PFAC_PATTERNS_CASELESS : 0u);
    // GPHF_NOCASE_LINES=<file>: per-pattern case rules (pfac_tables_build_file_rules): the patterns it numbers
    // match in either case, every other one byte for byte
    const char *nocase = getenv("GPHF_NOCASE_LINES");
    std::vector<uint8_t> rules;
    unsigned want_flags = pflags & PFAC_PATTERNS_CASELESS;
    if (nocase && *nocase) {
        if (pflags & PFAC_PATTERNS_CASELESS) {
            fprintf(stderr, "GPHF_NOCASE_LINES and GPHF_CASELESS=1 exclude each other\n");
            return 1;
        }
        std::vector<unsigned char> image;
        if (!read_all(argv[1], image)) {
            fprintf(stderr, "Open input file failed: %s\n", argv[1]);
            return 1;
        }
        if (!read_nocase_lines(nocase, count_patterns(image, (pflags & PFAC_PATTERNS_ESCAPES) != 0), rules)) return 1;
        const size_t ones = (size_t)std::count(rules.begin(), rules.end(), (uint8_t)1);
        want_flags = ones == rules.size() ? PFAC_PATTERNS_CASELESS : ones == 0 ? 0u : PFAC_PATTERNS_CASE_RULES;
    }
    const bool with_rules = !rules.empty();
    // GPHF_TABLE_CACHE=<file>: load the tables from it if it exists and was built from this pattern file
    // (hash of the file image + front-end flags [+ case rules] in the cache header) at this width, else build them
    // and write it
    const char *cache = getenv("GPHF_TABLE_CACHE");
    bool from_cache = false;
    if (cache && *cache) {
        FILE *probe = fopen(cache, "rb");
        if (probe) {
            fclose(probe);
            if (pfac_tables_load(cache, &tables)) return fail("load the table cache");
            uint64_t want = 0;
            if (with_rules ? pfac_pattern_file_hash_rules(argv[1], pflags, rules.data(), (uint32_t)rules.size(), &want)
                           : pfac_pattern_file_hash(argv[1], pflags, &want))
                return fail("read the pattern file");
            if (pfac_tables_width(tables) != width || pfac_tables_n_parts(tables) != 1 ||
                pfac_tables_source_hash(tables) != want || pfac_tables_flags(tables) != want_flags) {
                // built from another pattern file, width or front-end flags: rebuild (and rewrite the cache)
                fprintf(stderr, "%s does not belong to this pattern file / width: rebuilding the tables\n", cache);
                pfac_tables_destroy(tables);
                tables = nullptr;
            } else {
                from_cache = true;
            }
        }
    }
    if (!from_cache) {
        if (with_rules ? pfac_tables_build_file_rules(argv[1], 1, width, pflags, rules.data(), (uint32_t)rules.size(), &tables)
                       : pfac_tables_build_file_ext(argv[1], 1, width, pflags, &tables))
            return fail("create PFAC/PHF tables");
        if (cache && *cache && pfac_tables_save(tables, cache)) return fail("write the table cache");
    }
    double t1 = now();
    int32_t info[9];
    pfac_tables_part_info(tables, 0, info);
    printf("state num : %d\nfinal state num : %d\nmax pattern length : %d\nhash table size : %d\n", info[0],
           info[1], info[2], info[3]);

    // Input: the reference freads the file into a cudaHostAlloc buffer (main.cc:131-155).  Here the
    // file is mapped and the mapping pinned in place (no second copy of a multi-GB input); if either
    // step is refused, fall back to the reference's way.  GPHF_READER=fread forces the fallback.
    int fd = open(argv[4], O_RDONLY);
    if (fd < 0) {
        perror("Open input file failed.");
        return 1;
    }
    struct stat sb;
    if (fstat(fd, &sb) != 0) {
        perror("Open input file failed.");
        return 1;
    }
    const long long fsize = (long long)sb.st_size;
    const uint64_t input_size = fsize > 0 ? (uint64_t)fsize - 1 : 0;   // main.cc:138 (drops the last byte)
    printf("input size is %llu char\n", (unsigned long long)input_size);

    int n_gpu = 0;
    if (pfac_device_count(&n_gpu) || n_gpu < 1) return fail("no CUDA device");   // main.cc:50
    if (getenv("GPHF_GPUS")) n_gpu = std::max(1, std::min(n_gpu, atoi(getenv("GPHF_GPUS"))));

    void *input = nullptr, *mapped = nullptr;
    bool registered = false;
    // GPHF_READER = stream | mmap | fread.  Default: files of 256 MiB and more are streamed (reader threads
    // fill a ring of pinned buffers chunk by chunk, O_DIRECT where possible, while the chunks that are in
    // are scanned -- pfac_job_run_file); smaller ones are mapped and pinned in place.
    const char *reader_env = getenv("GPHF_READER");
    const bool want_stream = reader_env ? !strcmp(reader_env, "stream") : fsize >= (256ll << 20);
    const bool want_mmap = !want_stream && !(reader_env && !strcmp(reader_env, "fread"));
    if (want_stream) {
        close(fd);
        pfac_job *job = nullptr;
        if (pfac_job_create(tables, nullptr, n_gpu, streamnum, 0, &job)) return fail("create GPU contexts");
        printf("input reader: stream (reader thread per GPU, ring of pinned 64 MiB buffers)\n");
        double t2 = now();
        uint64_t n_matches = 0;
        if (pfac_job_run_file(job, argv[4], input_size, &n_matches)) return fail("scan");
        double t3 = now();
        if (write_results(job, out_name)) return 1;
        double t4 = now();
        printf("/////////////////////////////////////////////\n");
        printf("1.Time for  create PFAC + Hashtable : %lf seconds\n", t1 - t0);
        printf("2.Time for  %d GPU setup: %lf mseconds\n", n_gpu, (t2 - t1) * 1000);
        printf("3.Time for  %d GPU match progress, file read included: %lf mseconds (%.3f GB/s file to records)\n", n_gpu,
               (t3 - t2) * 1000, input_size / (t3 - t2) / 1e9);
        printf("4.Time for  writing %llu matches: %lf mseconds\n", (unsigned long long)n_matches, (t4 - t3) * 1000);
        printf("5.Wall time file -> %s: %lf seconds\n", out_name, t4 - t0);
        printf("matching process finshed\n");
        printf("/////////////////////////////////////////////\n");
        pfac_job_destroy(job);
        pfac_tables_destroy(tables);
        return 0;
    }
    if (want_mmap && fsize > 0) {
        mapped = mmap(nullptr, (size_t)fsize, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
        if (mapped == MAP_FAILED) mapped = nullptr;
    }
    if (mapped) {
        registered = pfac_host_register(mapped, (size_t)fsize, 1) == 0;
        input = mapped;
        printf("input reader: mmap%s\n", registered ? " + pinned in place" : " (pageable)");
    } else {
        if (pfac_host_alloc(&input, (size_t)input_size + 1)) return fail("cudaHostAlloc input");   // main.cc:147
        size_t got = 0;
        while (got < (size_t)input_size) {                                                          // main.cc:154
            ssize_t r = read(fd, (char *)input + got, (size_t)input_size - got);
            if (r <= 0) {
                fprintf(stderr, "short read on %s\n", argv[4]);
                return 1;
            }
            got += (size_t)r;
        }
        printf("input reader: fread into pinned memory\n");
    }
    close(fd);

    pfac_job *job = nullptr;
    if (pfac_job_create(tables, nullptr, n_gpu, streamnum, 0, &job)) return fail("create GPU contexts");
    double t2 = now();
    uint64_t n_matches = 0;
    if (pfac_job_run(job, input, input_size, &n_matches)) return fail("scan");
    double t3 = now();

    if (write_results(job, out_name)) return 1;
    double t4 = now();

    printf("/////////////////////////////////////////////\n");
    printf("1.Time for  create PFAC + Hashtable : %lf seconds\n", t1 - t0);
    printf("2.Time for  %d GPU setup: %lf mseconds\n", n_gpu, (t2 - t1) * 1000);
    printf("3.Time for  %d GPU match progress: %lf mseconds (%.3f GB/s end to end)\n", n_gpu, (t3 - t2) * 1000,
           input_size / (t3 - t2) / 1e9);
    printf("4.Time for  writing %llu matches: %lf mseconds\n", (unsigned long long)n_matches, (t4 - t3) * 1000);
    printf("5.Wall time file -> %s: %lf seconds\n", out_name, t4 - t0);
    printf("matching process finshed\n");
    printf("/////////////////////////////////////////////\n");
    pfac_job_destroy(job);
    if (mapped) {
        if (registered) pfac_host_unregister(mapped);
        munmap(mapped, (size_t)fsize);
    } else {
        pfac_host_free(input);
    }
    pfac_tables_destroy(tables);
    return 0;
}
