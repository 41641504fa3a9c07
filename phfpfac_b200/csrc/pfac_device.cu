// Device side of the C ABI (include/pfac_b200.h): contexts, table upload, the device-resident
// scan, the host pipeline, batch scans and streaming scans of many flows.  Replaces GPU_Malloc_Memory /
// GPU_TraceTable / GPU_Free_memory (reference master_kernel.cu:188-524).  There is no CPU fallback
// anywhere in this file: a missing GPU or any CUDA error is reported as PFAC_ERR_NO_DEVICE / PFAC_ERR_CUDA.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>

#include "pfac_batch.cuh"
#include "pfac_derive.h"
#include "pfac_flows.cuh"
#include "pfac_fold.cuh"
#include "pfac_internal.h"
#include "pfac_kernel.cuh"
#include "pfac_rules.cuh"

using namespace pfac;

#define CU_TRY(expr)                                                                         \
    do {                                                                                     \
        cudaError_t e_ = (expr);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return set_error(PFAC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                  \
                             cudaGetErrorString(e_), __FILE__, __LINE__);                    \
    } while (0)

namespace {

// cap() elements of T in device memory (Host: pinned host memory), owned: the destructor frees them.  Every
// buffer of this file is one of these.
template <typename T, bool Host = false>
class Buf {
public:
    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    ~Buf() { release(); }
    T *get() const { return p_; }
    size_t cap() const { return cap_; }
    size_t bytes() const { return cap_ * sizeof(T); }

    // n elements in place of the old ones, which nothing may still use; zero: filled with zero bytes.  On
    // failure the buffer is left empty.
    int alloc(size_t n, bool zero = false)
    {
        release();
        void *p = nullptr;
        const size_t b = n * sizeof(T);
        cudaError_t e = Host ? cudaHostAlloc(&p, b, cudaHostAllocPortable) : cudaMalloc(&p, b);
        if (e == cudaSuccess) {
            p_ = static_cast<T *>(p);
            if (zero) e = cudaMemset(p, 0, b);
        }
        if (e != cudaSuccess) {
            release();
            return set_error(PFAC_ERR_CUDA, "%s(%zu bytes) failed: %s", Host ? "cudaHostAlloc" : "cudaMalloc", b,
                             cudaGetErrorString(e));
        }
        cap_ = n;
        return PFAC_OK;
    }
    // At least n elements (a growth allocates max(n, floor)).  Growing synchronises `stream` first: the old
    // buffer may still be in use there.  Steady-state calls return at once.
    int reserve(size_t n, size_t floor, cudaStream_t stream, bool zero = false)
    {
        if (n <= cap_) return PFAC_OK;
        CU_TRY(cudaStreamSynchronize(stream));
        return alloc(std::max(n, floor), zero);
    }
    // a device copy of v
    int upload(const std::vector<T> &v)
    {
        int e = alloc(v.size());
        if (e) return e;
        CU_TRY(cudaMemcpy(p_, v.data(), bytes(), cudaMemcpyHostToDevice));
        return PFAC_OK;
    }

private:
    void release()
    {
        if (p_) Host ? cudaFreeHost(p_) : cudaFree(p_);
        p_ = nullptr;
        cap_ = 0;
    }
    T *p_ = nullptr;
    size_t cap_ = 0;
};

// Per-call arrays of a launch sequence (a batch's document offsets, a flow call's per-chunk arrays): filled in
// pinned memory and uploaded with one cudaMemcpyAsync.  Before the buffer is refilled the host waits for the
// event of its previous upload, so an asynchronous call is never overwritten by the next.
struct Staging {
    Buf<uint32_t, true> h;
    Buf<uint32_t> d;
    cudaEvent_t copied = nullptr;   // end of the last upload from h
    Staging() = default;
    Staging(const Staging &) = delete;
    Staging &operator=(const Staging &) = delete;
    ~Staging()
    {
        if (copied) cudaEventDestroy(copied);
    }
    // n words; fill(h) writes them and may refuse the call (its status is returned before anything is enqueued)
    template <typename Fill>
    int upload(size_t n, cudaStream_t stream, Fill &&fill)
    {
        if (!copied) CU_TRY(cudaEventCreateWithFlags(&copied, cudaEventDisableTiming));
        int e;
        if ((e = d.reserve(n, 4096, stream)) || (e = h.reserve(n, 4096, stream))) return e;
        CU_TRY(cudaEventSynchronize(copied));
        if ((e = fill(h.get()))) return e;
        CU_TRY(cudaMemcpyAsync(d.get(), h.get(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        CU_TRY(cudaEventRecord(copied, stream));
        return PFAC_OK;
    }
};

// Everything one in-flight scan needs besides the tables: control block, result block, tile
// directory and the arrival-order scratch.  One per user of a stream (the context's own slot for
// pfac_scan_device, one per pipeline stage for pfac_scan_host).
struct Slot {
    Buf<Ctrl> d_ctrl;
    Buf<Result> d_result;
    Buf<Result, true> h_result;
    // [2][kMaxParts] matches per tile range (walks -> ordering pass).  Two buffers, alternating per scan:
    // the walks of a scan add to one while its detector zeroes the other for the next scan (a buffer
    // zeroed at the start of the scan that uses it would race with the first walks)
    Buf<unsigned long long> d_partial;
    unsigned flip = 0;
    Buf<unsigned int> d_tile_cnt, d_tile_nc;
    Buf<unsigned long long> d_tile_src;
    Buf<uint2> d_scratch;
    bool dirty = false;       // a launch sequence failed half way: the control block is reset before the next scan
    // per-CTA counts of the stable expansions (pfac_compact.cuh: the split and verify passes), compact_grid + 1
    Buf<unsigned long long> d_blk;
    // batch scans (pfac_batch.cuh): raw records of the packed buffer and the global positions of the kept ones,
    // the document offsets
    Buf<uint2> d_raw;
    Buf<uint32_t> d_kpos;
    Staging doc;
    // caseless sets: the folded copy of caller-owned input (pfac_scan_device, pfac_scan_batch_device) at the
    // input's 16-byte phase; grows to the largest input scanned and is held until pfac_ctx_destroy.  Mixed sets
    // fold every input here, the library's own buffers included
    Buf<uint8_t> d_fold;
    // mixed sets (pfac_rules.cuh): the detector's records (owner ids), max(cap, 4096) of them
    Buf<uint2> d_pre;
};

struct Stage {   // one pipeline stage of pfac_scan_host
    cudaStream_t stream = nullptr;
    Buf<uint8_t> d_in;
    Buf<pfac_match> d_out;
    Slot slot;
    cudaEvent_t done = nullptr;
    ~Stage()
    {
        if (done) cudaEventDestroy(done);
        if (stream) cudaStreamDestroy(stream);
    }
};

// What a call enqueued: the counters of pfac_ctx_last_scan_info
struct Counters {
    uint64_t launches = 0, tiles = 0, ctas = 0, h2d = 0, d2h = 0, chunks = 1;
};

}  // namespace

struct pfac_ctx {
    int device = 0;
    int sm_count = 0;
    int n_streams = 1;
    size_t chunk_bytes = 0;
    // tables (device): canonical s0Table, r, {HT, val}, idmap + the detector's shared-memory image
    Buf<int32_t> d_r, d_idmap, d_s0;
    Buf<int2> d_htval;
    Buf<int4> d_step;       // {HT, val, r[row of val]}: the candidate walks' one-load layout (PHF width >= 256)
    Buf<int2> d_s0r;        // {s0Table[b], r[row of it]}
    Buf<uint8_t> d_patdir;  // pattern directory of the candidate walks (pfac_derive.h PatDir); empty: none
    Buf<uint8_t> d_image;
    Buf<uint8_t> d_gimage;  // mode 2: T1 | Tm | Tm2 | T3 in global memory
    Buf<uint8_t> d_wcache;  // walk cache of the dense-match kernel (pfac_derive.h)
    size_t dense_smem = 0;
    bool dense_first = false;      // no detector: the dense-match kernel walks every tile (sets with patterns <= 3 bytes)
    bool caseless = false;         // PFAC_PATTERNS_CASELESS: every scan folds its input first (pfac_fold.cuh)
    // PFAC_PATTERNS_CASE_RULES: the verify tables (pfac_rules.cuh); mixed: every scan folds out of place and ends
    // with the verify pass
    bool mixed = false;
    Buf<int2> d_vgrp;
    Buf<int4> d_vmem;
    Buf<uint8_t> d_vpool;
    uint32_t v_ids = 0;
    uint32_t max_group = 0;
    // batch scans: pattern length of every id; batch_rc != PFAC_OK: the set does not support them (batch_why)
    Buf<int32_t> d_patlen;
    uint32_t n_ids = 0;
    int batch_rc = PFAC_OK;
    std::string batch_why;
    Derived dv;   // image layout and hash parameters (the image bytes are dropped after the upload)
    uint32_t image_bytes = 0;
    int32_t max_pat_len = 0;
    uint32_t halo = 16;
    uint32_t n_stages = 0;
    size_t smem_bytes = 0;
    // the per-context part of every scan's kernel parameters (tables, image layout, walk cache); launch_scan
    // copies them and sets the per-scan fields
    ScanParams scan;
    DenseParams dense;
    // pfac_scan_device: own stream and slot
    cudaStream_t own_stream = nullptr;
    Slot own;                          // working set of pfac_scan_device[_sync] and pfac_scan_batch_device[_sync]
    cudaEvent_t own_done = nullptr;    // end of the last device scan; a call on another stream waits for it
    cudaStream_t own_last = nullptr;
    bool own_used = false;
    std::unique_ptr<Stage[]> stages;   // [n_streams], set up by the first pfac_scan_host that uses them
    uint64_t info[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // optional CUDA-event timing of the detector kernel alone (bench.py's roofline leg)
    bool timing = false;
    std::vector<cudaEvent_t> ev;   // pairs (before, after), used as a ring
    size_t ev_next = 0, ev_count = 0;
    uint32_t debug = 0;   // PFAC_DEBUG env (timing experiments only)
    bool use_pdl = true;  // PFAC_NO_PDL=1: plain stream-ordered launches (timing experiments only)
    std::mutex mu;

    size_t table_bytes() const
    {
        return d_r.bytes() + d_idmap.bytes() + d_s0.bytes() + d_htval.bytes() + d_step.bytes() + d_s0r.bytes() +
               d_patdir.bytes() + d_image.bytes() + d_gimage.bytes() + d_wcache.bytes() + d_patlen.bytes() +
               d_vgrp.bytes() + d_vmem.bytes() + d_vpool.bytes();
    }
};

// A set of flows for the streaming scan (pfac_flows.cuh): per flow the carried tail on the device and the bytes
// consumed on the host; the packed buffer and the per-chunk arrays of a call.  mu serialises the calls on it.
struct pfac_flows {
    pfac_ctx *ctx = nullptr;
    uint32_t n_flows = 0;
    uint32_t keep = 0;                // M - 1: bytes carried per flow
    uint32_t stride = 0;              // tail row: keep rounded up to 16
    Buf<uint8_t> d_tails;             // n_flows rows
    std::vector<uint64_t> pos;        // P_f
    Buf<uint8_t> d_packed;
    Staging stage;                    // doc[n + 1] | tail[n] | flow[n] | src[n]
    std::vector<uint32_t> seen;       // per flow: the last call that named it (duplicate flow ids)
    uint32_t call = 0;
    mutable std::mutex mu;
};

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// The detector kernels: mode 2 (global tables), mode 1 (T1 + T2), and mode 0 (pfac_scan2_kernel<HAS_SHORT, HAS_SC,
// W3>) with patterns of <= 3 bytes, then with or without patterns of 4 bytes (ShortC) and the third window.
using DetectorKernel = void (*)(ScanParams);
const DetectorKernel kDetectors[7] = {
    pfac_scan_kernel<2>,
    pfac_scan_kernel<1>,
    pfac_scan2_kernel<true, true, false>,
    pfac_scan2_kernel<false, true, true>,
    pfac_scan2_kernel<false, true, false>,
    pfac_scan2_kernel<false, false, true>,
    pfac_scan2_kernel<false, false, false>,
};

// The detector kernel a context's derived tables select (unless the dense-match kernel runs alone: dense_first)
DetectorKernel detector_kernel(const Derived &d)
{
    if (d.mode == 2) return kDetectors[0];
    if (d.mode == 1) return kDetectors[1];
    if (d.has_short) return kDetectors[2];
    return kDetectors[3 + (d.has_shortc ? 0 : 2) + (d.has_w3 ? 0 : 1)];
}

// Every kernel of a scan is a programmatic dependent launch: its CTAs are set up (and the detector's filter
// image is on its way into shared memory) while the kernel before it -- the ordering pass of the previous
// scan on this stream, for the detector -- still runs; each kernel waits (griddepcontrol.wait) before it
// touches anything an earlier kernel may write.
cudaLaunchConfig_t launch_config(const pfac_ctx *ctx, cudaStream_t stream, uint32_t grid, uint32_t block, size_t smem)
{
    static cudaLaunchAttribute pdl = [] {
        cudaLaunchAttribute a = {};
        a.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        a.val.programmaticStreamSerializationAllowed = 1;
        return a;
    }();
    cudaLaunchConfig_t lc = {};
    lc.stream = stream;
    lc.attrs = &pdl;
    lc.numAttrs = ctx->use_pdl ? 1 : 0;
    lc.gridDim = dim3(grid);
    lc.blockDim = dim3(block);
    lc.dynamicSmemBytes = smem;
    return lc;
}

// The device watchdog, then the records against the capacity: *count = r.count unless the watchdog tripped.
int check_result(const Result &r, uint64_t cap, uint64_t *count)
{
    if (r.error_flag) return set_error(PFAC_ERR_INTERNAL, "device watchdog tripped (code %u)", r.error_flag);
    *count = r.count;
    if (r.count > cap)
        return set_error(PFAC_ERR_OUTPUT_FULL, "%llu matches exceed the capacity of %llu records",
                         (unsigned long long)r.count, (unsigned long long)cap);
    return PFAC_OK;
}

void set_info(pfac_ctx *ctx, const Counters &c)
{
    const uint64_t v[8] = {c.launches, c.tiles, c.ctas, ctx->smem_bytes, c.h2d, c.d2h, c.chunks, 0};
    memcpy(ctx->info, v, sizeof v);
}

// CTAs of the count and write kernels of a stable expansion (pfac_compact.cuh)
uint32_t compact_grid(const pfac_ctx *ctx) { return 2u * (uint32_t)ctx->sm_count; }

int slot_init(const pfac_ctx *ctx, Slot &s)
{
    if (s.h_result.get()) return PFAC_OK;
    int e;
    if ((e = s.d_ctrl.alloc(1, true)) || (e = s.d_result.alloc(1)) || (e = s.d_partial.alloc(2 * kMaxParts, true)) ||
        (e = s.d_blk.alloc(compact_grid(ctx) + 1)) || (e = s.h_result.alloc(1)))
        return e;
    return PFAC_OK;
}

// Enqueue a stable expansion (pfac_compact.cuh): its count kernel, then its write kernel, over the slot's per-CTA
// counts.  The passes of one call (a mixed batch's verify and split passes) share that buffer: a count kernel writes
// it only after griddepcontrol.wait, when the write kernel before it has finished reading it.
template <typename P>
int launch_compact(pfac_ctx *ctx, Slot &slot, void (*count)(P), void (*write)(P), P p, cudaStream_t stream, Counters &n)
{
    p.blk = slot.d_blk.get();
    const cudaLaunchConfig_t lc = launch_config(ctx, stream, compact_grid(ctx), kCompactThreads, 0);
    CU_TRY(cudaLaunchKernelEx(&lc, count, p));
    CU_TRY(cudaLaunchKernelEx(&lc, write, p));
    n.launches += 2;
    return PFAC_OK;
}

// Enqueue one scan (scan kernel + ordering pass) on `stream`.  On completion slot.d_result holds
// {count, error}; d_count (optional, device) receives the count as well.  n: tiles and CTAs, and the launches,
// added up as they are enqueued.
// own_input: d_in is the library's own buffer (a host scan's stage, a flow call's packed buffer), which a caseless
// set folds in place; the caller's input is folded into slot.d_fold instead and never written.  A mixed set folds
// every input into slot.d_fold (the verify pass reads the original bytes) and scans into slot.d_pre; the verify
// pass then writes d_out, d_count and slot.d_result.
int launch_scan(pfac_ctx *ctx, Slot &slot, const void *d_in, uint64_t n_starts, uint64_t n_valid, uint64_t base_pos,
                uint32_t pos_bias, void *d_out, uint64_t cap, void *d_count, cudaStream_t stream, Counters &n,
                bool own_input)
{
    if (n_valid < n_starts) return set_error(PFAC_ERR_ARG, "n_valid < n_starts");
    const uint64_t useful = n_starts + (uint64_t)(ctx->max_pat_len > 0 ? ctx->max_pat_len - 1 : 0);
    if (n_valid > useful) n_valid = useful;
    const uint32_t mis = (uint32_t)((uintptr_t)d_in & 15u);
    if (n_valid + mis + (uint64_t)kTile + 4096 >= (1ull << 32))
        return set_error(PFAC_ERR_LIMIT, "one scan call covers less than 4 GiB; split the input");
    int e = slot_init(ctx, slot);
    if (e) return e;
    if (n_starts == 0 || ctx->max_pat_len == 0) {
        CU_TRY(cudaMemsetAsync(slot.d_result.get(), 0, sizeof(Result), stream));
        if (d_count) CU_TRY(cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), stream));
        return PFAC_OK;
    }
    if (slot.dirty) {   // a previous launch sequence failed between the kernels: start from a clean control block
        CU_TRY(cudaMemsetAsync(slot.d_ctrl.get(), 0, sizeof(Ctrl), stream));
        CU_TRY(cudaMemsetAsync(slot.d_partial.get(), 0, slot.d_partial.bytes(), stream));
        slot.dirty = false;
    }
    struct DirtyOnError {   // set back to false on the success path
        Slot &s;
        bool armed = true;
        ~DirtyOnError() { if (armed) s.dirty = true; }
    } guard{slot};
    if (ctx->n_stages < (uint32_t)min_stages((int)ctx->dv.mode))
        return set_error(PFAC_ERR_INTERNAL, "input ring of %u stages is too shallow for the slot scheme", ctx->n_stages);
    const bool mixed = ctx->mixed;
    const uint8_t *orig_al = (const uint8_t *)d_in - mis;
    if (ctx->caseless || mixed) {   // the fold of the bytes the scan reads, at the input's phase: mis and every bound stay
        uint8_t *out_al = const_cast<uint8_t *>((const uint8_t *)d_in - mis);
        if (!own_input || mixed) {
            if ((e = slot.d_fold.reserve((size_t)(mis + n_valid), 0, stream))) return e;
            out_al = slot.d_fold.get();
        }
        const uint64_t words = (mis + n_valid + 15) / 16;
        const uint32_t fg = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((words + kFoldThreads * kFoldUnroll - 1) /
                                                                                   (kFoldThreads * kFoldUnroll),
                                                                               4ull * (uint64_t)ctx->sm_count));
        const cudaLaunchConfig_t fl = launch_config(ctx, stream, fg, kFoldThreads, 0);
        CU_TRY(cudaLaunchKernelEx(&fl, pfac_fold_kernel, (const uint8_t *)d_in - mis, out_al, (unsigned long long)mis,
                                  (unsigned long long)(mis + n_valid)));
        d_in = out_al + mis;
        n.launches += 1;
    }
    ScanParams p = ctx->scan;
    p.in_al = (const uint8_t *)d_in - mis;
    p.mis = mis;
    p.a_start_end = (uint32_t)(mis + n_starts);
    p.a_valid_end = (uint32_t)(mis + n_valid);
    p.n_tiles = (uint32_t)(((uint64_t)p.a_start_end + kTile - 1) / kTile);
    p.base_pos = base_pos;
    // tile directory and scratch (epoch 0 in tile_src = never published: DIRECT dense scans)
    if ((e = slot.d_tile_cnt.reserve(p.n_tiles, 1024, stream)) || (e = slot.d_tile_src.reserve(p.n_tiles, 1024, stream, true)) ||
        (e = slot.d_tile_nc.reserve(p.n_tiles, 1024, stream)) ||
        (e = slot.d_scratch.reserve((size_t)std::max<uint64_t>(cap, 4096), 4096, stream)))
        return e;
    p.tile_cnt = slot.d_tile_cnt.get();
    p.tile_nc = slot.d_tile_nc.get();
    unsigned long long *partial_now = slot.d_partial.get() + (slot.flip & 1u) * kMaxParts;
    p.partial = partial_now;
    p.partial_next = slot.d_partial.get() + ((slot.flip + 1u) & 1u) * kMaxParts;
    p.ctrl = slot.d_ctrl.get();
    // a mixed set's scan writes the owners' records to slot.d_pre; the verify pass writes the caller's
    void *scan_out = d_out, *scan_count = d_count;
    uint64_t scan_cap = cap;
    if (mixed) {
        const size_t want = (size_t)std::max<uint64_t>(cap, 4096);
        if ((e = slot.d_pre.reserve(want, want, stream))) return e;
        scan_out = slot.d_pre.get();
        scan_cap = slot.d_pre.cap();
        scan_count = nullptr;
    }
    const uint32_t grid = (uint32_t)std::min<uint64_t>(p.n_tiles, (uint64_t)ctx->sm_count);
    // tile ranges of the ordering pass: many small ones, so that dense outputs (every tile a long run
    // of records) are moved by the whole GPU
    const uint32_t fgrid = (uint32_t)std::min<uint64_t>((p.n_tiles + 7) / 8, (uint64_t)kMaxParts);
    const uint32_t tiles_per_part = (p.n_tiles + fgrid - 1) / fgrid;
    EmitParams &ep = p.emit;
    ep.in_al = p.in_al;
    ep.mis = p.mis;
    ep.a_start_end = p.a_start_end;
    ep.a_valid_end = p.a_valid_end;
    ep.base_pos = base_pos;
    ep.pos_bias = pos_bias;
    ep.scratch = slot.d_scratch.get();
    ep.scratch_cap = slot.d_scratch.cap();
    ep.tile_cnt = slot.d_tile_cnt.get();
    ep.tile_src = slot.d_tile_src.get();
    ep.tile_nc = slot.d_tile_nc.get();
    ep.n_tiles = p.n_tiles;
    ep.tiles_per_part = tiles_per_part;
    ep.partial = partial_now;
    ep.ctrl = slot.d_ctrl.get();

    p.ticket_batch = std::max<uint32_t>(1u, std::min<uint32_t>((uint32_t)kTicketBatch, p.n_tiles / (4u * grid)));
    cudaEvent_t ev_after = nullptr;
    if (ctx->timing && !ctx->ev.empty()) {
        const size_t slot_i = ctx->ev_next;
        ctx->ev_next = (ctx->ev_next + 2) % ctx->ev.size();
        ctx->ev_count = std::min(ctx->ev_count + 1, ctx->ev.size() / 2);
        CU_TRY(cudaEventRecord(ctx->ev[slot_i], stream));
        ev_after = ctx->ev[slot_i + 1];
    }
    // Pattern sets with patterns of <= 3 bytes (the reference's own fixtures: a dictionary, "a/aa/aaa")
    // match at a large share of the start positions of natural text: no filter pays off, the dense-match
    // kernel walks every tile straight away.
    const bool dense_first = ctx->dense_first;
    if (!dense_first) {
        const cudaLaunchConfig_t lc = launch_config(ctx, stream, grid, kThreads, ctx->smem_bytes);
        CU_TRY(cudaLaunchKernelEx(&lc, detector_kernel(ctx->dv), p));
        if (ev_after) CU_TRY(cudaEventRecord(ev_after, stream));
        n.launches += 1;
    }

    // the tiles the detector handed over whole (dense matches); returns at once when there are none
    DenseParams dp = ctx->dense;
    dp.e = ep;
    dp.n_dense = &slot.d_ctrl.get()->n_dense;
    const cudaLaunchConfig_t dl = launch_config(ctx, stream, grid, kDenseThreads, ctx->dense_smem);
    if (dense_first) {   // the dense-match kernel is the whole scan: records go straight to the caller's buffer
        dp.out = (uint2 *)scan_out;
        dp.cap = scan_cap;
        dp.prefix = slot.d_tile_src.get();
        dp.epoch = slot.flip % 0xFFFFFEu + 1u;
        dp.result = slot.d_result.get();
        dp.count_out = (unsigned long long *)scan_count;
        CU_TRY(cudaLaunchKernelEx(&dl, pfac_dense_kernel<true>, dp));
        if (ev_after) CU_TRY(cudaEventRecord(ev_after, stream));
        n.launches += 1;
    } else {   // dense-match pass and ordering pass
        CU_TRY(cudaLaunchKernelEx(&dl, pfac_dense_kernel<false>, dp));
        FinalizeParams f;
        f.tile_cnt = slot.d_tile_cnt.get();
        f.tile_src = slot.d_tile_src.get();
        f.scratch = slot.d_scratch.get();
        f.scratch_cap = slot.d_scratch.cap();
        f.out = (uint2 *)scan_out;
        f.cap = scan_cap;
        f.n_tiles = p.n_tiles;
        f.tiles_per_part = tiles_per_part;
        f.partial = partial_now;
        f.ctrl = slot.d_ctrl.get();
        f.result = slot.d_result.get();
        f.count_out = (unsigned long long *)scan_count;
        f.debug = ctx->debug;
        f.trace_ctas = grid;
        const cudaLaunchConfig_t fl = launch_config(ctx, stream, fgrid, kFinThreads, 0);
        CU_TRY(cudaLaunchKernelEx(&fl, pfac_finalize_kernel, f));
        n.launches += 2;
    }
    if (mixed) {   // the verify pass: owners' records -> the members' records that match the original bytes
        RulesParams rp;
        rp.pre = slot.d_pre.get();
        rp.pre_cap = slot.d_pre.cap();
        rp.in_al = orig_al;
        rp.mis = mis;
        rp.pos_bias = pos_bias;
        rp.grp = ctx->d_vgrp.get();
        rp.n_ids = ctx->v_ids;
        rp.mem = ctx->d_vmem.get();
        rp.pool = ctx->d_vpool.get();
        rp.max_group = ctx->max_group;
        rp.out = (uint2 *)d_out;
        rp.cap = cap;
        rp.result = slot.d_result.get();
        rp.count_out = (unsigned long long *)d_count;
        if ((e = launch_compact(ctx, slot, pfac_rules_count_kernel, pfac_rules_write_kernel, rp, stream, n))) return e;
    }
    n.tiles = p.n_tiles;
    n.ctas = grid;
    slot.flip++;
    guard.armed = false;
    return PFAC_OK;
}

// The slot's buffers of a batch or flow call: raw records and kept positions for max(cap, 4096) records
int split_prepare(pfac_ctx *ctx, Slot &slot, uint64_t cap, cudaStream_t stream)
{
    int e = slot_init(ctx, slot);
    if (e) return e;
    const size_t want = (size_t)std::max<uint64_t>(cap, 4096);
    if ((e = slot.d_raw.reserve(want, want, stream)) || (e = slot.d_kpos.reserve(want, want, stream))) return e;
    return PFAC_OK;
}

// Enqueue the split pass (pfac_batch.cuh) over the raw records of the packed scan: n_docs documents at the device
// offsets doc[n_docs + 1]; CARRY: the first tail[d] bytes of document d are carried (device, n_docs).
template <bool CARRY>
int launch_split(pfac_ctx *ctx, Slot &slot, const uint32_t *doc, const uint32_t *tail, uint32_t n_docs,
                 void *d_out, uint64_t cap, void *d_doc_first, void *d_count, cudaStream_t stream, Counters &n)
{
    BatchParams bp;
    memset(&bp, 0, sizeof bp);
    bp.raw = slot.d_raw.get();
    bp.raw_cap = slot.d_raw.cap();
    bp.doc = doc;
    bp.n_docs = n_docs;
    bp.len = ctx->d_patlen.get();
    bp.n_ids = ctx->n_ids;
    bp.out = (uint2 *)d_out;
    bp.cap = cap;
    bp.kpos = slot.d_kpos.get();
    bp.doc_first = (unsigned long long *)d_doc_first;
    bp.result = slot.d_result.get();
    bp.count_out = (unsigned long long *)d_count;
    bp.tail = tail;
    int e = launch_compact(ctx, slot, pfac_batch_count_kernel<CARRY>, pfac_batch_split_kernel<CARRY>, bp, stream, n);
    if (e) return e;
    const size_t n_off = (size_t)n_docs + 1;
    const cudaLaunchConfig_t dl = launch_config(
        ctx, stream, (uint32_t)std::min<uint64_t>((n_off + kCompactThreads - 1) / kCompactThreads, compact_grid(ctx)),
        kCompactThreads, 0);
    CU_TRY(cudaLaunchKernelEx(&dl, pfac_batch_docs_kernel, bp));
    n.launches += 1;
    return PFAC_OK;
}

// Enqueue a batch scan on `stream` (pfac_batch.cuh): the documents' offsets are uploaded, the packed buffer is
// scanned into the slot's raw-record buffer, the split pass writes the caller's records, d_doc_first and
// d_count.  On completion slot.d_result holds {count, error}.
int launch_batch(pfac_ctx *ctx, Slot &slot, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                 void *d_out, uint64_t cap, void *d_doc_first, void *d_count, cudaStream_t stream, Counters &n)
{
    if (ctx->batch_rc != PFAC_OK) return set_error(ctx->batch_rc, "%s", ctx->batch_why.c_str());
    if (n_docs == 0xFFFFFFFFu) return set_error(PFAC_ERR_LIMIT, "a batch holds fewer than 2^32 - 1 documents");
    if (doc_offsets[0] != 0)
        return set_error(PFAC_ERR_ARG, "doc_offsets[0] = %llu: the first document starts at 0", (unsigned long long)doc_offsets[0]);
    const uint64_t total = doc_offsets[n_docs];
    if (total >= (1ull << 32)) return set_error(PFAC_ERR_LIMIT, "one batch covers less than 4 GiB; split the input");
    if (!d_in && total) return set_error(PFAC_ERR_ARG, "null input of %llu bytes", (unsigned long long)total);
    int e = split_prepare(ctx, slot, cap, stream);
    if (e) return e;
    // the offsets, checked on the way (32 bits suffice: total < 4 GiB)
    const size_t n_off = (size_t)n_docs + 1;
    e = slot.doc.upload(n_off, stream, [&](uint32_t *h) {
        uint64_t prev = 0;
        bool decreasing = false;
        for (size_t i = 0; i < n_off; i++) {
            const uint64_t v = doc_offsets[i];
            decreasing |= v < prev;
            prev = v;
            h[i] = (uint32_t)v;
        }
        return decreasing ? set_error(PFAC_ERR_ARG, "doc_offsets decrease") : PFAC_OK;
    });
    if (e) return e;

    e = launch_scan(ctx, slot, d_in, total, total, 0, 0u, slot.d_raw.get(), slot.d_raw.cap(), nullptr, stream, n, false);
    if (e) return e;
    e = launch_split<false>(ctx, slot, slot.doc.d.get(), nullptr, n_docs, d_out, cap, d_doc_first, d_count, stream, n);
    if (e) return e;
    n.h2d = n_off * sizeof(uint32_t);
    return PFAC_OK;
}

// Enqueue a streaming call on `stream` (pfac_flows.cuh): per-chunk arrays uploaded, tails and chunks packed, the
// packed buffer scanned, the split pass with the carry-aware keep rule, the new tails written if the records fit.
// Every refusal comes before anything is enqueued; base[i] = P_f - t_f of chunk i.
int launch_flows(pfac_flows *f, Slot &slot, const void *d_in, const uint64_t *chunk_offsets, const uint32_t *flow_ids,
                 uint32_t n_chunks, void *d_out, uint64_t cap, void *d_chunk_first, uint64_t *base, cudaStream_t stream,
                 Counters &n)
{
    pfac_ctx *ctx = f->ctx;
    if (n_chunks == 0xFFFFFFFFu) return set_error(PFAC_ERR_LIMIT, "a call holds fewer than 2^32 - 1 chunks");
    if (chunk_offsets[0] != 0)
        return set_error(PFAC_ERR_ARG, "chunk_offsets[0] = %llu: the first chunk starts at 0", (unsigned long long)chunk_offsets[0]);
    if (++f->call == 0) {   // (the stamps wrapped: forget them all)
        std::fill(f->seen.begin(), f->seen.end(), 0u);
        f->call = 1;
    }
    uint64_t packed = 0;
    for (uint32_t i = 0; i < n_chunks; i++) {
        const uint32_t fl = flow_ids[i];
        if (fl >= f->n_flows) return set_error(PFAC_ERR_ARG, "flow id %u of chunk %u: the set has %u flows", fl, i, f->n_flows);
        if (f->seen[fl] == f->call) return set_error(PFAC_ERR_ARG, "flow %u takes two chunks in one call", fl);
        f->seen[fl] = f->call;
        if (chunk_offsets[i + 1] < chunk_offsets[i]) return set_error(PFAC_ERR_ARG, "chunk_offsets decrease");
        packed += std::min<uint64_t>(f->keep, f->pos[fl]) + (chunk_offsets[i + 1] - chunk_offsets[i]);
    }
    const uint64_t total_in = chunk_offsets[n_chunks];
    if (total_in >= (1ull << 32) || packed + (uint64_t)kTile + 4096 >= (1ull << 32))
        return set_error(PFAC_ERR_LIMIT, "one call covers less than 4 GiB of chunks and carried tails; split the input");
    if (!d_in && total_in) return set_error(PFAC_ERR_ARG, "null input of %llu bytes", (unsigned long long)total_in);
    int e = split_prepare(ctx, slot, cap, stream);
    if (e || (e = f->d_packed.reserve((size_t)packed + 48, std::max<size_t>((size_t)packed + 48, 1 << 20), stream))) return e;
    const size_t nc = n_chunks;
    e = f->stage.upload(4 * nc + 1, stream, [&](uint32_t *h) {
        uint32_t *doc = h, *tail = h + nc + 1, *flow = tail + nc, *src = flow + nc;
        doc[0] = 0;
        for (size_t i = 0; i < nc; i++) {
            const uint32_t fl = flow_ids[i];
            const uint64_t t = std::min<uint64_t>(f->keep, f->pos[fl]);
            base[i] = f->pos[fl] - t;
            doc[i + 1] = doc[i] + (uint32_t)(t + chunk_offsets[i + 1] - chunk_offsets[i]);
            tail[i] = (uint32_t)t;
            flow[i] = fl;
            src[i] = (uint32_t)chunk_offsets[i];
        }
        return PFAC_OK;
    });
    if (e) return e;
    const uint32_t *d_stage = f->stage.d.get();
    FlowParams fp;
    memset(&fp, 0, sizeof fp);
    fp.in = (const uint8_t *)d_in;
    fp.doc = d_stage;
    fp.tail = d_stage + nc + 1;
    fp.flow = fp.tail + nc;
    fp.src = fp.flow + nc;
    fp.n = n_chunks;
    fp.total = (uint32_t)packed;
    fp.tails = f->d_tails.get();
    fp.stride = f->stride;
    fp.keep = f->keep;
    fp.packed = f->d_packed.get();
    fp.result = slot.d_result.get();
    fp.cap = cap;
    const uint32_t pgrid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((packed + 4095) / 4096, 16ull * (uint64_t)ctx->sm_count));
    const cudaLaunchConfig_t pl = launch_config(ctx, stream, pgrid, kFlowThreads, 0);
    CU_TRY(cudaLaunchKernelEx(&pl, pfac_flow_pack_kernel, fp));
    n.launches = 1;
    Counters k;
    e = launch_scan(ctx, slot, fp.packed, packed, packed, 0, 0u, slot.d_raw.get(), slot.d_raw.cap(), nullptr, stream, k, true);
    if (e) return e;
    n.launches += k.launches;
    n.tiles = k.tiles;
    n.ctas = k.ctas;
    e = launch_split<true>(ctx, slot, fp.doc, fp.tail, n_chunks, d_out, cap, d_chunk_first, nullptr, stream, n);
    if (e) return e;
    const uint32_t tgrid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((nc + 7) / 8, 2ull * (uint64_t)ctx->sm_count));
    const cudaLaunchConfig_t tl = launch_config(ctx, stream, tgrid, kFlowThreads, 0);
    CU_TRY(cudaLaunchKernelEx(&tl, pfac_flow_tail_kernel, fp));
    n.launches += 1;
    n.h2d = (4 * nc + 1) * sizeof(uint32_t);
    return PFAC_OK;
}

// The entry points that scan into the context's own slot.  `launch(stream, counters)` enqueues the scan.
// With `count` (the _sync forms) the Result block is read back and the stream synchronised, then the records
// are checked against `cap`.  Device scans of one context share the slot: a scan enqueued on another stream
// than the one before it is ordered after it (own_done).
template <typename Launch>
int run_own(pfac_ctx *ctx, void *stream, uint64_t cap, uint64_t *count, Launch &&launch)
{
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    const cudaStream_t st = stream ? (cudaStream_t)stream : ctx->own_stream;
    if (ctx->own_used && ctx->own_last != st) CU_TRY(cudaStreamWaitEvent(st, ctx->own_done, 0));
    Counters n;
    int e = launch(st, n);
    if (e) return e;
    Slot &s = ctx->own;
    if (count) CU_TRY(cudaMemcpyAsync(s.h_result.get(), s.d_result.get(), sizeof(Result), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaEventRecord(ctx->own_done, st));
    ctx->own_last = st;
    ctx->own_used = true;
    if (count) CU_TRY(cudaStreamSynchronize(st));
    set_info(ctx, n);
    return count ? check_result(*s.h_result.get(), cap, count) : PFAC_OK;
}

// shared-memory budget: T1 and the per-warp queues are fixed; T3 / Tm2 / T2 shrink until at least
// four ring stages fit
int size_shared_memory(pfac_ctx &ctx, const Partition &P, size_t smem_max)
{
    uint32_t t2_bytes = 32768, t3_bytes = 32768, tm2_bytes = 32768;
    if (const char *v = getenv("PFAC_T2_BYTES")) t2_bytes = (uint32_t)atoi(v);
    if (const char *v = getenv("PFAC_T3_BYTES")) t3_bytes = (uint32_t)atoi(v);
    if (const char *v = getenv("PFAC_TM2_BYTES")) tm2_bytes = (uint32_t)atoi(v);
    bool widened = false;
    while (true) {
        derive_tables(P, t2_bytes, t3_bytes, tm2_bytes, ctx.dv);
        if (ctx.dv.mode == 2 && !widened && !getenv("PFAC_T2_BYTES")) {
            // global mode: T2 is stage 1 and the only shared-memory table -- give it all the room
            widened = true;
            t2_bytes = 131072;
            continue;
        }
        ctx.image_bytes = (uint32_t)ctx.dv.image.size();
        const size_t fixed = scan_smem_bytes(ctx.image_bytes, ctx.halo, 0, ctx.dv.mode);
        const size_t stride = scan_buf_stride(ctx.halo);
        const size_t fit = smem_max > fixed ? (smem_max - fixed) / stride : 0;
        const bool minimal = t2_bytes < 2048 && (ctx.dv.mode == 2 || (t3_bytes < 2048 && tm2_bytes < 2048));
        const size_t need = (size_t)min_stages((int)ctx.dv.mode);   // 2 (shared-memory mode) or 4 (global mode)
        // mode 0 wants a deep ring (bytes in flight hide the HBM latency): T3 gives way down to 16 KiB
        const bool deepen = ctx.dv.mode == 0 && fit < 9 && t3_bytes > 16384 && !getenv("PFAC_T3_BYTES");
        if (!deepen && (fit >= std::max<size_t>(3, need) || (fit >= need && minimal))) {
            ctx.n_stages = (uint32_t)std::min<size_t>(fit, kMaxStages);
            if (const char *v = getenv("PFAC_RING_STAGES"))   // tests: a ring as shallow as the slot scheme allows
                ctx.n_stages = (uint32_t)std::max<size_t>(need, std::min<size_t>(ctx.n_stages, (size_t)atoi(v)));
            ctx.smem_bytes = scan_smem_bytes(ctx.image_bytes, ctx.halo, ctx.n_stages, ctx.dv.mode);
            return PFAC_OK;
        }
        if (minimal)
            return set_error(PFAC_ERR_CUDA, "scan kernel needs more than the %zu B of shared memory the device offers",
                             smem_max);
        // halve the largest section that is actually in the image
        if (ctx.dv.mode == 2) {
            t2_bytes /= 2;
        } else if (ctx.dv.has_t3) {
            if (t3_bytes > 8192) t3_bytes /= 2;          // T3 first: it only gets a little less selective
            else if (tm2_bytes >= 2048) tm2_bytes /= 2;  // then level 2 (all or nothing per size)
            else t3_bytes /= 2;
        } else {
            t3_bytes = tm2_bytes = 0;
            t2_bytes /= 2;
        }
    }
}

// canonical arrays -> device, unchanged: s0Table, r, {HT, val} interleaved, idmap; + the detector images, the
// walks' one-load layout and the pattern directory.  Fills the per-context part of ctx.scan.
int upload_tables(pfac_ctx &ctx, const Partition &P)
{
    const size_t n_ht = std::max<size_t>((size_t)P.ht_size, 1);
    std::vector<int32_t> r(P.r), idmap(std::max<size_t>((size_t)P.n_final, 1), 0), s0(256, -1);
    r.resize(std::max<size_t>(P.r.size(), 1), -1);
    std::copy_n(P.idmap.begin(), (size_t)P.n_final, idmap.begin());
    if (!P.s0.empty()) std::copy_n(P.s0.begin(), 256, s0.begin());
    std::vector<int2> htval(n_ht, make_int2(-1, -1));
    for (int32_t i = 0; i < P.ht_size; i++) htval[(size_t)i] = make_int2(P.HT[(size_t)i], P.val[(size_t)i]);
    int e;
    if ((e = ctx.d_r.upload(r)) || (e = ctx.d_htval.upload(htval)) || (e = ctx.d_idmap.upload(idmap)) ||
        (e = ctx.d_s0.upload(s0)) || (e = ctx.d_image.upload(ctx.dv.image)))
        return e;
    const int width_bit = width_bits(P.width);
    if (width_bit >= 8 && !P.r.empty()) {
        // the one-load layout of the candidate walks: the row of a state's transitions depends on the state
        // alone when a row holds at least 256 keys, so every entry can carry its successor's r[] value
        const int sh = width_bit - 8;
        auto r_of = [&](int32_t state) -> int32_t {
            const size_t row = (size_t)state >> sh;
            return state >= 0 && row < P.r.size() ? P.r[row] : -1;
        };
        std::vector<int4> step(n_ht, make_int4(-1, -1, -1, 0));
        for (int32_t i = 0; i < P.ht_size; i++) step[(size_t)i] = make_int4(P.HT[(size_t)i], P.val[(size_t)i], r_of(P.val[(size_t)i]), 0);
        std::vector<int2> s0r(256);
        for (int b = 0; b < 256; b++) s0r[(size_t)b] = make_int2(s0[(size_t)b], r_of(s0[(size_t)b]));
        if ((e = ctx.d_step.upload(step)) || (e = ctx.d_s0r.upload(s0r))) return e;
    }
    PatDir pd;
    if (!getenv("PFAC_NO_PATDIR")) derive_patdir(P, pd);
    if (pd.n_slots && (e = ctx.d_patdir.upload(pd.image))) return e;
    if (!ctx.dv.gimage.empty() && (e = ctx.d_gimage.upload(ctx.dv.gimage))) return e;

    const Derived &d = ctx.dv;
    ScanParams &p = ctx.scan;
    memset(&p, 0, sizeof p);
    p.halo = ctx.halo;
    p.max_pat_len = (uint32_t)ctx.max_pat_len;
    p.use_ref_bound = ctx.max_pat_len > kRefHalo + 1;   // only then can the 4096+512 bound cut a walk
    p.image = reinterpret_cast<const uint4 *>(ctx.d_image.get());
    p.image_bytes = ctx.image_bytes;
    p.off_t2 = d.off_t2;
    p.off_tm = d.off_tm;
    p.off_tm2 = d.off_tm2;
    p.off_t3 = d.off_t3;
    p.t2_shift = d.t2_shift;
    p.has_short = d.has_short;
    p.has_t3 = d.has_t3;
    p.t3_shift = d.t3_shift;
    p.tm_bits = d.tm_bits;
    p.tm2_bits = d.tm2_bits;
    p.off_d1 = d.off_d1;
    p.off_e1 = d.off_e1;
    p.nb1 = d.nb1;
    p.ns1 = d.ns1;
    p.off_d2 = d.off_d2;
    p.off_e2 = d.off_e2;
    p.nb2 = d.nb2;
    p.ns2 = d.ns2;
    p.gimage = ctx.d_gimage.get();
    p.n_stages = ctx.n_stages;
    p.stage_magic = (uint32_t)((1ull << 32) / ctx.n_stages) + 1u;
    p.debug = ctx.debug;
    EmitParams &ep = p.emit;
    ep.max_pat_len = p.max_pat_len;
    ep.use_ref_bound = p.use_ref_bound;
    ep.r = ctx.d_r.get();
    ep.htval = ctx.d_htval.get();
    ep.idmap = ctx.d_idmap.get();
    ep.s0 = ctx.d_s0.get();
    ep.step = ctx.d_step.get();
    ep.s0r = ctx.d_s0r.get();
    if (pd.n_slots) {
        ep.dir = reinterpret_cast<const uint4 *>(ctx.d_patdir.get());
        ep.pool = ctx.d_patdir.get() + pd.off_pool;
        ep.dir_slots = pd.n_slots;
        ep.len_mask = pd.len_mask;
    }
    ep.ht_size = P.ht_size;
    ep.width_bit = width_bit;
    ep.n_final = P.n_final;
    return PFAC_OK;
}

// walk cache of the dense-match kernel: as deep as fits beside its text tile and result arrays.  Fills the
// per-context part of ctx.dense.
int upload_walk_cache(pfac_ctx &ctx, const Partition &P, size_t smem_max)
{
    const size_t fixed = dense_smem_bytes(0, ctx.halo);
    const uint32_t budget = smem_max > fixed + 4096 ? (uint32_t)std::min<size_t>(smem_max - fixed, 128u << 10) : 2048u;
    WalkCache wc;
    derive_walk_cache(P, budget, wc);
    const uint32_t wc_bytes = (uint32_t)((wc.image.size() + 15) & ~(size_t)15);
    wc.image.resize(wc_bytes, 0);
    ctx.dense_smem = dense_smem_bytes(wc_bytes, ctx.halo);
    if (ctx.dense_smem > smem_max)
        return set_error(PFAC_ERR_CUDA, "dense-match kernel needs %zu B of shared memory (patterns too long)", ctx.dense_smem);
    int e = ctx.d_wcache.upload(wc.image);
    if (e) return e;
    DenseParams &d = ctx.dense;
    memset(&d, 0, sizeof d);
    d.wc_image = ctx.d_wcache.get();
    d.wc_bytes = wc_bytes;
    d.wc_depth = wc.depth;
    d.wc_off_d = wc.off_d;
    d.wc_off_e = wc.off_e;
    d.wc_nb = wc.nb;
    d.wc_ns = wc.ns;
    d.halo = ctx.halo;
    return PFAC_OK;
}

// per-pattern case rules: the verify tables of pfac_rules.cuh, indexed by owner id
int upload_case_groups(pfac_ctx &ctx, const Partition &P)
{
    const Partition::CaseGroups &G = P.groups;
    int32_t max_owner = 0;
    for (int32_t o : G.owner) max_owner = std::max(max_owner, o);
    std::vector<int2> grp((size_t)max_owner + 1, make_int2(0, 0));
    for (size_t g = 0; g < G.owner.size(); g++) {
        grp[(size_t)G.owner[g]] = make_int2(G.first[g], G.first[g + 1] - G.first[g]);
        ctx.max_group = std::max<uint32_t>(ctx.max_group, (uint32_t)(G.first[g + 1] - G.first[g]));
    }
    std::vector<int4> mem(std::max<size_t>(G.id.size(), 1), make_int4(0, 0, -1, 0));
    for (size_t m = 0; m < G.id.size(); m++) mem[m] = make_int4(G.id[m], G.len[m], G.off[m], 0);
    std::vector<uint8_t> pool(G.pool);
    pool.resize(std::max<size_t>(pool.size(), 16), 0);
    ctx.v_ids = (uint32_t)grp.size();
    ctx.max_group = std::max<uint32_t>(ctx.max_group, 1u);
    int e;
    if ((e = ctx.d_vgrp.upload(grp)) || (e = ctx.d_vmem.upload(mem)) || (e = ctx.d_vpool.upload(pool))) return e;
    ctx.mixed = true;
    return PFAC_OK;
}

// batch scans need each id's pattern length (a tree-shaped automaton) and results that do not depend on
// where a document lies in the packed buffer (no reference tile bound: patterns of <= 513 bytes)
int upload_pattern_lengths(pfac_ctx &ctx, const Partition &P)
{
    std::vector<int32_t> len;
    if (pattern_lengths(P, len) != PFAC_OK) {
        ctx.batch_rc = PFAC_ERR_ARG;
        ctx.batch_why = pfac_last_error();
    } else if (P.max_len > kRefHalo + 1) {
        ctx.batch_rc = PFAC_ERR_LIMIT;
        ctx.batch_why = "batch scans need patterns of at most 513 bytes (the reference's 4096+512 tile bound "
                        "would make results depend on where a document lies in the batch)";
    } else {
        ctx.n_ids = (uint32_t)len.size();
        len.resize(std::max<size_t>(len.size(), 1), 0);
        return ctx.d_patlen.upload(len);
    }
    return PFAC_OK;
}

}  // namespace

extern "C" {

int pfac_device_count(int *count)
{
    if (!count) return set_error(PFAC_ERR_ARG, "null count");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        return set_error(PFAC_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *count = n;
    return PFAC_OK;
}

int pfac_ctx_create(int device, const pfac_tables *t, int part, int n_streams, size_t chunk_bytes, pfac_ctx **out)
{
    if (!out || !t || part < 0 || part >= (int)t->parts.size() || n_streams < 1 || n_streams > 64)
        return set_error(PFAC_ERR_ARG, "bad arguments to pfac_ctx_create");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return set_error(PFAC_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU path)");
    if (device < 0 || device >= ndev) return set_error(PFAC_ERR_ARG, "device %d out of range (%d devices)", device, ndev);
    DeviceGuard g(device);
    if (!g.ok) return set_error(PFAC_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    const Partition &P = t->parts[(size_t)part];
    // (every early return below releases what was allocated so far)
    std::unique_ptr<pfac_ctx, void (*)(pfac_ctx *)> ctx(new pfac_ctx, pfac_ctx_destroy);
    ctx->device = device;
    ctx->n_streams = n_streams;
    ctx->stages.reset(new Stage[(size_t)n_streams]);
    ctx->chunk_bytes = chunk_bytes ? chunk_bytes : ((size_t)32 << 20);
    ctx->chunk_bytes = (ctx->chunk_bytes + kTile - 1) / kTile * kTile;
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return set_error(PFAC_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only",
                         device, prop.major, prop.minor);
    ctx->sm_count = prop.multiProcessorCount;
    ctx->max_pat_len = P.max_len;
    ctx->halo = (uint32_t)std::max(16, ((P.max_len > 0 ? P.max_len - 1 : 0) + 15) / 16 * 16);
    if (const char *dbg = getenv("PFAC_DEBUG")) ctx->debug = (uint32_t)atoi(dbg);
    if (const char *v = getenv("PFAC_NO_PDL")) ctx->use_pdl = atoi(v) == 0;

    const size_t smem_max = (size_t)prop.sharedMemPerBlockOptin;
    int e;
    if ((e = size_shared_memory(*ctx, P, smem_max)) || (e = upload_tables(*ctx, P)) ||
        (e = upload_walk_cache(*ctx, P, smem_max)) || (e = upload_pattern_lengths(*ctx, P)))
        return e;
    ctx->dense_first = ctx->dv.has_short != 0;
    ctx->caseless = (t->flags & PFAC_PATTERNS_CASELESS) != 0;
    if ((t->flags & PFAC_PATTERNS_CASE_RULES) && (e = upload_case_groups(*ctx, P))) return e;
    if (const char *v = getenv("PFAC_DENSE_FIRST")) ctx->dense_first = atoi(v) != 0;   // experiments: force either path
    ctx->dv.image.clear();
    ctx->dv.image.shrink_to_fit();
    ctx->dv.gimage.clear();
    ctx->dv.gimage.shrink_to_fit();

    // the attribute is per function and device, not per context: always allow the device maximum
    std::vector<const void *> kernels = {(const void *)pfac_dense_kernel<false>, (const void *)pfac_dense_kernel<true>};
    for (DetectorKernel k : kDetectors) kernels.push_back((const void *)k);
    for (const void *k : kernels) CU_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    int bps = 0;
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, detector_kernel(ctx->dv), kThreads, ctx->smem_bytes));
    if (bps < 1) return set_error(PFAC_ERR_CUDA, "scan kernel does not fit on an SM (smem %zu B)", ctx->smem_bytes);

    CU_TRY(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreateWithFlags(&ctx->own_done, cudaEventDisableTiming));
    e = slot_init(ctx.get(), ctx->own);
    if (e) return e;
    *out = ctx.release();
    return PFAC_OK;
}

void pfac_ctx_destroy(pfac_ctx *ctx)
{
    if (!ctx) return;
    DeviceGuard g(ctx->device);
    cudaDeviceSynchronize();
    for (auto e : ctx->ev)
        if (e) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->own_done) cudaEventDestroy(ctx->own_done);
    delete ctx;   // (frees the buffers, slots and stages on the context's device)
}

int pfac_ctx_device(const pfac_ctx *ctx) { return ctx ? ctx->device : -1; }

int pfac_ctx_set_timing(pfac_ctx *ctx, int enable)
{
    if (!ctx) return set_error(PFAC_ERR_ARG, "bad arguments");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    if (enable && ctx->ev.empty()) {
        ctx->ev.resize(512, nullptr);
        for (auto &e : ctx->ev) CU_TRY(cudaEventCreate(&e));
    }
    ctx->timing = enable != 0;
    ctx->ev_next = ctx->ev_count = 0;
    return PFAC_OK;
}

int pfac_ctx_kernel_time(pfac_ctx *ctx, double *ms_total, int *n_launches)
{
    if (!ctx || !ms_total || !n_launches) return set_error(PFAC_ERR_ARG, "bad arguments");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    CU_TRY(cudaDeviceSynchronize());
    double total = 0;
    const size_t pairs = ctx->ev.size() / 2;
    for (size_t k = 0; k < ctx->ev_count; k++) {
        const size_t i = ((ctx->ev_next / 2 + pairs - 1 - k) % pairs) * 2;
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, ctx->ev[i], ctx->ev[i + 1]));
        total += ms;
    }
    *ms_total = total;
    *n_launches = (int)ctx->ev_count;
    ctx->ev_next = ctx->ev_count = 0;
    return PFAC_OK;
}

int pfac_ctx_derived_info(const pfac_ctx *ctx, uint64_t info[16])
{
    if (!ctx || !info) return set_error(PFAC_ERR_ARG, "bad arguments");
    const Derived &d = ctx->dv;
    const uint64_t v[16] = {ctx->image_bytes, d.t1_set, d.t2_shift >= 32 ? 0 : (1ull << (32 - d.t2_shift)), d.t2_set,
                            d.n_prefix4, d.has_short, d.tm_set, d.tm2_set,
                            d.t3_shift >= 32 ? 0 : (1ull << (32 - d.t3_shift)), d.t3_set, ctx->smem_bytes,
                            ctx->table_bytes(), ctx->n_stages, d.tm2_bits, d.mode, d.tm_bits};
    memcpy(info, v, sizeof v);
    return PFAC_OK;
}

int pfac_scan_device(pfac_ctx *ctx, const void *d_in, uint64_t n_starts, uint64_t n_valid, uint64_t base_pos,
                     void *d_out, uint64_t cap, void *d_count, void *stream)
{
    if (!ctx || (!d_in && n_starts) || (!d_out && cap) || !d_count) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_device");
    return run_own(ctx, stream, cap, nullptr, [&](cudaStream_t st, Counters &n) {
        return launch_scan(ctx, ctx->own, d_in, n_starts, n_valid, base_pos, 0u, d_out, cap, d_count, st, n, false);
    });
}

int pfac_scan_device_sync(pfac_ctx *ctx, const void *d_in, uint64_t n_starts, uint64_t n_valid, uint64_t base_pos,
                          void *d_out, uint64_t cap, uint64_t *count, void *stream)
{
    if (!ctx || !count || (!d_in && n_starts) || (!d_out && cap)) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_device_sync");
    return run_own(ctx, stream, cap, count, [&](cudaStream_t st, Counters &n) {
        return launch_scan(ctx, ctx->own, d_in, n_starts, n_valid, base_pos, 0u, d_out, cap, nullptr, st, n, false);
    });
}

int pfac_scan_batch_device(pfac_ctx *ctx, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                           void *d_out, uint64_t cap, void *d_doc_first, void *d_count, void *stream)
{
    if (!ctx || !doc_offsets || (!d_out && cap) || !d_doc_first || !d_count)
        return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_batch_device");
    return run_own(ctx, stream, cap, nullptr, [&](cudaStream_t st, Counters &n) {
        return launch_batch(ctx, ctx->own, d_in, doc_offsets, n_docs, d_out, cap, d_doc_first, d_count, st, n);
    });
}

int pfac_scan_batch_device_sync(pfac_ctx *ctx, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                                void *d_out, uint64_t cap, void *d_doc_first, uint64_t *count, void *stream)
{
    if (!ctx || !doc_offsets || (!d_out && cap) || !d_doc_first || !count)
        return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_batch_device_sync");
    return run_own(ctx, stream, cap, count, [&](cudaStream_t st, Counters &n) {
        return launch_batch(ctx, ctx->own, d_in, doc_offsets, n_docs, d_out, cap, d_doc_first, nullptr, st, n);
    });
}

int pfac_flows_create(pfac_ctx *ctx, uint32_t n_flows, pfac_flows **out)
{
    if (!ctx || !out || n_flows == 0) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_flows_create");
    if (ctx->batch_rc != PFAC_OK) return set_error(ctx->batch_rc, "%s", ctx->batch_why.c_str());
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    std::unique_ptr<pfac_flows> f(new pfac_flows);
    f->ctx = ctx;
    f->n_flows = n_flows;
    f->keep = (uint32_t)std::max(ctx->max_pat_len - 1, 0);
    f->stride = (f->keep + 15u) & ~15u;
    if (f->stride) {
        const int e = f->d_tails.alloc((size_t)n_flows * f->stride);
        if (e) return e;
    }
    f->pos.assign(n_flows, 0);
    f->seen.assign(n_flows, 0u);
    *out = f.release();
    return PFAC_OK;
}

void pfac_flows_destroy(pfac_flows *f)
{
    if (!f) return;
    std::lock_guard<std::mutex> lk(f->ctx->mu);
    DeviceGuard g(f->ctx->device);
    cudaDeviceSynchronize();   // (a failed call may have left work on a stream)
    delete f;                  // (frees the buffers on the context's device)
}

int pfac_flows_reset(pfac_flows *f, uint32_t flow)
{
    if (!f || flow >= f->n_flows) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_flows_reset");
    std::lock_guard<std::mutex> lk(f->mu);
    f->pos[flow] = 0;
    return PFAC_OK;
}

int pfac_flows_position(const pfac_flows *f, uint32_t flow, uint64_t *bytes)
{
    if (!f || !bytes || flow >= f->n_flows) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_flows_position");
    std::lock_guard<std::mutex> lk(f->mu);
    *bytes = f->pos[flow];
    return PFAC_OK;
}

int pfac_scan_flows_device_sync(pfac_flows *f, const void *d_in, const uint64_t *chunk_offsets, const uint32_t *flow_ids,
                                uint32_t n_chunks, void *d_out, uint64_t cap, void *d_chunk_first, uint64_t *base,
                                uint64_t *count, void *stream)
{
    if (!f || !chunk_offsets || (!flow_ids && n_chunks) || (!d_out && cap) || !d_chunk_first || (!base && n_chunks) || !count)
        return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_flows_device_sync");
    std::lock_guard<std::mutex> lk(f->mu);
    pfac_ctx *ctx = f->ctx;
    const int e = run_own(ctx, stream, cap, count, [&](cudaStream_t st, Counters &n) {
        return launch_flows(f, ctx->own, d_in, chunk_offsets, flow_ids, n_chunks, d_out, cap, d_chunk_first, base, st, n);
    });
    if (e) return e;   // nothing committed: the tail kernel wrote no tail either
    for (uint32_t i = 0; i < n_chunks; i++) f->pos[flow_ids[i]] += chunk_offsets[i + 1] - chunk_offsets[i];
    return PFAC_OK;
}

int pfac_host_alloc(void **ptr, size_t bytes)
{
    if (!ptr) return set_error(PFAC_ERR_ARG, "null ptr");
    CU_TRY(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocPortable));   // main.cc:147
    return PFAC_OK;
}

void pfac_host_free(void *ptr)
{
    if (ptr) cudaFreeHost(ptr);
}

int pfac_host_register(const void *ptr, size_t bytes, int read_only)
{
    if (!ptr || !bytes) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_host_register");
    unsigned flags = cudaHostRegisterPortable;
    if (read_only) flags |= cudaHostRegisterReadOnly;
    cudaError_t e = cudaHostRegister(const_cast<void *>(ptr), bytes, flags);
    if (e != cudaSuccess) {
        cudaGetLastError();   // not sticky: the caller may go on with pageable memory
        return set_error(PFAC_ERR_CUDA, "cudaHostRegister(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    }
    return PFAC_OK;
}

void pfac_host_unregister(const void *ptr)
{
    if (ptr) cudaHostUnregister(const_cast<void *>(ptr));
}

int pfac_ctx_last_scan_info(const pfac_ctx *ctx, uint64_t info[8])
{
    if (!ctx || !info) return set_error(PFAC_ERR_ARG, "bad arguments");
    memcpy(info, ctx->info, sizeof ctx->info);
    return PFAC_OK;
}

// H2D + kernel + D2H pipeline over n_streams stages (replaces the synchronous
// cudaMemcpy / launch / cudaMemcpy sequence of GPU_TraceTable, master_kernel.cu:359-428).
int pfac_scan_host(pfac_ctx *ctx, const void *h_in, uint64_t n_starts, uint64_t n_valid, uint64_t base_pos,
                   pfac_match *h_out, uint64_t cap, uint64_t *count)
{
    if (!ctx || (!h_in && n_starts) || (!h_out && cap) || !count || n_valid < n_starts)
        return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_host");
    if (n_valid >= (1ull << 32)) return set_error(PFAC_ERR_LIMIT, "pfac_scan_host takes less than 4 GiB per call");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    *count = 0;
    const uint64_t halo = ctx->max_pat_len > 0 ? (uint64_t)ctx->max_pat_len - 1 : 0;
    const uint64_t chunk = ctx->chunk_bytes;
    const uint64_t n_chunks = (n_starts + chunk - 1) / chunk;
    const int S = (int)std::min<uint64_t>((uint64_t)ctx->n_streams, std::max<uint64_t>(n_chunks, 1));
    const uint64_t first = std::min<uint64_t>(chunk, n_starts);
    for (int s = 0; s < S; s++) {
        Stage &st = ctx->stages[(size_t)s];
        int e;
        if (!st.stream) {
            CU_TRY(cudaStreamCreateWithFlags(&st.stream, cudaStreamNonBlocking));
            CU_TRY(cudaEventCreateWithFlags(&st.done, cudaEventDisableTiming));
            if ((e = slot_init(ctx, st.slot))) return e;
        }
        const size_t need_out = std::max<size_t>((size_t)(first / 8), 4096);
        if ((e = st.d_in.reserve((size_t)(first + halo + 64), 0, st.stream)) || (e = st.d_out.reserve(need_out, 0, st.stream)))
            return e;
    }
    // Whatever path leaves this function: no copy from h_in or into h_out may still be in flight (the
    // caller is free to release its buffers on an error).
    struct DrainOnExit {
        pfac_ctx *ctx;
        int S;
        ~DrainOnExit()
        {
            for (int s = 0; s < S; s++)
                if (ctx->stages[(size_t)s].stream) cudaStreamSynchronize(ctx->stages[(size_t)s].stream);
        }
    } drain{ctx, S};
    Counters n;
    n.chunks = n_chunks;
    auto enqueue = [&](uint64_t c) -> int {
        Stage &st = ctx->stages[(size_t)(c % (uint64_t)S)];
        const uint64_t off = c * chunk;
        const uint64_t ns = std::min<uint64_t>(chunk, n_starts - off);
        const uint64_t nv = std::min<uint64_t>(ns + halo, n_valid - off);
        CU_TRY(cudaMemcpyAsync(st.d_in.get(), (const uint8_t *)h_in + off, (size_t)nv, cudaMemcpyHostToDevice, st.stream));
        n.h2d += nv;
        Counters k;
        int e = launch_scan(ctx, st.slot, st.d_in.get(), ns, nv, base_pos + off, (uint32_t)off, st.d_out.get(),
                            st.d_out.cap(), nullptr, st.stream, k, true);
        if (e) return e;
        n.launches += k.launches;
        n.tiles += k.tiles;
        n.ctas = std::max(n.ctas, k.ctas);
        CU_TRY(cudaMemcpyAsync(st.slot.h_result.get(), st.slot.d_result.get(), sizeof(Result), cudaMemcpyDeviceToHost, st.stream));
        n.d2h += sizeof(Result);
        CU_TRY(cudaEventRecord(st.done, st.stream));
        return PFAC_OK;
    };
    int rc = PFAC_OK;
    for (uint64_t c = 0; c < std::min<uint64_t>((uint64_t)S, n_chunks); c++)
        if ((rc = enqueue(c)) != PFAC_OK) return rc;
    uint64_t total = 0;
    for (uint64_t c = 0; c < n_chunks; c++) {
        Stage &st = ctx->stages[(size_t)(c % (uint64_t)S)];
        uint64_t m = 0;
        CU_TRY(cudaEventSynchronize(st.done));
        if ((rc = check_result(*st.slot.h_result.get(), UINT64_MAX, &m))) return rc;   // (the watchdog alone)
        if (m > st.d_out.cap()) {
            // dense matches: grow this stage's record buffer and scan the sub-chunk again
            if ((rc = st.d_out.reserve((size_t)m, 0, st.stream)) || (rc = enqueue(c))) return rc;
            CU_TRY(cudaEventSynchronize(st.done));
            if ((rc = check_result(*st.slot.h_result.get(), UINT64_MAX, &m))) return rc;
        }
        // records already carry positions relative to h_in[0] (pos_bias = sub-chunk offset)
        const uint64_t room = total < cap ? cap - total : 0;
        const uint64_t ncopy = std::min<uint64_t>(m, room);
        if (ncopy) {
            CU_TRY(cudaMemcpyAsync(h_out + total, st.d_out.get(), (size_t)ncopy * sizeof(pfac_match),
                                   cudaMemcpyDeviceToHost, st.stream));
            n.d2h += ncopy * sizeof(pfac_match);
        }
        total += m;
        if (c + (uint64_t)S < n_chunks)
            if ((rc = enqueue(c + (uint64_t)S)) != PFAC_OK) return rc;
    }
    for (int s = 0; s < S; s++) CU_TRY(cudaStreamSynchronize(ctx->stages[(size_t)s].stream));
    set_info(ctx, n);
    return check_result(Result{total, 0u, 0u}, cap, count);
}

}  // extern "C"
