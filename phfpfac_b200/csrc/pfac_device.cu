// Device side of the C ABI (include/pfac_b200.h): contexts, table upload, the device-resident
// scan and the host pipeline.  Replaces GPU_Malloc_Memory / GPU_TraceTable / GPU_Free_memory
// (reference master_kernel.cu:188-524).  There is no CPU fallback anywhere in this file: a
// missing GPU or any CUDA error is reported as PFAC_ERR_NO_DEVICE / PFAC_ERR_CUDA.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>

#include "pfac_batch.cuh"
#include "pfac_derive.h"
#include "pfac_internal.h"
#include "pfac_kernel.cuh"

using namespace pfac;

#define CU_TRY(expr)                                                                         \
    do {                                                                                     \
        cudaError_t e_ = (expr);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return set_error(PFAC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                  \
                             cudaGetErrorString(e_), __FILE__, __LINE__);                    \
    } while (0)

namespace {

// Everything one in-flight scan needs besides the tables: control block, result block, tile
// directory and the arrival-order scratch.  One per user of a stream (the context's own slot for
// pfac_scan_device, one per pipeline stage for pfac_scan_host).
struct Slot {
    Ctrl *d_ctrl = nullptr;
    Result *d_result = nullptr;
    Result *h_result = nullptr;   // pinned
    // [2][kMaxParts] matches per tile range (walks -> ordering pass).  Two buffers, alternating per scan:
    // the walks of a scan add to one while its detector zeroes the other for the next scan (a buffer
    // zeroed at the start of the scan that uses it would race with the first walks)
    unsigned long long *d_partial = nullptr;
    unsigned flip = 0;
    unsigned int *d_tile_cnt = nullptr, *d_tile_nc = nullptr;
    unsigned long long *d_tile_src = nullptr;
    size_t tile_cap = 0;
    uint2 *d_scratch = nullptr;
    size_t scratch_cap = 0;   // records
    bool dirty = false;       // a launch sequence failed half way: the control block is reset before the next scan
    // batch scans (pfac_batch.cuh): raw records of the packed buffer and the global positions of the kept ones
    // (raw_cap each), the document offsets (pinned staging + device copy, doc_cap entries; doc_copied = end of
    // the last upload from the staging buffer) and the split pass's per-CTA counts
    uint2 *d_raw = nullptr;
    uint32_t *d_kpos = nullptr;
    size_t raw_cap = 0;
    uint32_t *h_doc = nullptr, *d_doc = nullptr;
    size_t doc_cap = 0;
    cudaEvent_t doc_copied = nullptr;
    unsigned long long *d_blk = nullptr;
};

struct Stage {   // one pipeline stage of pfac_scan_host
    cudaStream_t stream = nullptr;
    uint8_t *d_in = nullptr;
    size_t d_in_cap = 0;
    pfac_match *d_out = nullptr;
    size_t d_out_cap = 0;   // records
    Slot slot;
    cudaEvent_t done = nullptr;
};

}  // namespace

struct pfac_ctx {
    int device = 0;
    int sm_count = 0;
    int n_streams = 1;
    size_t chunk_bytes = 0;
    // tables (device): canonical s0Table, r, {HT, val}, idmap + the detector's shared-memory image
    int32_t *d_r = nullptr, *d_idmap = nullptr, *d_s0 = nullptr;
    int2 *d_htval = nullptr;
    int4 *d_step = nullptr;    // {HT, val, r[row of val]}: the candidate walks' one-load layout (PHF width >= 256)
    int2 *d_s0r = nullptr;     // {s0Table[b], r[row of it]}
    uint8_t *d_patdir = nullptr;   // pattern directory of the candidate walks (pfac_derive.h PatDir); null: none
    PatDir pd;                     // its layout (the image bytes are dropped after the upload)
    uint4 *d_image = nullptr;
    uint8_t *d_gimage = nullptr;   // mode 2: T1 | Tm | Tm2 | T3 in global memory
    uint8_t *d_wcache = nullptr;   // walk cache of the dense-match kernel (pfac_derive.h)
    WalkCache wc;                  // its layout (the image bytes are dropped after the upload)
    uint32_t wc_bytes = 0;
    size_t dense_smem = 0;
    bool dense_first = false;      // no detector: the dense-match kernel walks every tile (sets with patterns <= 3 bytes)
    // batch scans: pattern length of every id; batch_rc != PFAC_OK: the set does not support them (batch_why)
    int32_t *d_patlen = nullptr;
    uint32_t n_ids = 0;
    int batch_rc = PFAC_OK;
    std::string batch_why;
    Derived dv;   // image layout and hash parameters (the image bytes are dropped after the upload)
    uint32_t image_bytes = 0;
    int32_t ht_size = 0, width_bit = 0, n_final = 0, max_pat_len = 0;
    uint32_t halo = 16;
    uint32_t n_stages = 0;
    size_t smem_bytes = 0;
    size_t table_bytes = 0;
    // pfac_scan_device: own stream and slot
    cudaStream_t own_stream = nullptr;
    Slot own;                          // working set of pfac_scan_device[_sync]
    cudaEvent_t own_done = nullptr;    // end of the last device scan; a call on another stream waits for it
    cudaStream_t own_last = nullptr;
    bool own_used = false;
    std::vector<Stage> stages;
    uint64_t info[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // optional CUDA-event timing of the detector kernel alone (bench.py's roofline leg)
    bool timing = false;
    std::vector<cudaEvent_t> ev;   // pairs (before, after), used as a ring
    size_t ev_next = 0, ev_count = 0;
    uint32_t debug = 0;   // PFAC_DEBUG env (timing experiments only)
    bool use_pdl = true;  // PFAC_NO_PDL=1: plain stream-ordered launches (timing experiments only)
    std::mutex mu;
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

int slot_init(Slot &s)
{
    if (s.d_ctrl) return PFAC_OK;
    CU_TRY(cudaMalloc(&s.d_ctrl, sizeof(Ctrl)));
    CU_TRY(cudaMemset(s.d_ctrl, 0, sizeof(Ctrl)));
    CU_TRY(cudaMalloc(&s.d_result, sizeof(Result)));
    CU_TRY(cudaMalloc(&s.d_partial, 2 * kMaxParts * sizeof(unsigned long long)));
    CU_TRY(cudaMemset(s.d_partial, 0, 2 * kMaxParts * sizeof(unsigned long long)));
    CU_TRY(cudaHostAlloc(&s.h_result, sizeof(Result), cudaHostAllocPortable));
    return PFAC_OK;
}

void slot_free(Slot &s)
{
    if (s.d_ctrl) cudaFree(s.d_ctrl);
    if (s.d_result) cudaFree(s.d_result);
    if (s.d_partial) cudaFree(s.d_partial);
    if (s.h_result) cudaFreeHost(s.h_result);
    if (s.d_tile_cnt) cudaFree(s.d_tile_cnt);
    if (s.d_tile_src) cudaFree(s.d_tile_src);
    if (s.d_tile_nc) cudaFree(s.d_tile_nc);
    if (s.d_scratch) cudaFree(s.d_scratch);
    if (s.d_raw) cudaFree(s.d_raw);
    if (s.d_kpos) cudaFree(s.d_kpos);
    if (s.d_doc) cudaFree(s.d_doc);
    if (s.h_doc) cudaFreeHost(s.h_doc);
    if (s.doc_copied) cudaEventDestroy(s.doc_copied);
    if (s.d_blk) cudaFree(s.d_blk);
    s = Slot();
}

// Grow the tile directory / scratch of a slot.  Growing synchronises the stream first (the old
// buffers may still be in use); steady-state calls never get here.
int slot_reserve(Slot &s, size_t n_tiles, size_t records, cudaStream_t stream)
{
    if (n_tiles > s.tile_cap) {
        CU_TRY(cudaStreamSynchronize(stream));
        if (s.d_tile_cnt) cudaFree(s.d_tile_cnt);
        if (s.d_tile_src) cudaFree(s.d_tile_src);
        if (s.d_tile_nc) cudaFree(s.d_tile_nc);
                s.d_tile_cnt = s.d_tile_nc = nullptr;
        s.d_tile_src = nullptr;
        s.tile_cap = 0;
        const size_t n = std::max<size_t>(n_tiles, 1024);
        CU_TRY(cudaMalloc(&s.d_tile_cnt, n * sizeof(unsigned int)));
        CU_TRY(cudaMalloc(&s.d_tile_src, n * sizeof(unsigned long long)));
        CU_TRY(cudaMemset(s.d_tile_src, 0, n * sizeof(unsigned long long)));   // (epoch 0 = never published: DIRECT dense scans)
        CU_TRY(cudaMalloc(&s.d_tile_nc, n * sizeof(unsigned int)));
        s.tile_cap = n;
    }
    if (records > s.scratch_cap) {
        CU_TRY(cudaStreamSynchronize(stream));
        if (s.d_scratch) cudaFree(s.d_scratch);
        s.d_scratch = nullptr;
        s.scratch_cap = 0;
        const size_t n = std::max<size_t>(records, 4096);
        CU_TRY(cudaMalloc(&s.d_scratch, n * sizeof(uint2)));
        s.scratch_cap = n;
    }
    return PFAC_OK;
}

// Enqueue one scan (scan kernel + ordering pass) on `stream`.  On completion slot.d_result holds
// {count, error}; d_count (optional, device) receives the count as well.
int launch_scan(pfac_ctx *ctx, Slot &slot, const void *d_in, uint64_t n_starts, uint64_t n_valid, uint64_t base_pos,
                uint32_t pos_bias, void *d_out, uint64_t cap, void *d_count, cudaStream_t stream,
                uint64_t *tiles_out, uint64_t *ctas_out, uint64_t *launches_out)
{
    if (n_valid < n_starts) return set_error(PFAC_ERR_ARG, "n_valid < n_starts");
    const uint64_t useful = n_starts + (uint64_t)(ctx->max_pat_len > 0 ? ctx->max_pat_len - 1 : 0);
    if (n_valid > useful) n_valid = useful;
    const uint32_t mis = (uint32_t)((uintptr_t)d_in & 15u);
    if (n_valid + mis + (uint64_t)kTile + 4096 >= (1ull << 32))
        return set_error(PFAC_ERR_LIMIT, "one scan call covers less than 4 GiB; split the input");
    if (tiles_out) *tiles_out = 0;
    if (ctas_out) *ctas_out = 0;
    if (launches_out) *launches_out = 0;
    int e = slot_init(slot);
    if (e) return e;
    if (n_starts == 0 || ctx->max_pat_len == 0) {
        CU_TRY(cudaMemsetAsync(slot.d_result, 0, sizeof(Result), stream));
        if (d_count) CU_TRY(cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), stream));
        return PFAC_OK;
    }
    if (slot.dirty) {   // a previous launch sequence failed between the kernels: start from a clean control block
        CU_TRY(cudaMemsetAsync(slot.d_ctrl, 0, sizeof(Ctrl), stream));
        CU_TRY(cudaMemsetAsync(slot.d_partial, 0, 2 * kMaxParts * sizeof(unsigned long long), stream));
        slot.dirty = false;
    }
    struct DirtyOnError {   // set back to false on the success path
        Slot &s;
        bool armed = true;
        ~DirtyOnError() { if (armed) s.dirty = true; }
    } guard{slot};
    ScanParams p;
    memset(&p, 0, sizeof p);
    p.in_al = (const uint8_t *)d_in - mis;
    p.mis = mis;
    p.a_start_end = (uint32_t)(mis + n_starts);
    p.a_valid_end = (uint32_t)(mis + n_valid);
    p.n_tiles = (uint32_t)(((uint64_t)p.a_start_end + kTile - 1) / kTile);
    p.halo = ctx->halo;
    p.max_pat_len = (uint32_t)ctx->max_pat_len;
    p.use_ref_bound = ctx->max_pat_len > kRefHalo + 1;   // only then can the 4096+512 bound cut a walk
    p.base_pos = base_pos;
    p.image = ctx->d_image;
    p.image_bytes = ctx->image_bytes;
    p.off_t2 = ctx->dv.off_t2;
    p.off_tm = ctx->dv.off_tm;
    p.off_tm2 = ctx->dv.off_tm2;
    p.off_t3 = ctx->dv.off_t3;
    p.t2_shift = ctx->dv.t2_shift;
    p.has_short = ctx->dv.has_short;
    p.has_t3 = ctx->dv.has_t3;
    p.t3_shift = ctx->dv.t3_shift;
    p.tm_bits = ctx->dv.tm_bits;
    p.tm2_bits = ctx->dv.tm2_bits;
    p.off_d1 = ctx->dv.off_d1;
    p.off_e1 = ctx->dv.off_e1;
    p.nb1 = ctx->dv.nb1;
    p.ns1 = ctx->dv.ns1;
    p.off_d2 = ctx->dv.off_d2;
    p.off_e2 = ctx->dv.off_e2;
    p.nb2 = ctx->dv.nb2;
    p.ns2 = ctx->dv.ns2;
    p.gimage = ctx->d_gimage;
    if (ctx->n_stages < (uint32_t)min_stages((int)ctx->dv.mode))
        return set_error(PFAC_ERR_INTERNAL, "input ring of %u stages is too shallow for the slot scheme", ctx->n_stages);
    p.n_stages = ctx->n_stages;
    p.stage_magic = (uint32_t)((1ull << 32) / ctx->n_stages) + 1u;
    e = slot_reserve(slot, p.n_tiles, (size_t)std::max<uint64_t>(cap, 4096), stream);
    if (e) return e;
    p.tile_cnt = slot.d_tile_cnt;
    p.tile_nc = slot.d_tile_nc;
    unsigned long long *partial_now = slot.d_partial + (slot.flip & 1u) * kMaxParts;
    p.partial = partial_now;
    p.partial_next = slot.d_partial + ((slot.flip + 1u) & 1u) * kMaxParts;
    p.ctrl = slot.d_ctrl;
    p.debug = ctx->debug;
    const uint32_t grid = (uint32_t)std::min<uint64_t>(p.n_tiles, (uint64_t)ctx->sm_count);
    // tile ranges of the ordering pass: many small ones, so that dense outputs (every tile a long run
    // of records) are moved by the whole GPU
    const uint32_t fgrid = (uint32_t)std::min<uint64_t>((p.n_tiles + 7) / 8, (uint64_t)kMaxParts);
    const uint32_t tiles_per_part = (p.n_tiles + fgrid - 1) / fgrid;
    EmitParams ep;
    memset(&ep, 0, sizeof ep);
    ep.in_al = p.in_al;
    ep.mis = p.mis;
    ep.a_start_end = p.a_start_end;
    ep.a_valid_end = p.a_valid_end;
    ep.max_pat_len = p.max_pat_len;
    ep.use_ref_bound = p.use_ref_bound;
    ep.base_pos = base_pos;
    ep.pos_bias = pos_bias;
    ep.r = ctx->d_r;
    ep.htval = ctx->d_htval;
    ep.idmap = ctx->d_idmap;
    ep.s0 = ctx->d_s0;
    ep.step = ctx->d_step;
    ep.s0r = ctx->d_s0r;
    if (ctx->d_patdir) {
        ep.dir = reinterpret_cast<const uint4 *>(ctx->d_patdir);
        ep.pool = ctx->d_patdir + ctx->pd.off_pool;
        ep.dir_slots = ctx->pd.n_slots;
        ep.len_mask = ctx->pd.len_mask;
    }
    ep.ht_size = ctx->ht_size;
    ep.width_bit = ctx->width_bit;
    ep.n_final = ctx->n_final;
    ep.scratch = slot.d_scratch;
    ep.scratch_cap = slot.scratch_cap;
    ep.tile_cnt = slot.d_tile_cnt;
    ep.tile_src = slot.d_tile_src;
    ep.tile_nc = slot.d_tile_nc;
    ep.n_tiles = p.n_tiles;
    ep.tiles_per_part = tiles_per_part;
    ep.partial = partial_now;
    ep.ctrl = slot.d_ctrl;
    p.emit = ep;

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
    // Every kernel of a scan is a programmatic dependent launch: its CTAs are set up (and the detector's filter
    // image is on its way into shared memory) while the kernel before it -- the ordering pass of the previous
    // scan on this stream, for the detector -- still runs; each kernel waits (griddepcontrol.wait) before it
    // touches anything an earlier kernel may write.
    cudaLaunchAttribute pdl[1];
    pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof lc);
    lc.stream = stream;
    lc.attrs = pdl;
    lc.numAttrs = ctx->use_pdl ? 1 : 0;
    lc.gridDim = dim3(grid);
    lc.blockDim = dim3(kThreads);
    lc.dynamicSmemBytes = ctx->smem_bytes;
    if (dense_first) {}
    else if (ctx->dv.mode == 2) CU_TRY(cudaLaunchKernelEx(&lc, pfac_scan_kernel<2>, p));
    else if (ctx->dv.mode == 1) CU_TRY(cudaLaunchKernelEx(&lc, pfac_scan_kernel<1>, p));
    else if (ctx->dv.has_short) CU_TRY(cudaLaunchKernelEx(&lc, pfac_scan2_kernel<true, true, false>, p));
    else if (ctx->dv.has_shortc && ctx->dv.has_w3) CU_TRY(cudaLaunchKernelEx(&lc, pfac_scan2_kernel<false, true, true>, p));
    else if (ctx->dv.has_shortc) CU_TRY(cudaLaunchKernelEx(&lc, pfac_scan2_kernel<false, true, false>, p));
    else if (ctx->dv.has_w3) CU_TRY(cudaLaunchKernelEx(&lc, pfac_scan2_kernel<false, false, true>, p));
    else CU_TRY(cudaLaunchKernelEx(&lc, pfac_scan2_kernel<false, false, false>, p));
    if (ev_after && !dense_first) CU_TRY(cudaEventRecord(ev_after, stream));


    // the tiles the detector handed over whole (dense matches); returns at once when there are none
    DenseParams dp;
    memset(&dp, 0, sizeof dp);
    dp.e = ep;
    dp.wc_image = ctx->d_wcache;
    dp.wc_bytes = ctx->wc_bytes;
    dp.wc_depth = ctx->wc.depth;
    dp.wc_off_d = ctx->wc.off_d;
    dp.wc_off_e = ctx->wc.off_e;
    dp.wc_nb = ctx->wc.nb;
    dp.wc_ns = ctx->wc.ns;
    dp.halo = ctx->halo;
    dp.n_dense = &slot.d_ctrl->n_dense;
    if (dense_first) {   // the dense-match kernel is the whole scan: records go straight to the caller's buffer
        dp.out = (uint2 *)d_out;
        dp.cap = cap;
        dp.prefix = slot.d_tile_src;
        dp.epoch = slot.flip % 0xFFFFFEu + 1u;
        dp.result = slot.d_result;
        dp.count_out = (unsigned long long *)d_count;
        lc.gridDim = dim3(grid);
        lc.blockDim = dim3(kDenseThreads);
        lc.dynamicSmemBytes = ctx->dense_smem;
        CU_TRY(cudaLaunchKernelEx(&lc, pfac_dense_kernel<true>, dp));
        if (ev_after) CU_TRY(cudaEventRecord(ev_after, stream));
        if (tiles_out) *tiles_out = p.n_tiles;
        if (ctas_out) *ctas_out = grid;
        if (launches_out) *launches_out = 1;
        slot.flip++;
        guard.armed = false;
        return PFAC_OK;
    }
    // dense-match pass and ordering pass
    lc.gridDim = dim3(grid);
    lc.blockDim = dim3(kDenseThreads);
    lc.dynamicSmemBytes = ctx->dense_smem;
    CU_TRY(cudaLaunchKernelEx(&lc, pfac_dense_kernel<false>, dp));

    FinalizeParams f;
    f.tile_cnt = slot.d_tile_cnt;
    f.tile_src = slot.d_tile_src;
    f.scratch = slot.d_scratch;
    f.scratch_cap = slot.scratch_cap;
    f.out = (uint2 *)d_out;
    f.cap = cap;
    f.n_tiles = p.n_tiles;
    f.tiles_per_part = tiles_per_part;
    f.partial = partial_now;
    f.ctrl = slot.d_ctrl;
    f.result = slot.d_result;
    f.count_out = (unsigned long long *)d_count;
    f.debug = ctx->debug;
    f.trace_ctas = grid;
    lc.gridDim = dim3(fgrid);
    lc.blockDim = dim3(kFinThreads);
    lc.dynamicSmemBytes = 0;
    CU_TRY(cudaLaunchKernelEx(&lc, pfac_finalize_kernel, f));
    if (tiles_out) *tiles_out = p.n_tiles;
    if (ctas_out) *ctas_out = grid;
    if (launches_out) *launches_out = 3;
    slot.flip++;
    guard.armed = false;
    return PFAC_OK;
}

// Enqueue a batch scan on `stream` (pfac_batch.cuh): the documents' offsets are uploaded, the packed buffer is
// scanned into the slot's raw-record buffer, the split pass writes the caller's records, d_doc_first and
// d_count.  On completion slot.d_result holds {count, error}.  info: the counters of pfac_ctx_last_scan_info.
int launch_batch(pfac_ctx *ctx, Slot &slot, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                 void *d_out, uint64_t cap, void *d_doc_first, void *d_count, cudaStream_t stream, uint64_t info[8])
{
    if (ctx->batch_rc != PFAC_OK) return set_error(ctx->batch_rc, "%s", ctx->batch_why.c_str());
    if (n_docs == 0xFFFFFFFFu) return set_error(PFAC_ERR_LIMIT, "a batch holds fewer than 2^32 - 1 documents");
    if (doc_offsets[0] != 0)
        return set_error(PFAC_ERR_ARG, "doc_offsets[0] = %llu: the first document starts at 0", (unsigned long long)doc_offsets[0]);
    const uint64_t total = doc_offsets[n_docs];
    if (total >= (1ull << 32)) return set_error(PFAC_ERR_LIMIT, "one batch covers less than 4 GiB; split the input");
    if (!d_in && total) return set_error(PFAC_ERR_ARG, "null input of %llu bytes", (unsigned long long)total);
    int e = slot_init(slot);
    if (e) return e;
    const uint32_t grid = 2u * (uint32_t)ctx->sm_count;   // CTAs of the count and split kernels
    if (!slot.d_blk) CU_TRY(cudaMalloc(&slot.d_blk, (grid + 1) * sizeof(unsigned long long)));
    if (!slot.doc_copied) CU_TRY(cudaEventCreateWithFlags(&slot.doc_copied, cudaEventDisableTiming));
    // grow the offset and raw-record buffers (synchronises the stream first: the old ones may still be in use)
    const size_t n_off = (size_t)n_docs + 1;
    if (n_off > slot.doc_cap) {
        CU_TRY(cudaStreamSynchronize(stream));
        if (slot.d_doc) cudaFree(slot.d_doc);
        if (slot.h_doc) cudaFreeHost(slot.h_doc);
        slot.d_doc = slot.h_doc = nullptr;
        slot.doc_cap = 0;
        const size_t n = std::max<size_t>(n_off, 4096);
        CU_TRY(cudaMalloc(&slot.d_doc, n * sizeof(uint32_t)));
        CU_TRY(cudaHostAlloc(&slot.h_doc, n * sizeof(uint32_t), cudaHostAllocPortable));
        slot.doc_cap = n;
    }
    const size_t want = (size_t)std::max<uint64_t>(cap, 4096);
    if (want > slot.raw_cap) {
        CU_TRY(cudaStreamSynchronize(stream));
        if (slot.d_raw) cudaFree(slot.d_raw);
        if (slot.d_kpos) cudaFree(slot.d_kpos);
        slot.d_raw = nullptr;
        slot.d_kpos = nullptr;
        slot.raw_cap = 0;
        CU_TRY(cudaMalloc(&slot.d_raw, want * sizeof(uint2)));
        CU_TRY(cudaMalloc(&slot.d_kpos, want * sizeof(uint32_t)));
        slot.raw_cap = want;
    }
    // offsets -> pinned staging once the previous upload from it is done, checked on the way (32 bits suffice:
    // total < 4 GiB) -> device
    CU_TRY(cudaEventSynchronize(slot.doc_copied));
    uint64_t prev = 0;
    bool decreasing = false;
    for (size_t i = 0; i < n_off; i++) {
        const uint64_t v = doc_offsets[i];
        decreasing |= v < prev;
        prev = v;
        slot.h_doc[i] = (uint32_t)v;
    }
    if (decreasing) return set_error(PFAC_ERR_ARG, "doc_offsets decrease");
    CU_TRY(cudaMemcpyAsync(slot.d_doc, slot.h_doc, n_off * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    CU_TRY(cudaEventRecord(slot.doc_copied, stream));

    uint64_t tiles = 0, ctas = 0, launches = 0;
    e = launch_scan(ctx, slot, d_in, total, total, 0, 0u, slot.d_raw, slot.raw_cap, nullptr, stream, &tiles, &ctas,
                    &launches);
    if (e) return e;
    BatchParams bp;
    memset(&bp, 0, sizeof bp);
    bp.raw = slot.d_raw;
    bp.raw_cap = slot.raw_cap;
    bp.doc = slot.d_doc;
    bp.n_docs = n_docs;
    bp.len = ctx->d_patlen;
    bp.n_ids = ctx->n_ids;
    bp.blk = slot.d_blk;
    bp.out = (uint2 *)d_out;
    bp.cap = cap;
    bp.kpos = slot.d_kpos;
    bp.doc_first = (unsigned long long *)d_doc_first;
    bp.result = slot.d_result;
    bp.count_out = (unsigned long long *)d_count;
    cudaLaunchAttribute pdl[1];
    pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t lc = {};
    lc.stream = stream;
    lc.attrs = pdl;
    lc.numAttrs = ctx->use_pdl ? 1 : 0;
    lc.blockDim = dim3(kBatchThreads);
    lc.gridDim = dim3(grid);
    CU_TRY(cudaLaunchKernelEx(&lc, pfac_batch_count_kernel, bp));
    CU_TRY(cudaLaunchKernelEx(&lc, pfac_batch_split_kernel, bp));
    lc.gridDim = dim3((uint32_t)std::min<uint64_t>((n_off + kBatchThreads - 1) / kBatchThreads, grid));
    CU_TRY(cudaLaunchKernelEx(&lc, pfac_batch_docs_kernel, bp));
    info[0] = launches + 3;
    info[1] = tiles;
    info[2] = ctas;
    info[3] = ctx->smem_bytes;
    info[4] = n_off * sizeof(uint32_t);
    info[5] = 0;
    info[6] = 1;
    info[7] = 0;
    return PFAC_OK;
}

void free_stage(Stage &s)
{
    if (s.d_in) cudaFree(s.d_in);
    if (s.d_out) cudaFree(s.d_out);
    slot_free(s.slot);
    if (s.done) cudaEventDestroy(s.done);
    if (s.stream) cudaStreamDestroy(s.stream);
    s = Stage();
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
    // (every early return below releases what was allocated so far: pfac_ctx_destroy tolerates null members)
    std::unique_ptr<pfac_ctx, void (*)(pfac_ctx *)> ctx(new pfac_ctx, pfac_ctx_destroy);
    ctx->device = device;
    ctx->n_streams = n_streams;
    ctx->chunk_bytes = chunk_bytes ? chunk_bytes : ((size_t)32 << 20);
    ctx->chunk_bytes = (ctx->chunk_bytes + kTile - 1) / kTile * kTile;
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return set_error(PFAC_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only",
                         device, prop.major, prop.minor);
    ctx->sm_count = prop.multiProcessorCount;
    ctx->ht_size = P.ht_size;
    ctx->width_bit = width_bits(P.width);
    ctx->n_final = P.n_final;
    ctx->max_pat_len = P.max_len;
    ctx->halo = (uint32_t)std::max(16, ((P.max_len > 0 ? P.max_len - 1 : 0) + 15) / 16 * 16);
    if (const char *dbg = getenv("PFAC_DEBUG")) ctx->debug = (uint32_t)atoi(dbg);
    if (const char *v = getenv("PFAC_NO_PDL")) ctx->use_pdl = atoi(v) == 0;

    // shared-memory budget: T1 and the per-warp queues are fixed; T3 / Tm2 / T2 shrink until at least
    // four ring stages fit
    const size_t smem_max = (size_t)prop.sharedMemPerBlockOptin;
    uint32_t t2_bytes = 32768, t3_bytes = 32768, tm2_bytes = 32768;
    if (const char *v = getenv("PFAC_T2_BYTES")) t2_bytes = (uint32_t)atoi(v);
    if (const char *v = getenv("PFAC_T3_BYTES")) t3_bytes = (uint32_t)atoi(v);
    if (const char *v = getenv("PFAC_TM2_BYTES")) tm2_bytes = (uint32_t)atoi(v);
    bool widened = false;
    while (true) {
        derive_tables(P, t2_bytes, t3_bytes, tm2_bytes, ctx->dv);
        if (ctx->dv.mode == 2 && !widened && !getenv("PFAC_T2_BYTES")) {
            // global mode: T2 is stage 1 and the only shared-memory table -- give it all the room
            widened = true;
            t2_bytes = 131072;
            continue;
        }
        ctx->image_bytes = (uint32_t)ctx->dv.image.size();
        const size_t fixed = scan_smem_bytes(ctx->image_bytes, ctx->halo, 0, ctx->dv.mode);
        const size_t stride = scan_buf_stride(ctx->halo);
        const size_t fit = smem_max > fixed ? (smem_max - fixed) / stride : 0;
        const bool minimal = t2_bytes < 2048 && (ctx->dv.mode == 2 || (t3_bytes < 2048 && tm2_bytes < 2048));
        const size_t need = (size_t)min_stages((int)ctx->dv.mode);   // 2 (shared-memory mode) or 4 (global mode)
        // mode 0 wants a deep ring (bytes in flight hide the HBM latency): T3 gives way down to 16 KiB
        const bool deepen = ctx->dv.mode == 0 && fit < 9 && t3_bytes > 16384 && !getenv("PFAC_T3_BYTES");
        if (!deepen && (fit >= std::max<size_t>(3, need) || (fit >= need && minimal))) {
            ctx->n_stages = (uint32_t)std::min<size_t>(fit, kMaxStages);
            if (const char *v = getenv("PFAC_RING_STAGES"))   // tests: a ring as shallow as the slot scheme allows
                ctx->n_stages = (uint32_t)std::max<size_t>(need, std::min<size_t>(ctx->n_stages, (size_t)atoi(v)));
            ctx->smem_bytes = scan_smem_bytes(ctx->image_bytes, ctx->halo, ctx->n_stages, ctx->dv.mode);
            break;
        }
        if (minimal)
            return set_error(PFAC_ERR_CUDA, "scan kernel needs more than the %zu B of shared memory the device offers",
                             smem_max);
        // halve the largest section that is actually in the image
        if (ctx->dv.mode == 2) {
            t2_bytes /= 2;
        } else if (ctx->dv.has_t3) {
            if (t3_bytes > 8192) t3_bytes /= 2;          // T3 first: it only gets a little less selective
            else if (tm2_bytes >= 2048) tm2_bytes /= 2;  // then level 2 (all or nothing per size)
            else t3_bytes /= 2;
        } else {
            t3_bytes = tm2_bytes = 0;
            t2_bytes /= 2;
        }
    }

    // canonical arrays -> device, unchanged: s0Table, r, {HT, val} interleaved, idmap; + the detector image
    const size_t n_r = std::max<size_t>(P.r.size(), 1), n_ht = std::max<size_t>((size_t)P.ht_size, 1);
    const size_t n_id = std::max<size_t>((size_t)P.n_final, 1);
    std::vector<int2> htval(n_ht, make_int2(-1, -1));
    for (int32_t i = 0; i < P.ht_size; i++) htval[(size_t)i] = make_int2(P.HT[(size_t)i], P.val[(size_t)i]);
    std::vector<int32_t> s0(256, -1);
    if (!P.s0.empty()) s0 = P.s0;
    CU_TRY(cudaMalloc(&ctx->d_r, n_r * sizeof(int32_t)));
    CU_TRY(cudaMalloc(&ctx->d_htval, n_ht * sizeof(int2)));
    CU_TRY(cudaMalloc(&ctx->d_idmap, n_id * sizeof(int32_t)));
    CU_TRY(cudaMalloc(&ctx->d_s0, 256 * sizeof(int32_t)));
    CU_TRY(cudaMalloc(&ctx->d_image, ctx->image_bytes));
    CU_TRY(cudaMemset(ctx->d_r, 0xFF, n_r * sizeof(int32_t)));
    CU_TRY(cudaMemset(ctx->d_idmap, 0, n_id * sizeof(int32_t)));
    if (!P.r.empty()) CU_TRY(cudaMemcpy(ctx->d_r, P.r.data(), P.r.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(ctx->d_htval, htval.data(), n_ht * sizeof(int2), cudaMemcpyHostToDevice));
    if (P.n_final) CU_TRY(cudaMemcpy(ctx->d_idmap, P.idmap.data(), (size_t)P.n_final * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(ctx->d_s0, s0.data(), 256 * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(ctx->d_image, ctx->dv.image.data(), ctx->image_bytes, cudaMemcpyHostToDevice));
    if (ctx->width_bit >= 8 && !P.r.empty()) {
        // the one-load layout of the candidate walks: the row of a state's transitions depends on the state
        // alone when a row holds at least 256 keys, so every entry can carry its successor's r[] value
        const int sh = ctx->width_bit - 8;
        auto r_of = [&](int32_t state) -> int32_t {
            const size_t row = (size_t)state >> sh;
            return state >= 0 && row < P.r.size() ? P.r[row] : -1;
        };
        std::vector<int4> step(n_ht, make_int4(-1, -1, -1, 0));
        for (int32_t i = 0; i < P.ht_size; i++) step[(size_t)i] = make_int4(P.HT[(size_t)i], P.val[(size_t)i], r_of(P.val[(size_t)i]), 0);
        std::vector<int2> s0r(256);
        for (int b = 0; b < 256; b++) s0r[(size_t)b] = make_int2(s0[(size_t)b], r_of(s0[(size_t)b]));
        CU_TRY(cudaMalloc(&ctx->d_step, n_ht * sizeof(int4)));
        CU_TRY(cudaMalloc(&ctx->d_s0r, 256 * sizeof(int2)));
        CU_TRY(cudaMemcpy(ctx->d_step, step.data(), n_ht * sizeof(int4), cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(ctx->d_s0r, s0r.data(), 256 * sizeof(int2), cudaMemcpyHostToDevice));
    }
    if (!getenv("PFAC_NO_PATDIR")) derive_patdir(P, ctx->pd);
    if (ctx->pd.n_slots) {
        CU_TRY(cudaMalloc(&ctx->d_patdir, ctx->pd.image.size()));
        CU_TRY(cudaMemcpy(ctx->d_patdir, ctx->pd.image.data(), ctx->pd.image.size(), cudaMemcpyHostToDevice));
        ctx->table_bytes += ctx->pd.image.size();
        ctx->pd.image.clear();
        ctx->pd.image.shrink_to_fit();
    }
    if (!ctx->dv.gimage.empty()) {
        CU_TRY(cudaMalloc(&ctx->d_gimage, ctx->dv.gimage.size()));
        CU_TRY(cudaMemcpy(ctx->d_gimage, ctx->dv.gimage.data(), ctx->dv.gimage.size(), cudaMemcpyHostToDevice));
    }
    {   // walk cache of the dense-match kernel: as deep as fits beside its text tile and result arrays
        const size_t fixed = dense_smem_bytes(0, ctx->halo);
        const uint32_t budget = smem_max > fixed + 4096 ? (uint32_t)std::min<size_t>(smem_max - fixed, 128u << 10) : 2048u;
        derive_walk_cache(P, budget, ctx->wc);
        ctx->wc_bytes = (uint32_t)((ctx->wc.image.size() + 15) & ~(size_t)15);
        ctx->wc.image.resize(ctx->wc_bytes, 0);
        ctx->dense_smem = dense_smem_bytes(ctx->wc_bytes, ctx->halo);
        if (ctx->dense_smem > smem_max)
            return set_error(PFAC_ERR_CUDA, "dense-match kernel needs %zu B of shared memory (patterns too long)", ctx->dense_smem);
        CU_TRY(cudaMalloc(&ctx->d_wcache, ctx->wc_bytes));
        CU_TRY(cudaMemcpy(ctx->d_wcache, ctx->wc.image.data(), ctx->wc_bytes, cudaMemcpyHostToDevice));
        ctx->wc.image.clear();
        ctx->wc.image.shrink_to_fit();
        CU_TRY(cudaFuncSetAttribute(pfac_dense_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        CU_TRY(cudaFuncSetAttribute(pfac_dense_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    }
    {   // batch scans need each id's pattern length (a tree-shaped automaton) and results that do not depend on
        // where a document lies in the packed buffer (no reference tile bound: patterns of <= 513 bytes)
        std::vector<int32_t> len;
        if (pattern_lengths(P, len) != PFAC_OK) {
            ctx->batch_rc = PFAC_ERR_ARG;
            ctx->batch_why = pfac_last_error();
        } else if (P.max_len > kRefHalo + 1) {
            ctx->batch_rc = PFAC_ERR_LIMIT;
            ctx->batch_why = "batch scans need patterns of at most 513 bytes (the reference's 4096+512 tile bound "
                             "would make results depend on where a document lies in the batch)";
        } else {
            ctx->n_ids = (uint32_t)len.size();
            CU_TRY(cudaMalloc(&ctx->d_patlen, std::max<size_t>(len.size(), 1) * sizeof(int32_t)));
            if (!len.empty())
                CU_TRY(cudaMemcpy(ctx->d_patlen, len.data(), len.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
            ctx->table_bytes += std::max<size_t>(len.size(), 1) * sizeof(int32_t);
        }
    }
    ctx->dense_first = ctx->dv.has_short != 0;
    if (const char *v = getenv("PFAC_DENSE_FIRST")) ctx->dense_first = atoi(v) != 0;   // experiments: force either path
    ctx->table_bytes += n_r * 4 + n_ht * 8 + n_id * 4 + 1024 + ctx->image_bytes + ctx->dv.gimage.size() + ctx->wc_bytes + (ctx->d_step ? n_ht * 16 + 2048 : 0);
    ctx->dv.image.clear();
    ctx->dv.image.shrink_to_fit();
    ctx->dv.gimage.clear();
    ctx->dv.gimage.shrink_to_fit();

    // the attribute is per function and device, not per context: always allow the device maximum
    CU_TRY(cudaFuncSetAttribute(pfac_scan_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    CU_TRY(cudaFuncSetAttribute(pfac_scan_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    CU_TRY(cudaFuncSetAttribute(pfac_scan2_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    CU_TRY(cudaFuncSetAttribute(pfac_scan2_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    CU_TRY(cudaFuncSetAttribute(pfac_scan2_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    CU_TRY(cudaFuncSetAttribute(pfac_scan2_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    CU_TRY(cudaFuncSetAttribute(pfac_scan2_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    int bps = 0;
    if (ctx->dv.mode == 2)
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, pfac_scan_kernel<2>, kThreads, ctx->smem_bytes));
    else if (ctx->dv.mode == 1)
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, pfac_scan_kernel<1>, kThreads, ctx->smem_bytes));
    else
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, pfac_scan2_kernel<true, true, false>, kThreads, ctx->smem_bytes));
    if (bps < 1) return set_error(PFAC_ERR_CUDA, "scan kernel does not fit on an SM (smem %zu B)", ctx->smem_bytes);

    CU_TRY(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreateWithFlags(&ctx->own_done, cudaEventDisableTiming));
    int e = slot_init(ctx->own);
    if (e) return e;
    *out = ctx.release();
    return PFAC_OK;
}

void pfac_ctx_destroy(pfac_ctx *ctx)
{
    if (!ctx) return;
    DeviceGuard g(ctx->device);
    cudaDeviceSynchronize();
    for (auto &s : ctx->stages) free_stage(s);
    slot_free(ctx->own);
    if (ctx->d_r) cudaFree(ctx->d_r);
    if (ctx->d_htval) cudaFree(ctx->d_htval);
    if (ctx->d_step) cudaFree(ctx->d_step);
    if (ctx->d_s0r) cudaFree(ctx->d_s0r);
    if (ctx->d_patdir) cudaFree(ctx->d_patdir);
    if (ctx->d_idmap) cudaFree(ctx->d_idmap);
    if (ctx->d_image) cudaFree(ctx->d_image);
    if (ctx->d_s0) cudaFree(ctx->d_s0);
    if (ctx->d_gimage) cudaFree(ctx->d_gimage);
    if (ctx->d_wcache) cudaFree(ctx->d_wcache);
    if (ctx->d_patlen) cudaFree(ctx->d_patlen);
    for (auto e : ctx->ev)
        if (e) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->own_done) cudaEventDestroy(ctx->own_done);
    delete ctx;
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
                            ctx->table_bytes, ctx->n_stages, d.tm2_bits, d.mode, d.tm_bits};
    memcpy(info, v, sizeof v);
    return PFAC_OK;
}

// Device scans of one context share one working set (control block, tile directory, scratch): a scan
// enqueued on another stream than the one before it is ordered after it.
static int own_enter(pfac_ctx *ctx, cudaStream_t st)
{
    if (ctx->own_used && ctx->own_last != st) CU_TRY(cudaStreamWaitEvent(st, ctx->own_done, 0));
    return PFAC_OK;
}
static int own_leave(pfac_ctx *ctx, cudaStream_t st)
{
    CU_TRY(cudaEventRecord(ctx->own_done, st));
    ctx->own_last = st;
    ctx->own_used = true;
    return PFAC_OK;
}

int pfac_scan_device(pfac_ctx *ctx, const void *d_in, uint64_t n_starts, uint64_t n_valid, uint64_t base_pos,
                     void *d_out, uint64_t cap, void *d_count, void *stream)
{
    if (!ctx || (!d_in && n_starts) || (!d_out && cap) || !d_count) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_device");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->own_stream;
    uint64_t tiles = 0, ctas = 0, launches = 0;
    int e = own_enter(ctx, st);
    if (e) return e;
    e = launch_scan(ctx, ctx->own, d_in, n_starts, n_valid, base_pos, 0u, d_out, cap, d_count, st, &tiles, &ctas, &launches);
    if (e) return e;
    e = own_leave(ctx, st);
    if (e) return e;
    ctx->info[0] = launches;
    ctx->info[1] = tiles;
    ctx->info[2] = ctas;
    ctx->info[3] = ctx->smem_bytes;
    ctx->info[4] = ctx->info[5] = 0;
    ctx->info[6] = 1;
    return PFAC_OK;
}

int pfac_scan_device_sync(pfac_ctx *ctx, const void *d_in, uint64_t n_starts, uint64_t n_valid, uint64_t base_pos,
                          void *d_out, uint64_t cap, uint64_t *count, void *stream)
{
    if (!ctx || !count || (!d_in && n_starts) || (!d_out && cap)) return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_device_sync");
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->own_stream;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        DeviceGuard g(ctx->device);
        uint64_t tiles = 0, ctas = 0, launches = 0;
        int e = own_enter(ctx, st);
        if (e) return e;
        e = launch_scan(ctx, ctx->own, d_in, n_starts, n_valid, base_pos, 0u, d_out, cap, nullptr, st, &tiles, &ctas, &launches);
        if (e) return e;
        CU_TRY(cudaMemcpyAsync(ctx->own.h_result, ctx->own.d_result, sizeof(Result), cudaMemcpyDeviceToHost, st));
        e = own_leave(ctx, st);
        if (e) return e;
        CU_TRY(cudaStreamSynchronize(st));
        ctx->info[0] = launches;
        ctx->info[1] = tiles;
        ctx->info[2] = ctas;
        ctx->info[3] = ctx->smem_bytes;
        ctx->info[4] = ctx->info[5] = 0;
        ctx->info[6] = 1;
        if (ctx->own.h_result->error_flag)
            return set_error(PFAC_ERR_INTERNAL, "device watchdog tripped (code %u)", ctx->own.h_result->error_flag);
        *count = ctx->own.h_result->count;
    }
    if (*count > cap) return set_error(PFAC_ERR_OUTPUT_FULL, "%llu matches exceed the capacity of %llu records",
                                       (unsigned long long)*count, (unsigned long long)cap);
    return PFAC_OK;
}

int pfac_scan_batch_device(pfac_ctx *ctx, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                           void *d_out, uint64_t cap, void *d_doc_first, void *d_count, void *stream)
{
    if (!ctx || !doc_offsets || (!d_out && cap) || !d_doc_first || !d_count)
        return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_batch_device");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceGuard g(ctx->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->own_stream;
    uint64_t info[8];
    int e = own_enter(ctx, st);
    if (e) return e;
    e = launch_batch(ctx, ctx->own, d_in, doc_offsets, n_docs, d_out, cap, d_doc_first, d_count, st, info);
    if (e) return e;
    e = own_leave(ctx, st);
    if (e) return e;
    memcpy(ctx->info, info, sizeof info);
    return PFAC_OK;
}

int pfac_scan_batch_device_sync(pfac_ctx *ctx, const void *d_in, const uint64_t *doc_offsets, uint32_t n_docs,
                                void *d_out, uint64_t cap, void *d_doc_first, uint64_t *count, void *stream)
{
    if (!ctx || !doc_offsets || (!d_out && cap) || !d_doc_first || !count)
        return set_error(PFAC_ERR_ARG, "bad arguments to pfac_scan_batch_device_sync");
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->own_stream;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        DeviceGuard g(ctx->device);
        uint64_t info[8];
        int e = own_enter(ctx, st);
        if (e) return e;
        e = launch_batch(ctx, ctx->own, d_in, doc_offsets, n_docs, d_out, cap, d_doc_first, nullptr, st, info);
        if (e) return e;
        CU_TRY(cudaMemcpyAsync(ctx->own.h_result, ctx->own.d_result, sizeof(Result), cudaMemcpyDeviceToHost, st));
        e = own_leave(ctx, st);
        if (e) return e;
        CU_TRY(cudaStreamSynchronize(st));
        memcpy(ctx->info, info, sizeof info);
        if (ctx->own.h_result->error_flag)
            return set_error(PFAC_ERR_INTERNAL, "device watchdog tripped (code %u)", ctx->own.h_result->error_flag);
        *count = ctx->own.h_result->count;
    }
    if (*count > cap) return set_error(PFAC_ERR_OUTPUT_FULL, "%llu matches exceed the capacity of %llu records",
                                       (unsigned long long)*count, (unsigned long long)cap);
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
    if ((int)ctx->stages.size() < S) ctx->stages.resize((size_t)S);
    for (int s = 0; s < S; s++) {
        Stage &st = ctx->stages[(size_t)s];
        if (!st.stream) {
            CU_TRY(cudaStreamCreateWithFlags(&st.stream, cudaStreamNonBlocking));
            CU_TRY(cudaEventCreateWithFlags(&st.done, cudaEventDisableTiming));
            int e = slot_init(st.slot);
            if (e) return e;
        }
        const size_t need_in = (size_t)(std::min<uint64_t>(chunk, n_starts) + halo + 64);
        if (st.d_in_cap < need_in) {
            if (st.d_in) cudaFree(st.d_in);
            st.d_in = nullptr;
            st.d_in_cap = 0;
            CU_TRY(cudaMalloc(&st.d_in, need_in));
            st.d_in_cap = need_in;
        }
        const size_t need_out = std::max<size_t>((size_t)(std::min<uint64_t>(chunk, n_starts) / 8), 4096);
        if (st.d_out_cap < need_out) {
            if (st.d_out) cudaFree(st.d_out);
            st.d_out = nullptr;
            st.d_out_cap = 0;
            CU_TRY(cudaMalloc(&st.d_out, need_out * sizeof(pfac_match)));
            st.d_out_cap = need_out;
        }
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
    uint64_t h2d = 0, d2h = 0, launches = 0, tiles_total = 0, ctas_max = 0;
    auto enqueue = [&](uint64_t c) -> int {
        Stage &st = ctx->stages[(size_t)(c % (uint64_t)S)];
        const uint64_t off = c * chunk;
        const uint64_t ns = std::min<uint64_t>(chunk, n_starts - off);
        const uint64_t nv = std::min<uint64_t>(ns + halo, n_valid - off);
        CU_TRY(cudaMemcpyAsync(st.d_in, (const uint8_t *)h_in + off, (size_t)nv, cudaMemcpyHostToDevice, st.stream));
        h2d += nv;
        uint64_t tiles = 0, ctas = 0, nl = 0;
        int e = launch_scan(ctx, st.slot, st.d_in, ns, nv, base_pos + off, (uint32_t)off, st.d_out, st.d_out_cap, nullptr,
                            st.stream, &tiles, &ctas, &nl);
        if (e) return e;
        launches += nl;
        tiles_total += tiles;
        ctas_max = std::max(ctas_max, ctas);
        CU_TRY(cudaMemcpyAsync(st.slot.h_result, st.slot.d_result, sizeof(Result), cudaMemcpyDeviceToHost, st.stream));
        d2h += sizeof(Result);
        CU_TRY(cudaEventRecord(st.done, st.stream));
        return PFAC_OK;
    };
    int rc = PFAC_OK;
    for (uint64_t c = 0; c < std::min<uint64_t>((uint64_t)S, n_chunks); c++)
        if ((rc = enqueue(c)) != PFAC_OK) return rc;
    uint64_t total = 0;
    for (uint64_t c = 0; c < n_chunks; c++) {
        Stage &st = ctx->stages[(size_t)(c % (uint64_t)S)];
        CU_TRY(cudaEventSynchronize(st.done));
        if (st.slot.h_result->error_flag)
            return set_error(PFAC_ERR_INTERNAL, "device watchdog tripped (code %u)", st.slot.h_result->error_flag);
        uint64_t m = st.slot.h_result->count;
        if (m > st.d_out_cap) {
            // dense matches: grow this stage's record buffer and scan the sub-chunk again
            CU_TRY(cudaStreamSynchronize(st.stream));
            cudaFree(st.d_out);
            st.d_out = nullptr;
            st.d_out_cap = 0;
            CU_TRY(cudaMalloc(&st.d_out, (size_t)m * sizeof(pfac_match)));
            st.d_out_cap = (size_t)m;
            if ((rc = enqueue(c)) != PFAC_OK) return rc;
            CU_TRY(cudaEventSynchronize(st.done));
            if (st.slot.h_result->error_flag)
                return set_error(PFAC_ERR_INTERNAL, "device watchdog tripped (code %u)", st.slot.h_result->error_flag);
            m = st.slot.h_result->count;
        }
        // records already carry positions relative to h_in[0] (pos_bias = sub-chunk offset)
        const uint64_t room = total < cap ? cap - total : 0;
        const uint64_t ncopy = std::min<uint64_t>(m, room);
        if (ncopy) {
            CU_TRY(cudaMemcpyAsync(h_out + total, st.d_out, (size_t)ncopy * sizeof(pfac_match),
                                   cudaMemcpyDeviceToHost, st.stream));
            d2h += ncopy * sizeof(pfac_match);
        }
        total += m;
        if (c + (uint64_t)S < n_chunks)
            if ((rc = enqueue(c + (uint64_t)S)) != PFAC_OK) return rc;
    }
    for (int s = 0; s < S; s++) CU_TRY(cudaStreamSynchronize(ctx->stages[(size_t)s].stream));
    *count = total;
    ctx->info[0] = launches;
    ctx->info[1] = tiles_total;
    ctx->info[2] = ctas_max;
    ctx->info[3] = ctx->smem_bytes;
    ctx->info[4] = h2d;
    ctx->info[5] = d2h;
    ctx->info[6] = n_chunks;
    if (total > cap)
        return set_error(PFAC_ERR_OUTPUT_FULL, "%llu matches exceed the capacity of %llu records",
                         (unsigned long long)total, (unsigned long long)cap);
    return PFAC_OK;
}

}  // extern "C"
