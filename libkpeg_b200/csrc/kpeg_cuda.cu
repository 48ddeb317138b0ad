// kpeg_cuda.cu -- C-ABI host side of the B200 decode path (include/kpeg_cuda.h).
//
// A context owns eight LANES (CUDA stream + grow-only device scratch + pinned bookkeeping each) and
// the device tables built from a kpeg_plan.  A job is enqueued on a lane (K0..K3, kernels.cu) and
// finished later (stream sync, device status word, and -- rarely -- extra relay rounds).  Single
// decodes use lane 0; a large host-pointer batch is cut into chunks that rotate through the
// lanes so the H2D copy of one chunk, the kernels of another and the D2H copy of a third overlap
// (the end-to-end path is PCIe-bound: 3 bytes per pixel have to leave the device).
//
// There is no CPU decode in here: the only host arithmetic is table preparation (Huffman LUTs,
// AAN-prescaled quantisers, the 64 double cosines the exact IDCT path needs -- evaluated with the
// host libm exactly as the reference evaluates them, src/MCU.cpp:193).
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "encode.cuh"
#include "encode_host.h"
#include "host_tables.h"
#include "kernels.cuh"
#include "kpeg_common.h"
#include "kpeg_cuda.h"
#include "transcode_host.h"

using namespace kpeg;

namespace {

// Grow-only device scratch (ensure), freed with its owner.  Not movable: guard mode keeps pointers to the buffers.
struct DevBuf {
    const char *name;    // in guard-mode messages
    void *p = nullptr;   // what the kernels get
    size_t cap = 0;
    void *raw = nullptr; // the allocation (== p, or p - GUARD_BYTES in guard mode)

    DevBuf(const char *n) : name(n) {}
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    void release()
    {
        if (raw)
            cudaFree(raw);
        raw = p = nullptr;
        cap = 0;
    }
};

// KPEG_GUARD=1 (debugging aid; the pool this was developed on has no compute-sanitizer): every device buffer is
// allocated at exactly the size asked for, between two guard areas of a known byte, which are checked after each job.
constexpr size_t GUARD_BYTES = 256;
constexpr int GUARD_PATTERN = 0xA5;

// Grow-only pinned host memory (ensure_pinned), freed with its owner.
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;

    PinBuf() = default;
    PinBuf(const PinBuf &) = delete;
    PinBuf &operator=(const PinBuf &) = delete;
    ~PinBuf() { release(); }
    cudaError_t release()
    {
        const cudaError_t e = p ? cudaFreeHost(p) : cudaSuccess;
        p = nullptr;
        cap = 0;
        return e;
    }
};

constexpr int MAX_EVENTS = 192;
constexpr int NLANES = 8;

struct Copy {
    void *dst;
    const void *src;
    size_t bytes;
    int peer = -1; // >= 0: dst is device memory of that device (peer copy), otherwise host memory
};

// One in-flight job between job_enqueue and job_finish.
struct Job {
    bool active = false;
    JobGeom g = {};
    EntropyArgs ea = {};
    ExpandArgs xa = {};
    IdctArgs ia = {};
    int rounds = 0;
    uint32_t launches = 0;
    uint32_t extra_iterations = 0;
    bool use_records = true;
    bool loop_used = true; // relay rounds 2.. ran as the cooperative device-side loop (DevMeta::relay_rounds is meaningful)
    size_t scan_len = 0;
    std::vector<Copy> d2h; // result copies to (re)issue after the downstream stages
    bool entropy_only = false; // stop after K2: the tiles are the result (one scan of a frame coded one scan per component)
};

struct Lane {
    cudaStream_t stream = nullptr;
    DevBuf scan{"scan"}, words{"words"}, seg_bit{"seg_bit"}, tile_kept{"tile_kept"}, tile_rst{"tile_rst"}, cls{"cls"},
        state{"state"}, work{"work"}, seg_hint{"seg_hint"}, start_slot{"start_slot"}, scan_tiles{"scan_tiles"};
    DevBuf coef{"coef"}, dcdiff{"dcdiff"}, dc{"dc"}, tiles{"tiles"}, tie_rec{"tie_rec"}, tie_cnt{"tie_cnt"}, pixels{"pixels"},
        meta{"meta"}, rec{"rec"}, nrec{"nrec"}, rec_alt{"rec_alt"}, strip_sub{"strip_sub"}, dcs{"dcs"}, dcpre{"dcpre"},
        scan_tiles_dcs{"scan_tiles_dcs"};
    PinBuf h_meta;
    // host-buffer batches: pinned staging of the small scans + the separator positions, and their device copy
    PinBuf h_stage, h_ends;
    DevBuf d_ends{"d_ends"}, d_stage{"d_stage"};
    cudaEvent_t ev[MAX_EVENTS] = {};
    int ev_stage[MAX_EVENTS] = {};
    int nev = 0;
    Job job;

    ~Lane()
    {
        for (cudaEvent_t e : ev)
            if (e)
                cudaEventDestroy(e);
        if (stream)
            cudaStreamDestroy(stream);
    }
};

// Grow-only device scratch of the encoder (on lane 0's stream), and its tables, rebuilt when the quality changes.
// opt_tables / hist: the optimised mode's per-encode tables and symbol counts (the cached tables stay Annex K).
struct EncScratch {
    DevBuf buf[enc::BUF_COUNT] = {{"enc.coef"}, {"enc.raw"},      {"enc.dc"},    {"enc.has_ac"}, {"enc.bits"},
                                  {"enc.off"},  {"enc.seg_byte"}, {"enc.words"}, {"enc.agg"},    {"enc.tile_ff"}}; // BUF_* order
    DevBuf tables{"enc.tables"}, meta{"enc.meta"}, pixels{"enc.pixels"}, out{"enc.out"}, opt_tables{"enc.opt_tables"},
        hist{"enc.hist"};
    PinBuf h_tables, h_meta;
    int quality = -1;
};

} // namespace

struct kpeg_ctx {
    int device = 0;
    std::string err;
    bool profiling = false;
    uint32_t sub_bits = 512;
    // no size asked for (set_tuning / KPEG_SUB_BITS): 1024 bits for streams whose restart segments are long (>= 4 Mbit on
    // average: large images without restart markers) and whose blocks are long (>= 96 bits on average: high quality) -- the relay then converges in two rounds instead of five and the
    // cooperative loop, which holds SM slots while it waits out one serial subsequence decode per round, is a third as
    // long: +3 % on the 4K workload), 512 otherwise (segment boundaries are synchronisation points: 512 is 10-17 % faster
    // on the 512x512 batch and on the image with a restart interval per MCU row)
    bool sub_bits_auto = true;
    int relay_rounds = 8;
    bool use_records = true; // final pass = record expansion (KPEG_NO_RECORDS=1: Huffman final pass)
    int split_parts = 4;     // concurrent jobs a device-resident batch is cut into (KPEG_SPLIT)
    int host_chunks = 8;     // pipeline depth of a host-pointer batch (KPEG_HOST_CHUNKS)
    int submit_parts = 1;    // jobs one deferred submission is cut into (KPEG_SUBMIT_SPLIT)
    // bands a large restart-marked image from host memory is cut into, one per lane (KPEG_BANDS; 1 = off)
    int band_parts = 4;
    DevBuf band_counts{"band_counts"}; // RSTn markers counted per band (decode_banded)
    PinBuf h_band_counts;
    // result copies of the lanes leave one after another (each waits for the one enqueued before it): copies to the
    // host that run at the same time share the link AND slow each other down (measured: four concurrent 200 MB copies
    // take twice as long as the same four back to back); KPEG_D2H_CHAIN=0 turns the ordering off
    // relay round 2 as a launch of its own, rounds 3.. in the cooperative loop (KPEG_RELAY_ROUND2_WIDE=1).  Off: measured, the
    // loop takes as long without round 2 (every round costs the latency of one serial subsequence decode, ~35 us, whatever
    // the length of its list) and the extra launch costs 2 % of the throughput
    bool relay_round2_wide = false;
    bool d2h_chain = true;
    bool d2h_chain_armed = false;
    cudaEvent_t d2h_done = nullptr;
    Lane lane[NLANES];

    DevBuf tables{"tables"}, merged{"merged"};
    // frames coded one scan per component: the components' tiles before they are interleaved
    DevBuf scan_tiles[3] = {{"scan_tiles[0]"}, {"scan_tiles[1]"}, {"scan_tiles[2]"}};
    PinBuf h_tables, h_sep;
    cudaEvent_t tables_ready = nullptr;
    kpeg_plan plan_cached;
    bool have_plan = false;

    int last_lane = -1; // lane of the last finished job (kpeg_cuda_read_coefficients)
    JobGeom last_g = {};

    // deferred submissions (kpeg_cuda_submit_* / kpeg_cuda_wait): lanes are handed out round-robin and a
    // lane's previous job is finished only when the lane comes up again, so several batches are in flight
    bool counted = false; // registered with kernels_context_created
    bool guard = false;   // KPEG_GUARD=1
    std::vector<const DevBuf *> guarded; // guard mode: every buffer allocated so far (check_guards)
    bool plan_fits_records = true;
    int next_lane = 0;
    int deferred_rc = KPEG_OK;
    std::string deferred_err;
    kpeg_stats deferred_stats = {};

    EncScratch enc; // kpeg_cuda_encode*

    // the buffers free themselves after this; kpeg_cuda_destroy has synchronised every lane
    ~kpeg_ctx()
    {
        if (tables_ready)
            cudaEventDestroy(tables_ready);
        if (d2h_done)
            cudaEventDestroy(d2h_done);
    }
};

namespace {

static_assert(SCALE_FLAG_MASK == KPEG_FLAG_SCALE_MASK && (KPEG_FLAG_SCALE_1_2 >> SCALE_FLAG_SHIFT) == 1u &&
                  (KPEG_FLAG_SCALE_1_4 >> SCALE_FLAG_SHIFT) == 2u && (KPEG_FLAG_SCALE_1_8 >> SCALE_FLAG_SHIFT) == 3u,
              "kpeg_common.h's scale codes (scale_denom) are kpeg_cuda.h's KPEG_FLAG_SCALE_*");

// the decoded image of a plan (full size or reduced: KPEG_FLAG_SCALE_*)
OutGeom out_of(const kpeg_plan *pl) { return out_geom(pl->width, pl->height, pl->ncomp, pl->flags); }

int fail(kpeg_ctx *c, int code, const char *what, cudaError_t e = cudaSuccess)
{
    char buf[512];
    if (e != cudaSuccess)
        snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    else
        snprintf(buf, sizeof buf, "%s", what);
    if (c)
        c->err = buf;
    return code;
}

#define CK(call)                                                                                                       \
    do {                                                                                                               \
        cudaError_t e_ = (call);                                                                                       \
        if (e_ != cudaSuccess)                                                                                         \
            return fail(ctx, KPEG_ERR_CUDA, #call, e_);                                                                \
    } while (0)

#define TRY(expr)                                                                                                      \
    do {                                                                                                               \
        int rc_ = (expr);                                                                                              \
        if (rc_ != KPEG_OK)                                                                                            \
            return rc_;                                                                                                \
    } while (0)

int ensure(kpeg_ctx *ctx, cudaStream_t stream, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap)
        return KPEG_OK;
    if (b.raw) {
        CK(cudaStreamSynchronize(stream));
        b.release();
    }
    const bool guard = ctx->guard;
    const size_t want = guard ? ((bytes + 15u) & ~(size_t)15u) : bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.raw, want + (guard ? 2 * GUARD_BYTES : 0));
    if (e != cudaSuccess) {
        b.raw = nullptr;
        return fail(ctx, KPEG_ERR_NOMEM, "cudaMalloc", e);
    }
    b.p = b.raw;
    if (guard) {
        b.p = (uint8_t *)b.raw + GUARD_BYTES;
        if (std::find(ctx->guarded.begin(), ctx->guarded.end(), &b) == ctx->guarded.end())
            ctx->guarded.push_back(&b);
        CK(cudaMemsetAsync(b.raw, GUARD_PATTERN, GUARD_BYTES, stream));
        CK(cudaMemsetAsync((uint8_t *)b.p + want, GUARD_PATTERN, GUARD_BYTES, stream));
    }
    b.cap = want;
    return KPEG_OK;
}

int ensure_pinned(kpeg_ctx *ctx, cudaStream_t stream, PinBuf &b, size_t bytes)
{
    if (bytes <= b.cap)
        return KPEG_OK;
    if (b.p) {
        CK(cudaStreamSynchronize(stream));
        CK(b.release());
    }
    const size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMallocHost(&b.p, want);
    if (e != cudaSuccess) {
        b.p = nullptr;
        return fail(ctx, KPEG_ERR_NOMEM, "cudaMallocHost", e);
    }
    b.cap = want;
    return KPEG_OK;
}

// ---- plan -> device tables (shared by all lanes) ---------------------------------------------------
// The device tables (Huffman LUTs, quantisers) depend on the components' table selectors and the tables themselves,
// not on the image's dimensions, restart interval or flags: jobs that differ only in those -- the restart-interval
// bands of one image, say -- share the tables and can be in flight together.
bool same_tables(const kpeg_plan *a, const kpeg_plan *b)
{
    kpeg_plan x = *a, y = *b;
    x.width = y.width = x.height = y.height = 0;
    x.restart_interval = y.restart_interval = 0;
    x.flags = y.flags = 0;
    return memcmp(&x, &y, sizeof x) == 0;
}

int upload_plan(kpeg_ctx *ctx, const kpeg_plan *pl)
{
    if (ctx->have_plan && same_tables(&ctx->plan_cached, pl))
        return KPEG_OK;
    // a new plan: nothing may still be reading the old tables
    for (Lane &L : ctx->lane)
        CK(cudaStreamSynchronize(L.stream));
    cudaStream_t s0 = ctx->lane[0].stream;
    TRY(ensure_pinned(ctx, s0, ctx->h_tables, sizeof(DeviceTables)));
    TRY(ensure(ctx, s0, ctx->tables, sizeof(DeviceTables)));
    const char *why = nullptr;
    const int rc = build_device_tables(pl, (DeviceTables *)ctx->h_tables.p, &why);
    if (rc != KPEG_OK)
        return fail(ctx, rc, why);
    CK(cudaMemcpyAsync(ctx->tables.p, ctx->h_tables.p, sizeof(DeviceTables), cudaMemcpyHostToDevice, s0));
    CK(cudaEventRecord(ctx->tables_ready, s0));
    for (int i = 1; i < NLANES; ++i)
        CK(cudaStreamWaitEvent(ctx->lane[i].stream, ctx->tables_ready, 0));
    ctx->plan_cached = *pl;
    ctx->have_plan = true;
    // symbol records keep 11 magnitude bits (all baseline JPEG has: DC categories 0..11, AC 0..10, T.81
    // F.1.2.1.2 / F.1.2.2.1); a table that declares wider ones is decoded with the Huffman final pass
    ctx->plan_fits_records = true;
    for (int cls = 0; cls < 2; ++cls)
        for (int id = 0; id < 4; ++id) {
            if (!pl->ht_present[cls][id])
                continue;
            int nsym = 0;
            for (int L = 0; L < 16; ++L)
                nsym += pl->ht[cls][id].counts[L];
            for (int i = 0; i < nsym && i < 256; ++i)
                if ((pl->ht[cls][id].symbols[i] & 15) > 11)
                    ctx->plan_fits_records = false;
        }
    return KPEG_OK;
}

// ---- profiling: an event after every stage; mark(.., -1) opens a window on a lane -------------------
void mark(kpeg_ctx *ctx, Lane &L, int stage)
{
    if (!ctx->profiling)
        return;
    if (stage < 0)
        L.nev = 0;
    if (L.nev >= MAX_EVENTS)
        return;
    if (!L.ev[L.nev])
        cudaEventCreate(&L.ev[L.nev]);
    cudaEventRecord(L.ev[L.nev], L.stream);
    L.ev_stage[L.nev] = stage;
    ++L.nev;
}

void add_times(kpeg_ctx *ctx, Lane &L, kpeg_stats *stats)
{
    if (!stats || !ctx->profiling || L.nev < 2)
        return;
    static const bool timeline = getenv("KPEG_TIMELINE") != nullptr; // development: when every stage of every lane ended, relative to lane 0's window
    if (timeline && ctx->lane[0].ev[0]) {
        fprintf(stderr, "[kpeg timeline] lane %d:", (int)(&L - ctx->lane));
        for (int i = 0; i < L.nev; ++i) {
            float at = 0.0f;
            if (cudaEventElapsedTime(&at, ctx->lane[0].ev[0], L.ev[i]) != cudaSuccess)
                cudaGetLastError();
            fprintf(stderr, " %d@%.2f", L.ev_stage[i], at);
        }
        fprintf(stderr, "\n");
    }
    for (int i = 1; i < L.nev; ++i) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, L.ev[i - 1], L.ev[i]) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        const int st = L.ev_stage[i];
        if (st >= 0 && st < KPEG_T_COUNT) {
            stats->ms[st] += ms;
            stats->ms_total += ms;
        }
    }
    L.nev = 0;
}

int status_to_rc(kpeg_ctx *ctx, uint32_t st)
{
    if (st == 0)
        return KPEG_OK;
    char buf[160];
    snprintf(buf, sizeof buf, "corrupt entropy-coded data (device status 0x%x:%s%s%s%s%s%s)", st,
             (st & ST_BAD_CODE) ? " bad-code" : "", (st & ST_SLOT_OVERFLOW) ? " slot-overflow" : "",
             (st & ST_SEG_MISMATCH) ? " segment-length" : "", (st & ST_BAD_MARKER) ? " marker-in-scan" : "",
             (st & ST_EXIT_MISMATCH) ? " relay-mismatch" : "", (st & ST_SEG_COUNT) ? " restart-count" : "");
    ctx->err = buf;
    return KPEG_ERR_STREAM;
}

// everything downstream of the relay + the result copies + the bookkeeping read-back
int enqueue_downstream(kpeg_ctx *ctx, Lane &L)
{
    Job &J = L.job;
    cudaStream_t s = L.stream;
    launch_entropy_scan(J.ea, s, &J.launches);
    mark(ctx, L, KPEG_T_ENTROPY_SCAN);
    if (J.use_records) {
        launch_expand(J.xa, s, &J.launches); // K2
        mark(ctx, L, KPEG_T_ENTROPY_WRITE);
    } else {
        // fallback: the Huffman final pass writes a plain coefficient matrix (every slot of every block: no zero-fill)
        // and the DC differences; DC prediction and the conversion into K3's tiles are separate small kernels
        const size_t coef_bytes = (size_t)J.g.total_blocks * 128u;
        TRY(ensure(ctx, s, L.coef, coef_bytes + 256));
        TRY(ensure(ctx, s, L.dcdiff, (size_t)J.g.total_blocks * 2u + 16));
        TRY(ensure(ctx, s, L.dc, (size_t)J.g.total_blocks * 2u + 16));
        J.ea.coef = (int16_t *)L.coef.p;
        J.ea.dcdiff = (int16_t *)L.dcdiff.p;
        launch_entropy_write(J.ea, s, &J.launches);
        mark(ctx, L, KPEG_T_ENTROPY_WRITE);
        launch_dc_integrate(J.g, (const int16_t *)L.dcdiff.p, (int16_t *)L.dc.p, s, &J.launches);
        launch_tiles_from_matrix(J.g, (const int16_t *)L.coef.p, (const int16_t *)L.dc.p, J.xa.tiles, s, &J.launches);
        mark(ctx, L, KPEG_T_DC_SCAN);
    }
    if (!J.entropy_only) {
        CK(launch_idct(J.ia, s, &J.launches));
        mark(ctx, L, KPEG_T_IDCT);
    }
    const bool chain = ctx->d2h_chain && ctx->d2h_done && !J.d2h.empty();
    if (chain && ctx->d2h_chain_armed)
        CK(cudaStreamWaitEvent(s, ctx->d2h_done, 0));
    for (const Copy &c : J.d2h) {
        if (c.peer >= 0)
            CK(cudaMemcpyPeerAsync(c.dst, c.peer, c.src, ctx->device, c.bytes, s));
        else
            CK(cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToHost, s));
    }
    if (chain) {
        CK(cudaEventRecord(ctx->d2h_done, s));
        ctx->d2h_chain_armed = true;
    }
    if (!J.d2h.empty())
        mark(ctx, L, KPEG_T_D2H);
    CK(cudaMemcpyAsync(L.h_meta.p, L.meta.p, sizeof(DevMeta), cudaMemcpyDeviceToHost, s));
    return KPEG_OK;
}

int job_finish(kpeg_ctx *ctx, int li, kpeg_stats *stats);

// complete a deferred job; its outcome is reported by the next kpeg_cuda_wait
void finish_deferred(kpeg_ctx *ctx, int li)
{
    const int rc = job_finish(ctx, li, &ctx->deferred_stats);
    if (rc != KPEG_OK && ctx->deferred_rc == KPEG_OK) {
        ctx->deferred_rc = rc;
        ctx->deferred_err = ctx->err;
    }
}

// every pending deferred submission is completed first (its outcome is reported by kpeg_cuda_wait)
void finish_all_deferred(kpeg_ctx *ctx)
{
    for (int i = 0; i < NLANES; ++i)
        if (ctx->lane[i].job.active)
            finish_deferred(ctx, i);
}

// Lane 0 with no deferred job on it: such a job still reads the lane's scan / pixel buffers, which the caller is about to
// reuse.  Only lane 0: a deferred batch on the other lanes keeps overlapping the caller's synchronous work.
Lane &idle_lane0(kpeg_ctx *ctx)
{
    if (ctx->lane[0].job.active)
        finish_deferred(ctx, 0);
    return ctx->lane[0];
}

void reset_deferred(kpeg_ctx *ctx)
{
    ctx->deferred_rc = KPEG_OK;
    ctx->deferred_err.clear();
    memset(&ctx->deferred_stats, 0, sizeof ctx->deferred_stats);
}

// A synchronous call that runs its work as deferred submissions: the outcome of the caller's earlier submissions (for
// the caller's kpeg_cuda_wait) is set aside while it runs and restored when it returns.  Those submissions must be
// finished first (finish_all_deferred).
struct DeferredOutcomeSaved {
    kpeg_ctx *ctx;
    const int rc;
    const std::string err;
    const kpeg_stats stats;

    explicit DeferredOutcomeSaved(kpeg_ctx *c) : ctx(c), rc(c->deferred_rc), err(c->deferred_err), stats(c->deferred_stats)
    {
        reset_deferred(c);
    }
    ~DeferredOutcomeSaved()
    {
        ctx->deferred_rc = rc;
        ctx->deferred_err = err;
        ctx->deferred_stats = stats;
    }
};

// K3's arguments for geometry g on lane L: its tie lists and meta, and the context's tables
IdctArgs idct_args(kpeg_ctx *ctx, Lane &L, const JobGeom &g, uint32_t nstrips, const void *tiles, uint8_t *pixels)
{
    IdctArgs ia = {};
    ia.tiles = tiles;
    ia.nstrips = nstrips;
    ia.tables = (const DeviceTables *)ctx->tables.p;
    ia.pixels = pixels;
    ia.tie_rec = (uint4 *)L.tie_rec.p;
    ia.tie_cnt = (uint32_t *)L.tie_cnt.p;
    ia.meta = (DevMeta *)L.meta.p;
    ia.g = g;
    return ia;
}

// Enqueue the whole device pipeline for one job whose stuffed bytes are (or will be, in stream
// order) at d_scan.  Optimistic: the stages downstream of the relay are issued before it is known
// whether the pre-issued relay rounds reached the fixed point; job_finish repairs that if not.
int job_enqueue(kpeg_ctx *ctx, int li, const kpeg_plan *pl, const uint8_t *d_scan, size_t scan_len, uint32_t nimages,
                uint8_t *d_pixels, std::vector<Copy> d2h, void *tiles_only = nullptr)
{
    Lane &L = ctx->lane[li];
    Job &J = L.job;
    cudaStream_t s = L.stream;
    if (J.active) // a deferred job still owns this lane's scratch: complete it first
        finish_deferred(ctx, li);
    if (ctx->have_plan && !same_tables(&ctx->plan_cached, pl))
        finish_all_deferred(ctx); // the tables are shared: nothing deferred may outlive them
    JobGeom g;
    const char *why = nullptr;
    uint32_t sub_bits = ctx->sub_bits;
    if (ctx->sub_bits_auto) {
        const uint64_t segs = (uint64_t)nimages * (pl->restart_interval ? ((uint64_t)((pl->width + 7u) / 8u) * ((pl->height + 7u) / 8u) + pl->restart_interval - 1u) / pl->restart_interval : 1u);
        // ... and whose blocks are long (>= 96 bits on average, i.e. high quality settings): streams of short blocks
        // re-synchronise within a few hundred bits, their relay needs one or two rounds at 512 bits already (4K q50:
        // 145 Gpixel/s at 512 bits, 139 at 1024; 1080p q90: equal; 4K q95: 80 vs 87)
        const uint64_t blocks = (uint64_t)nimages * ((pl->width + 7u) / 8u) * ((pl->height + 7u) / 8u) * pl->ncomp;
        const uint64_t bits = (uint64_t)scan_len * 8u;
        sub_bits = (bits >= segs * ((uint64_t)4 << 20) && bits >= blocks * 96u) ? 1024u : 512u;
    }
    int rc = make_job_geom(pl, nimages, sub_bits, &g, &why);
    if (rc != KPEG_OK)
        return fail(ctx, rc, why);
    if ((pl->restart_interval != 0 || nimages > 1) && restart_padding_decodes(pl))
        return fail(ctx, KPEG_ERR_UNSUPPORTED, "the DC table fills the code space: the padding before a restart or image "
                                               "boundary would decode as a symbol (one image without restart markers decodes)");
    if (scan_len == 0 || scan_len >= (1ull << 29))
        return fail(ctx, KPEG_ERR_ARG, "entropy-coded segment must be 1 byte .. 512 MiB");
    TRY(upload_plan(ctx, pl));

    const uint32_t S = (uint32_t)scan_len;
    const uint32_t ntiles = (S + 15u + UNSTUFF_TILE - 1) / UNSTUFF_TILE; // + 15: chunks are cut on address boundaries
    const uint32_t nsub_max = (uint32_t)(((uint64_t)S * 8u + g.sub_bits - 1u) / g.sub_bits) + 1u;
    const uint32_t total_mcus = g.nimages * g.mcus_per_image;
    const uint32_t nstrips = (total_mcus + IDCT_MCUS_PER_CTA - 1) / IDCT_MCUS_PER_CTA;
    const size_t words_bytes = ((size_t)S + 3u) / 4u * 4u + 64u;

    TRY(ensure(ctx, s, L.words, words_bytes));
    TRY(ensure(ctx, s, L.seg_bit, ((size_t)g.nseg + 2u) * 4u));
    TRY(ensure(ctx, s, L.tile_kept, (size_t)ntiles * 4u));
    TRY(ensure(ctx, s, L.tile_rst, (size_t)ntiles * 4u));
    TRY(ensure(ctx, s, L.cls, (size_t)ntiles * UNSTUFF_THREADS * 4u));
    TRY(ensure(ctx, s, L.state, (size_t)nsub_max * sizeof(SubState)));
    TRY(ensure(ctx, s, L.work, (size_t)nsub_max * 2u * sizeof(uint32_t)));
    TRY(ensure(ctx, s, L.seg_hint, (size_t)nsub_max * 4u));
    TRY(ensure(ctx, s, L.start_slot, (size_t)nsub_max * 4u));
    TRY(ensure(ctx, s, L.scan_tiles, ((size_t)nsub_max / 1024u + 2u) * sizeof(uint2)));
    TRY(ensure(ctx, s, L.strip_sub, ((size_t)nstrips + 1u) * sizeof(uint32_t)));
    TRY(ensure(ctx, s, L.dcs, (size_t)nsub_max * sizeof(long long)));
    TRY(ensure(ctx, s, L.dcpre, (size_t)nsub_max * sizeof(long long)));
    TRY(ensure(ctx, s, L.scan_tiles_dcs, ((size_t)nsub_max / 1024u + 2u) * sizeof(long long)));
    TRY(ensure(ctx, s, L.tiles, (size_t)nstrips * IDCT_MCUS_PER_CTA * g.ncomp * 128u + 256u));
    TRY(ensure(ctx, s, L.tie_rec, (size_t)nstrips * IDCT_TIE_LIST_CAP * sizeof(uint4)));
    TRY(ensure(ctx, s, L.tie_cnt, (size_t)nstrips * sizeof(uint32_t)));
    TRY(ensure(ctx, s, L.meta, sizeof(DevMeta)));
    TRY(ensure_pinned(ctx, s, L.h_meta, sizeof(DevMeta)));
    // records: one per value-carrying symbol (host_tables.h rec_kmax_of)
    const uint32_t rec_kmax = rec_kmax_of(g.sub_bits);
    const uint32_t rec_alt_cap = nsub_max / 4u + 1024u; // beyond it a redone subsequence rewrites its interleaved column
    if (ctx->use_records) {
        TRY(ensure(ctx, s, L.rec, (size_t)rec_kmax * ((size_t)nsub_max / 32u + 1u) * 32u * sizeof(uint32_t)));
        TRY(ensure(ctx, s, L.nrec, (size_t)nsub_max * sizeof(uint32_t)));
        TRY(ensure(ctx, s, L.rec_alt, (size_t)rec_alt_cap * rec_kmax * sizeof(uint32_t)));
    }

    J = Job();
    J.use_records = ctx->use_records && ctx->plan_fits_records;
    J.active = true;
    J.g = g;
    J.scan_len = scan_len;
    J.d2h = std::move(d2h);
    J.entropy_only = tiles_only != nullptr;
    void *const tiles = tiles_only ? tiles_only : L.tiles.p;
    DevMeta *d_meta = (DevMeta *)L.meta.p;

    CK(cudaMemsetAsync(d_meta, 0, sizeof(DevMeta), s));
    mark(ctx, L, KPEG_T_MEMSET);

    UnstuffArgs ua;
    ua.scan = d_scan;
    ua.scan_len = S;
    ua.ntiles = ntiles;
    ua.tile_kept = (uint32_t *)L.tile_kept.p;
    ua.tile_rst = (uint32_t *)L.tile_rst.p;
    ua.cls = (uint32_t *)L.cls.p;
    ua.words = (uint8_t *)L.words.p;
    ua.seg_bit = (uint32_t *)L.seg_bit.p;
    ua.nseg = g.nseg;
    ua.meta = d_meta;
    launch_unstuff(ua, g.sub_bits, s, &J.launches);
    mark(ctx, L, KPEG_T_UNSTUFF);

    EntropyArgs &ea = J.ea;
    ea.words = (const uint32_t *)L.words.p;
    ea.seg_bit = (const uint32_t *)L.seg_bit.p;
    ea.tables = (const DeviceTables *)ctx->tables.p;
    ea.meta = d_meta;
    ea.state = (SubState *)L.state.p;
    ea.worklist[0] = (uint32_t *)L.work.p;
    ea.worklist[1] = (uint32_t *)L.work.p + nsub_max;
    ea.seg_hint = (uint32_t *)L.seg_hint.p;
    ea.start_slot = (uint32_t *)L.start_slot.p;
    ea.scan_tiles = (uint2 *)L.scan_tiles.p;
    ea.scan_tiles_dcs = (long long *)L.scan_tiles_dcs.p;
    ea.dcs = (long long *)L.dcs.p;
    ea.dcpre = (long long *)L.dcpre.p;
    ea.rec = J.use_records ? (uint32_t *)L.rec.p : nullptr;
    ea.nrec = (uint32_t *)L.nrec.p;
    ea.rec_kmax = rec_kmax;
    ea.rec_alt = (uint32_t *)L.rec_alt.p;
    ea.rec_alt_cap = rec_alt_cap;
    ea.coef = nullptr; // only the Huffman final pass writes coefficients to global memory (enqueue_downstream)
    ea.dcdiff = nullptr;
    ea.strip_sub = (uint32_t *)L.strip_sub.p;
    ea.strip_slots = k3_strip_slots(g.ncomp);
    ea.nstrips = nstrips;
    ea.nsub_max = nsub_max;
    ea.g = g;

    ExpandArgs &xa = J.xa;
    xa.rec = ea.rec;
    xa.nrec = ea.nrec;
    xa.rec_alt = ea.rec_alt;
    xa.rec_kmax = rec_kmax;
    xa.start_slot = ea.start_slot;
    xa.strip_sub = ea.strip_sub;
    xa.dcpre = ea.dcpre;
    xa.tiles = tiles;
    xa.nstrips = nstrips;
    xa.meta = d_meta;
    xa.g = g;

    J.ia = idct_args(ctx, L, g, nstrips, tiles, d_pixels);

    launch_entropy_cold(ea, s, &J.launches);
    mark(ctx, L, KPEG_T_ENTROPY_COLD);
    J.rounds = ctx->relay_rounds < 2 ? 2 : (ctx->relay_rounds > MAX_RELAY_ROUNDS - 1 ? MAX_RELAY_ROUNDS - 1 : ctx->relay_rounds);
    launch_entropy_relay(ea, 1, s, &J.launches);
    mark(ctx, L, KPEG_T_ENTROPY_RELAY);
    // (experiment knob, off: round 2 -- 6 % of the subsequences at 4K q95 -- as a wide launch of its own)
    if (ctx->relay_round2_wide)
        launch_entropy_relay(ea, 2, s, &J.launches);
    const int loop_first = ctx->relay_round2_wide ? 3 : 2;
    // the later rounds (0.5 %, 0.04 %, ...) in one cooperative launch (device-side loop, stops at the fixed point); the
    // cap only bounds the loop -- a stream that needs more is finished by job_finish
    J.rounds = MAX_RELAY_ROUNDS - 2;
    if (launch_entropy_relay_loop(ea, loop_first, J.rounds, s, &J.launches) != cudaSuccess) {
        // the driver refused the cooperative launch (MPS / a partitioned device): the same rounds as separate
        // launches; job_finish adds more if these do not reach the fixed point
        J.loop_used = false;
        J.rounds = std::max(loop_first, std::min(ctx->relay_rounds, MAX_RELAY_ROUNDS - 1));
        for (int r = loop_first; r <= J.rounds; ++r)
            launch_entropy_relay(ea, r, s, &J.launches);
    }
    mark(ctx, L, KPEG_T_RELAY_SPARSE);
    return enqueue_downstream(ctx, L);
}

// guard mode: the bytes on either side of every device buffer of the context must still hold the pattern.  The lanes
// are synchronised first: a buffer of another lane may have its guard areas still to be written on that lane's stream.
int check_guards(kpeg_ctx *ctx)
{
    for (Lane &L : ctx->lane)
        CK(cudaStreamSynchronize(L.stream));
    uint8_t host[2 * GUARD_BYTES];
    for (const DevBuf *bp : ctx->guarded) {
        const DevBuf &b = *bp;
        if (!b.raw)
            continue;
        CK(cudaMemcpy(host, b.raw, GUARD_BYTES, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(host + GUARD_BYTES, (const uint8_t *)b.p + b.cap, GUARD_BYTES, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < 2 * GUARD_BYTES; ++i)
            if (host[i] != (uint8_t)GUARD_PATTERN) {
                char msg[160];
                snprintf(msg, sizeof msg, "guard bytes %s device buffer '%s' (%zu bytes) were overwritten at offset %zu",
                         i < GUARD_BYTES ? "before" : "after", b.name, b.cap, i % GUARD_BYTES);
                return fail(ctx, KPEG_ERR_CUDA, msg);
            }
    }
    return KPEG_OK;
}

// Wait for the job, check the device status word and -- rarely -- run more relay rounds and redo the
// downstream stages.  Adds the job's figures to *stats (which the caller zeroed).
int job_finish(kpeg_ctx *ctx, int li, kpeg_stats *stats)
{
    Lane &L = ctx->lane[li];
    Job &J = L.job;
    if (!J.active)
        return KPEG_OK;
    J.active = false;
    cudaStream_t s = L.stream;
    DevMeta *d_meta = (DevMeta *)L.meta.p;
    DevMeta *h_meta = (DevMeta *)L.h_meta.p;
    for (;;) {
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        if (h_meta->status & (ST_BAD_MARKER | ST_SEG_COUNT))
            break; // malformed container-level structure: more rounds will not help
        // the loop's grid barrier gave up (its CTAs were not co-resident: another process on the device): rounds up
        // to relay_rounds are complete, the next one may be partly done and is repeated on its partly filled list
        const bool timed_out = (h_meta->status & ST_RELAY_TIMEOUT) != 0u;
        if (J.extra_iterations == 0u && J.loop_used)
            J.rounds = (int)std::max<uint32_t>(h_meta->relay_rounds, 1u); // last round the device loop completed
        const bool converged_now = !timed_out && h_meta->changed[relay_slot(J.rounds)] == 0u;
        if (converged_now && J.use_records && (h_meta->status & ST_REC_OVERFLOW)) {
            // a subsequence held more symbols than the record list: redo the final pass the Huffman way
            J.use_records = false;
            CK(cudaMemsetAsync(&d_meta->status, 0, sizeof(uint32_t), s));
            CK(cudaMemsetAsync(&d_meta->exact_samples, 0, 2 * sizeof(uint32_t), s));
            TRY(enqueue_downstream(ctx, L));
            continue;
        }
        if (converged_now)
            break; // the last relay round changed nothing: fixed point, results are final
        // Rare: the relay needed more rounds than were pre-issued.  Run two more at a time until a
        // round changes nothing, then redo the downstream stages.
        bool converged = false;
        bool repeat = timed_out; // the first round issued here continues a partly filled list: its count is kept
        const uint32_t cap = h_meta->nsub / 2u + 4u;
        while (!converged && J.extra_iterations < cap) {
            ++J.extra_iterations;
            for (int k = 0; k < 2; ++k) {
                ++J.rounds;
                if (!repeat)
                    CK(cudaMemsetAsync(&d_meta->changed[relay_slot(J.rounds)], 0, sizeof(uint32_t), s));
                repeat = false;
                launch_entropy_relay(J.ea, J.rounds, s, &J.launches);
            }
            mark(ctx, L, KPEG_T_RELAY_SPARSE);
            CK(cudaMemcpyAsync(h_meta, d_meta, sizeof(DevMeta), cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            converged = h_meta->changed[relay_slot(J.rounds)] == 0u;
        }
        if (!converged)
            return fail(ctx, KPEG_ERR_NOT_CONVERGED, "speculative decode did not reach a fixed point");
        CK(cudaMemsetAsync(&d_meta->status, 0, sizeof(uint32_t), s));
        CK(cudaMemsetAsync(&d_meta->exact_samples, 0, 2 * sizeof(uint32_t), s));
        TRY(enqueue_downstream(ctx, L));
    }
    if (ctx->guard)
        TRY(check_guards(ctx));
    ctx->last_lane = li;
    ctx->last_g = J.g;
    if (stats) {
        const OutGeom o = out_geom(J.g);
        stats->width = o.width;
        stats->height = o.height;
        stats->ncomp = J.g.ncomp;
        stats->scan_bytes += J.scan_len;
        stats->unstuffed_bytes += h_meta->total_kept;
        stats->segments += h_meta->total_rst + 1u;
        stats->subsequences += h_meta->nsub;
        uint32_t used_rounds = (uint32_t)J.rounds;
        if (J.extra_iterations == 0u) { // rounds that still changed something
            used_rounds = 0;
            for (int r = 1; r <= J.rounds && r < MAX_RELAY_ROUNDS; ++r)
                if (h_meta->changed[r])
                    used_rounds = (uint32_t)r;
        }
        stats->sync_rounds = std::max(stats->sync_rounds, used_rounds);
        stats->exact_samples += h_meta->exact_samples; // IDCT samples re-evaluated in the reference's operation order
        stats->kernel_launches += J.launches;
        add_times(ctx, L, stats);
    }
    return status_to_rc(ctx, h_meta->status & ~(ST_REC_OVERFLOW | ST_RELAY_TIMEOUT));
}

void zero_stats(kpeg_stats *stats)
{
    if (stats)
        memset(stats, 0, sizeof *stats);
}

// the figures of one part of a call added to the call's, as job_finish adds a job's (the output size is the caller's)
void add_stats(kpeg_stats &to, const kpeg_stats &part)
{
    to.scan_bytes += part.scan_bytes;
    to.unstuffed_bytes += part.unstuffed_bytes;
    to.segments += part.segments;
    to.subsequences += part.subsequences;
    to.sync_rounds = std::max(to.sync_rounds, part.sync_rounds);
    to.exact_samples += part.exact_samples;
    to.kernel_launches += part.kernel_launches;
    for (int t = 0; t < KPEG_T_COUNT; ++t)
        to.ms[t] += part.ms[t];
    to.ms_total += part.ms_total;
}

// A scan in host memory decoded on lane 0 (which the caller has made idle), complete on return: copied into the lane's
// scan buffer, then job_enqueue's pixels / d2h / tiles_only and job_finish's stats.
int decode_host_scan(kpeg_ctx *ctx, const kpeg_plan *pl, const uint8_t *scan, size_t scan_len, uint8_t *d_pixels,
                     std::vector<Copy> d2h, void *tiles_only, kpeg_stats *stats)
{
    Lane &L = ctx->lane[0];
    TRY(ensure(ctx, L.stream, L.scan, scan_len + 64));
    mark(ctx, L, -1);
    CK(cudaMemcpyAsync(L.scan.p, scan, scan_len, cudaMemcpyHostToDevice, L.stream));
    mark(ctx, L, KPEG_T_H2D);
    TRY(job_enqueue(ctx, 0, pl, (const uint8_t *)L.scan.p, scan_len, 1, d_pixels, std::move(d2h), tiles_only));
    return job_finish(ctx, 0, stats);
}

// The three scans of a frame coded one scan per component, entropy-decoded one after another on lane 0 into the
// components' tiles ctx->scan_tiles[c] (nmcu_padded blocks each); their figures are added to *stats.
int entropy_decode_component_scans(kpeg_ctx *ctx, const kpeg_scan *scans, const uint8_t *file, uint32_t flags, uint32_t nmcu_padded,
                                   kpeg_stats *stats)
{
    for (int c = 0; c < 3; ++c)
        TRY(ensure(ctx, ctx->lane[0].stream, ctx->scan_tiles[c], (size_t)nmcu_padded * 128u + 256u));
    for (int k = 0; k < 3; ++k) {
        kpeg_plan pl = scans[k].plan;
        pl.flags = flags;
        kpeg_stats part = {};
        TRY(decode_host_scan(ctx, &pl, file + scans[k].off, scans[k].len, nullptr, {}, ctx->scan_tiles[scans[k].comp[0]].p,
                             stats ? &part : nullptr));
        if (stats)
            add_stats(*stats, part);
    }
    return KPEG_OK;
}

// One large restart-marked image from host memory: bands of whole MCU rows, each a complete image of the same width
// and tables, go through the lanes one band per lane, so the copy in of one band, the kernels of another and the copy
// out of a third overlap.  The scan is cut at BYTE positions (the first RSTn marker at or after k/parts of its length: a
// memchr over a few hundred bytes); how many restart intervals -- hence MCU rows -- each band holds is counted on the GPU
// from the band's own bytes once they are there (count_restart_markers_kernel: 10 us for 24 MB), so the host never walks
// the scan.  (Finding cut points at given ROWS instead is a marker walk over the whole scan, 12 ms for 96 MB, more
// than the overlap gains: profiles/README.md.)  Needs a restart interval of whole MCU rows.  Synchronous.
// KPEG_ERR_UNSUPPORTED when the image does not qualify (nothing has been enqueued then).
int decode_banded(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len, uint8_t *pixels_out, kpeg_stats *stats)
{
    const uint32_t mx = (plan->width + 7u) / 8u, my = (plan->height + 7u) / 8u, ri = plan->restart_interval;
    if (ri == 0 || ri % mx != 0 || scan_len < (1u << 20))
        return KPEG_ERR_UNSUPPORTED;
    const uint32_t rows_per_interval = ri / mx;
    const uint32_t parts = (uint32_t)std::min(ctx->band_parts, NLANES);
    if (parts < 2 || my < parts * rows_per_interval * 2u)
        return KPEG_ERR_UNSUPPORTED;
    // cut points: the first RSTn marker at or after k / parts of the scan
    size_t begin[NLANES + 1], end[NLANES];
    begin[0] = 0;
    for (uint32_t k = 1; k < parts; ++k) {
        const uint8_t *p = scan + std::max(scan_len * k / parts, begin[k - 1] + 1), *stop = scan + scan_len;
        const uint8_t *cut = nullptr;
        while (p + 1 < stop) {
            const uint8_t *q = (const uint8_t *)memchr(p, 0xFF, (size_t)(stop - 1 - p));
            if (!q)
                break;
            if ((q[1] & 0xF8u) == 0xD0u) {
                cut = q;
                break;
            }
            p = q + 1;
        }
        if (!cut)
            return KPEG_ERR_UNSUPPORTED; // no marker in the rest of the scan: not the stream the plan describes; decoded whole
        end[k - 1] = (size_t)(cut - scan);
        begin[k] = end[k - 1] + 2u;
    }
    end[parts - 1] = scan_len;
    finish_all_deferred(ctx);
    // copies in + marker counts, every band on its own lane
    TRY(ensure(ctx, ctx->lane[0].stream, ctx->band_counts, NLANES * sizeof(uint32_t)));
    TRY(ensure_pinned(ctx, ctx->lane[0].stream, ctx->h_band_counts, NLANES * sizeof(uint32_t)));
    uint32_t *d_counts = (uint32_t *)ctx->band_counts.p, *h_counts = (uint32_t *)ctx->h_band_counts.p;
    for (uint32_t k = 0; k < parts; ++k) {
        Lane &L = ctx->lane[k];
        const size_t blen = end[k] - begin[k];
        TRY(ensure(ctx, L.stream, L.scan, blen + 64));
        mark(ctx, L, -1);
        CK(cudaMemcpyAsync(L.scan.p, scan + begin[k], blen, cudaMemcpyHostToDevice, L.stream));
        if (k + 1 < parts) { // the last band holds whatever rows are left
            CK(cudaMemsetAsync(d_counts + k, 0, sizeof(uint32_t), L.stream));
            launch_count_restart_markers((const uint8_t *)L.scan.p, (uint32_t)blen, d_counts + k, L.stream);
            CK(cudaMemcpyAsync(h_counts + k, d_counts + k, sizeof(uint32_t), cudaMemcpyDeviceToHost, L.stream));
        }
        mark(ctx, L, KPEG_T_H2D);
    }
    int rc = KPEG_OK, used[NLANES], nused = 0;
    uint32_t row0 = 0; // first MCU row of the band
    for (uint32_t k = 0; k < parts && rc == KPEG_OK; ++k) {
        Lane &L = ctx->lane[k];
        uint32_t rows = my - row0;
        if (k + 1 < parts) {
            CK(cudaStreamSynchronize(L.stream)); // the band is on the device and its markers are counted
            const uint64_t r = ((uint64_t)h_counts[k] + 1u) * rows_per_interval;
            if (r >= rows) { // more intervals than the frame has rows for: corrupt stream
                rc = fail(ctx, KPEG_ERR_STREAM, "restart markers do not match the restart interval");
                break;
            }
            rows = (uint32_t)r;
        }
        const uint32_t y0 = row0 * 8u, y1 = std::min<uint32_t>((row0 + rows) * 8u, plan->height);
        kpeg_plan bp = *plan;
        bp.height = (uint16_t)(y1 - y0);
        const OutGeom bo = out_of(&bp); // the band's output: its rows begin where its first MCU row's do
        const size_t bpix = bo.bytes();
        rc = ensure(ctx, L.stream, L.pixels, bpix + 64);
        if (rc != KPEG_OK)
            break;
        rc = job_enqueue(ctx, (int)k, &bp, (const uint8_t *)L.scan.p, end[k] - begin[k], 1, (uint8_t *)L.pixels.p,
                         {Copy{pixels_out + (size_t)bo.mcu_row(row0) * bo.row_bytes(), L.pixels.p, bpix}});
        if (rc == KPEG_OK)
            used[nused++] = (int)k;
        row0 += rows;
    }
    const std::string first_err = ctx->err;
    for (int i = 0; i < nused; ++i) { // every enqueued band is completed, whatever happened to the others
        const int frc = job_finish(ctx, used[i], stats);
        if (rc == KPEG_OK && frc != KPEG_OK)
            rc = frc;
        else if (frc != KPEG_OK)
            ctx->err = first_err;
    }
    for (uint32_t k = 0; k < parts; ++k) // lanes whose copies were issued but whose band was never enqueued
        cudaStreamSynchronize(ctx->lane[k].stream);
    if (stats) {
        const OutGeom o = out_of(plan);
        stats->width = o.width;
        stats->height = o.height;
    }
    return rc;
}

} // namespace

// ==================================================================================================
// C ABI
// ==================================================================================================

extern "C" size_t kpeg_output_size(const kpeg_plan *plan, uint32_t *w, uint32_t *h)
{
    if (!plan || plan->width == 0 || plan->height == 0 || (plan->ncomp != 1 && plan->ncomp != 3))
        return 0;
    const OutGeom o = out_of(plan);
    if (w)
        *w = o.width;
    if (h)
        *h = o.height;
    return (size_t)o.bytes();
}

extern "C" int kpeg_cuda_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int kpeg_cuda_create(int device, kpeg_ctx **out)
{
    if (!out)
        return KPEG_ERR_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return KPEG_ERR_CUDA; // no CPU fallback: the caller gets an error
    }
    if (cudaSetDevice(device) != cudaSuccess)
        return KPEG_ERR_CUDA;
    kpeg_ctx *ctx = new (std::nothrow) kpeg_ctx();
    if (!ctx)
        return KPEG_ERR_NOMEM;
    ctx->device = device;
    for (Lane &L : ctx->lane) {
        if (cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking) != cudaSuccess) {
            kpeg_cuda_destroy(ctx);
            return KPEG_ERR_CUDA;
        }
    }
    cudaEventCreateWithFlags(&ctx->tables_ready, cudaEventDisableTiming);
    kernels_configure(NLANES);
    kernels_context_created();
    ctx->counted = true;
    if (const char *sb = getenv("KPEG_SUB_BITS")) {
        const long v = strtol(sb, nullptr, 10);
        if (v >= 64 && v <= 1024 && (v & (v - 1)) == 0) {
            ctx->sub_bits = (uint32_t)v;
            ctx->sub_bits_auto = false;
        }
    }
    if (const char *nr = getenv("KPEG_NO_RECORDS"))
        ctx->use_records = !(nr[0] == '1');
    if (const char *e = getenv("KPEG_GUARD"))
        ctx->guard = e[0] == '1';
    if (const char *e = getenv("KPEG_SPLIT"))
        ctx->split_parts = std::max(1, std::min(NLANES, atoi(e)));
    if (const char *e = getenv("KPEG_SUBMIT_SPLIT"))
        ctx->submit_parts = std::max(1, std::min(NLANES, atoi(e)));
    if (const char *e = getenv("KPEG_HOST_CHUNKS"))
        ctx->host_chunks = std::max(1, std::min(64, atoi(e)));
    if (const char *e = getenv("KPEG_BANDS"))
        ctx->band_parts = std::max(1, std::min(NLANES, atoi(e)));
    if (const char *e = getenv("KPEG_RELAY_ROUND2_WIDE"))
        ctx->relay_round2_wide = e[0] != '0';
    if (const char *e = getenv("KPEG_D2H_CHAIN"))
        ctx->d2h_chain = e[0] != '0';
    cudaEventCreateWithFlags(&ctx->d2h_done, cudaEventDisableTiming);
    if (const char *rr = getenv("KPEG_RELAY_ROUNDS")) {
        const long v = strtol(rr, nullptr, 10);
        if (v >= 2 && v < MAX_RELAY_ROUNDS)
            ctx->relay_rounds = (int)v;
    }
    // 8 RSTn separators for packed batches
    cudaMallocHost(&ctx->h_sep.p, 64);
    if (ctx->h_sep.p) {
        ctx->h_sep.cap = 64;
        uint8_t *sep = (uint8_t *)ctx->h_sep.p;
        for (int k = 0; k < 8; ++k) {
            sep[2 * k] = 0xFF;
            sep[2 * k + 1] = (uint8_t)(0xD0 + k);
        }
    }
    if (cudaGetLastError() != cudaSuccess || !ctx->h_sep.p) {
        kpeg_cuda_destroy(ctx);
        return KPEG_ERR_CUDA;
    }
    *out = ctx;
    return KPEG_OK;
}

extern "C" void kpeg_cuda_destroy(kpeg_ctx *ctx)
{
    if (!ctx)
        return;
    cudaSetDevice(ctx->device);
    if (ctx->counted)
        kernels_context_destroyed();
    for (Lane &L : ctx->lane) // the members free the buffers: nothing may still use one
        if (L.stream)
            cudaStreamSynchronize(L.stream);
    delete ctx;
}

extern "C" const char *kpeg_cuda_last_error(const kpeg_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }

extern "C" int kpeg_cuda_set_profiling(kpeg_ctx *ctx, int on)
{
    if (!ctx)
        return KPEG_ERR_ARG;
    ctx->profiling = on != 0;
    return KPEG_OK;
}

extern "C" int kpeg_cuda_set_tuning(kpeg_ctx *ctx, int sub_bits, int relay_rounds)
{
    if (!ctx)
        return KPEG_ERR_ARG;
    if (sub_bits > 0) {
        if (sub_bits < 64 || sub_bits > 1024 || (sub_bits & (sub_bits - 1)))
            return KPEG_ERR_ARG; // power of two: the kernels address the staged stream with shifts
        ctx->sub_bits = (uint32_t)sub_bits;
        ctx->sub_bits_auto = false;
    } else if (sub_bits < 0) {
        ctx->sub_bits_auto = true; // back to the size chosen per job
    }
    if (relay_rounds > 0) {
        if (relay_rounds < 2 || relay_rounds >= MAX_RELAY_ROUNDS)
            return KPEG_ERR_ARG;
        ctx->relay_rounds = relay_rounds;
    }
    return KPEG_OK;
}

extern "C" void *kpeg_cuda_stream(kpeg_ctx *ctx) { return ctx ? (void *)ctx->lane[0].stream : nullptr; }

extern "C" void *kpeg_cuda_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { // pinned for every device's context
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

extern "C" int kpeg_cuda_host_register(void *p, size_t bytes)
{
    if (!p || !bytes)
        return KPEG_ERR_ARG;
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) {
        cudaGetLastError();
        return KPEG_ERR_CUDA;
    }
    return KPEG_OK;
}

extern "C" void kpeg_cuda_host_unregister(void *p)
{
    if (p && cudaHostUnregister(p) != cudaSuccess)
        cudaGetLastError();
}

extern "C" void kpeg_cuda_host_free(void *p)
{
    if (p)
        cudaFreeHost(p);
}

extern "C" void *kpeg_cuda_device_alloc(kpeg_ctx *ctx, size_t bytes)
{
    if (!ctx)
        return nullptr;
    cudaSetDevice(ctx->device);
    void *p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

extern "C" void kpeg_cuda_device_free(kpeg_ctx *ctx, void *p)
{
    if (ctx && p) {
        cudaSetDevice(ctx->device);
        for (Lane &L : ctx->lane)
            cudaStreamSynchronize(L.stream);
        cudaFree(p);
    }
}

extern "C" int kpeg_cuda_memcpy_h2d(kpeg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    if (!ctx)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->lane[0].stream));
    CK(cudaStreamSynchronize(ctx->lane[0].stream));
    return KPEG_OK;
}

extern "C" int kpeg_cuda_memcpy_d2h(kpeg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    if (!ctx)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->lane[0].stream));
    CK(cudaStreamSynchronize(ctx->lane[0].stream));
    return KPEG_OK;
}

extern "C" int kpeg_cuda_decode_device(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *d_scan, size_t scan_len,
                                       uint8_t *d_pixels_out, kpeg_stats *stats)
{
    if (!ctx || !plan || !d_scan || !d_pixels_out)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    mark(ctx, ctx->lane[0], -1);
    TRY(job_enqueue(ctx, 0, plan, d_scan, scan_len, 1, d_pixels_out, {}));
    return job_finish(ctx, 0, stats);
}

extern "C" int kpeg_cuda_decode(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len,
                                uint8_t *pixels_out, kpeg_stats *stats)
{
    if (!ctx || !plan || !scan || !pixels_out)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    Lane &L = idle_lane0(ctx);
    // bands pay off for a large image whatever its output size: the decision is taken on the full-size pixels
    const size_t full_pix = (size_t)plan->width * plan->height * plan->ncomp;
    const size_t npix = out_of(plan).bytes();
    if (ctx->band_parts > 1 && plan->restart_interval != 0 && full_pix >= ((size_t)64 << 20)) {
        const int brc = decode_banded(ctx, plan, scan, scan_len, pixels_out, stats);
        if (brc != KPEG_ERR_UNSUPPORTED) // UNSUPPORTED: the restart interval does not line up with MCU rows -- whole image below
            return brc;
    }
    TRY(ensure(ctx, L.stream, L.pixels, npix + 64));
    return decode_host_scan(ctx, plan, scan, scan_len, (uint8_t *)L.pixels.p, {Copy{pixels_out, L.pixels.p, npix}}, nullptr, stats);
}

// Batch stream format: the n stuffed scans back to back, each followed by one 2-byte RSTn marker
// (FF D0+(i&7)); to K0 an image boundary is then just another restart boundary.
extern "C" size_t kpeg_batch_packed_size(int n, const size_t *scan_lens)
{
    size_t t = 0;
    for (int i = 0; i < n; ++i)
        t += scan_lens[i] + 2;
    return t;
}

extern "C" int kpeg_batch_pack(int n, const uint8_t *const *scans, const size_t *scan_lens, uint8_t *dst, size_t cap)
{
    size_t o = 0;
    for (int i = 0; i < n; ++i) {
        if (o + scan_lens[i] + 2 > cap)
            return KPEG_ERR_ARG;
        memcpy(dst + o, scans[i], scan_lens[i]);
        o += scan_lens[i];
        dst[o++] = 0xFF;
        dst[o++] = (uint8_t)(0xD0 + (i & 7));
    }
    return KPEG_OK;
}

extern "C" int kpeg_cuda_decode_batch_packed_device(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_packed,
                                                    size_t packed_len, uint8_t *d_pixels_out, kpeg_stats *stats)
{
    if (!ctx || !plan || n <= 0 || !d_packed || !d_pixels_out)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    mark(ctx, ctx->lane[0], -1);
    TRY(job_enqueue(ctx, 0, plan, d_packed, packed_len, (uint32_t)n, d_pixels_out, {}));
    return job_finish(ctx, 0, stats);
}

// Same, with the offsets of the n scans inside the packed stream (packed_offsets[n] = its length): the
// batch is decoded as up to four concurrent jobs, one per lane, so the latency-bound phases of one part
// (late relay rounds, record expansion) overlap the issue-bound phases of the others.
extern "C" int kpeg_cuda_decode_batch_packed_device_split(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_packed,
                                                          const uint64_t *packed_offsets, uint8_t *d_pixels_out,
                                                          kpeg_stats *stats)
{
    if (!ctx || !plan || n <= 0 || !d_packed || !packed_offsets || !d_pixels_out)
        return KPEG_ERR_ARG;
    if (n < 2 || ctx->profiling) // per-kernel event times are only meaningful without a concurrent lane
        return kpeg_cuda_decode_batch_packed_device(ctx, plan, n, d_packed, (size_t)(packed_offsets[n] - packed_offsets[0]),
                                                    d_pixels_out, stats);
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    const size_t npix = out_of(plan).bytes();
    const int parts = std::max(1, std::min({n, NLANES, ctx->split_parts}));
    for (int li = 0; li < parts; ++li) {
        const int lo = (int)((long long)n * li / parts), hi = (int)((long long)n * (li + 1) / parts);
        mark(ctx, ctx->lane[li], -1);
        const int erc = job_enqueue(ctx, li, plan, d_packed + packed_offsets[lo], (size_t)(packed_offsets[hi] - packed_offsets[lo]),
                                    (uint32_t)(hi - lo), d_pixels_out + npix * (size_t)lo, {});
        if (erc != KPEG_OK) { // the parts already enqueued hold the caller's pointers: complete them before returning
            const std::string why = ctx->err;
            for (int k = 0; k < li; ++k)
                job_finish(ctx, k, nullptr);
            ctx->err = why;
            return erc;
        }
    }
    int rc_all = KPEG_OK;
    for (int li = 0; li < parts; ++li) {
        const int rc = job_finish(ctx, li, stats);
        if (rc != KPEG_OK && (rc_all == KPEG_OK || rc_all == KPEG_ERR_STREAM))
            rc_all = rc; // every lane is completed whatever the outcome; a hard failure outranks a corrupt stream
    }
    return rc_all;
}

// Deferred form of the call above: enqueue and return.  Lanes are taken round-robin; a lane's previous job is
// completed (its status checked, the rare slow path run) only when the lane is needed again or in
// kpeg_cuda_wait, so consecutive batches overlap on the device: the latency-bound phases of one (late relay
// rounds, one-block scans, kernel tails) are filled by the wide kernels of another.  d_packed and
// d_pixels_out must stay valid until kpeg_cuda_wait returns.
extern "C" int kpeg_cuda_submit_batch_packed_device(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_packed,
                                                    const uint64_t *packed_offsets, uint8_t *d_pixels_out)
{
    if (!ctx || !plan || n <= 0 || !d_packed || !packed_offsets || !d_pixels_out)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const size_t npix = out_of(plan).bytes();
    // consecutive submissions already overlap; cutting one further only shortens its kernels (measured)
    const int parts = ctx->profiling ? 1 : std::max(1, std::min({n, NLANES, ctx->submit_parts}));
    for (int k = 0; k < parts; ++k) {
        const int lo = (int)((long long)n * k / parts), hi = (int)((long long)n * (k + 1) / parts);
        const int li = ctx->next_lane;
        ctx->next_lane = (ctx->next_lane + 1) % NLANES;
        if (ctx->lane[li].job.active)
            finish_deferred(ctx, li);
        mark(ctx, ctx->lane[li], -1);
        TRY(job_enqueue(ctx, li, plan, d_packed + packed_offsets[lo], (size_t)(packed_offsets[hi] - packed_offsets[lo]),
                        (uint32_t)(hi - lo), d_pixels_out + npix * (size_t)lo, {}));
    }
    return KPEG_OK;
}

// Complete everything submitted since the last wait.  Returns the first failure among those jobs (its text
// in kpeg_cuda_last_error); *stats receives their accumulated figures.
extern "C" int kpeg_cuda_wait(kpeg_ctx *ctx, kpeg_stats *stats)
{
    if (!ctx)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    for (int k = 0; k < NLANES; ++k) { // oldest submission first
        const int li = (ctx->next_lane + k) % NLANES;
        if (ctx->lane[li].job.active)
            finish_deferred(ctx, li);
    }
    if (stats)
        *stats = ctx->deferred_stats;
    const int rc = ctx->deferred_rc;
    if (rc != KPEG_OK)
        ctx->err = ctx->deferred_err;
    reset_deferred(ctx);
    return rc;
}

extern "C" int kpeg_cuda_decode_batch_device(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_scans,
                                             const uint64_t *scan_offsets, uint8_t *d_pixels_out, kpeg_stats *stats)
{
    // Device-resident scans without separators: re-pack on the device with n small copies.
    if (!ctx || !plan || n <= 0 || !d_scans || !scan_offsets || !d_pixels_out)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    Lane &L = idle_lane0(ctx);
    const size_t total = (size_t)(scan_offsets[n] - scan_offsets[0]) + 2u * (size_t)n;
    TRY(ensure(ctx, L.stream, L.scan, total + 64));
    const uint8_t *sep = (const uint8_t *)ctx->h_sep.p;
    size_t o = 0;
    mark(ctx, L, -1);
    for (int i = 0; i < n; ++i) {
        const size_t len = (size_t)(scan_offsets[i + 1] - scan_offsets[i]);
        CK(cudaMemcpyAsync((uint8_t *)L.scan.p + o, d_scans + scan_offsets[i], len, cudaMemcpyDeviceToDevice, L.stream));
        o += len;
        CK(cudaMemcpyAsync((uint8_t *)L.scan.p + o, sep + 2 * (i & 7), 2, cudaMemcpyHostToDevice, L.stream));
        o += 2;
    }
    mark(ctx, L, KPEG_T_H2D);
    TRY(job_enqueue(ctx, 0, plan, (const uint8_t *)L.scan.p, total, (uint32_t)n, d_pixels_out, {}));
    return job_finish(ctx, 0, stats);
}

// Host-pointer batch, deferred.  Scans go straight from the caller's (ideally pinned) buffers into a lane's
// packed stream (no host-side packing pass); a batch large enough for it to matter is cut into chunks that
// rotate through the lanes, so copies in, kernels and copies out of different chunks -- and of consecutive
// submissions -- overlap.  The end-to-end path is bound by the copy out (3 bytes per pixel over PCIe): the
// point is to keep that copy engine busy from the first chunk to the last.
extern "C" int kpeg_cuda_submit_batch(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *const *scans,
                                      const size_t *scan_lens, uint8_t *const *pixels_out)
{
    if (!ctx || !plan || n <= 0 || !scans || !scan_lens || !pixels_out)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const size_t npix = out_of(plan).bytes(); // per output image
    // chunking: pipeline only when the pixel traffic is worth it (>= 32 MB); chunks of about 8 MB of pixels
    // or more each, at most host_chunks of them
    int per_chunk = n;
    if (n >= 2 && npix * (size_t)n >= (32u << 20)) {
        const int min_imgs = (int)std::max<size_t>(1, (8u << 20) / std::max<size_t>(npix, 1));
        per_chunk = std::max(min_imgs, (n + ctx->host_chunks - 1) / ctx->host_chunks);
    }
    const int nchunks = (n + per_chunk - 1) / per_chunk;
    for (int c = 0; c < nchunks; ++c) {
        const int li = ctx->next_lane;
        ctx->next_lane = (ctx->next_lane + 1) % NLANES;
        Lane &L = ctx->lane[li];
        if (L.job.active) // the lane's previous chunk must be complete before its buffers are reused
            finish_deferred(ctx, li);
        const int i0 = c * per_chunk, i1 = std::min(n, i0 + per_chunk), m = i1 - i0;
        size_t total = 0;
        for (int i = i0; i < i1; ++i)
            total += scan_lens[i] + 2;
        TRY(ensure(ctx, L.stream, L.scan, total + 64));
        TRY(ensure(ctx, L.stream, L.pixels, npix * (size_t)m + 64));
        // Copies in.  A cudaMemcpyAsync costs the host a couple of microseconds whatever its size, so (1) the 2-byte
        // separators are written by a kernel from a table of positions (one small copy per chunk), (2) runs of small
        // scans are gathered in pinned staging memory first and go over as one copy, (3) large scans go straight
        // from the caller's buffer.  With 4096 images of 512x512 this is ~4k copy calls less per batch.
        constexpr size_t SMALL_SCAN = 24u << 10;
        size_t small_bytes = 0;
        for (int i = i0; i < i1; ++i)
            if (scan_lens[i] < SMALL_SCAN)
                small_bytes += scan_lens[i] + 2;
        TRY(ensure_pinned(ctx, L.stream, L.h_ends, (size_t)m * sizeof(uint64_t)));
        TRY(ensure(ctx, L.stream, L.d_ends, (size_t)m * sizeof(uint64_t)));
        if (small_bytes)
            TRY(ensure_pinned(ctx, L.stream, L.h_stage, small_bytes));
        mark(ctx, L, -1);
        uint64_t *ends = (uint64_t *)L.h_ends.p;
        // (0) scans that lie back to back in host memory (a caller that keeps its files in one arena): ONE copy of the
        // whole run into a device staging buffer, and a kernel that moves every scan to its place (the separators need
        // two bytes between scans, so the run cannot be copied to its final place directly)
        bool contiguous = m >= 2;
        for (int i = i0; contiguous && i + 1 < i1; ++i)
            contiguous = scans[i] + scan_lens[i] == scans[i + 1];
        if (contiguous) {
            const size_t run = total - 2u * (size_t)m;
            TRY(ensure(ctx, L.stream, L.d_stage, run + 64));
            size_t o = 0;
            for (int i = i0; i < i1; ++i) {
                o += scan_lens[i];
                ends[i - i0] = o;
                o += 2;
            }
            CK(cudaMemcpyAsync(L.d_stage.p, scans[i0], run, cudaMemcpyHostToDevice, L.stream));
            CK(cudaMemcpyAsync(L.d_ends.p, ends, (size_t)m * sizeof(uint64_t), cudaMemcpyHostToDevice, L.stream));
            launch_repack_scans((const uint8_t *)L.d_stage.p, (uint8_t *)L.scan.p, (const uint64_t *)L.d_ends.p, (uint32_t)m, L.stream);
        } else {
            uint8_t *stage = (uint8_t *)L.h_stage.p;
            size_t o = 0, so = 0, run_o = 0, run_so = 0; // device offset, staging offset, start of the open staged run
            auto flush_run = [&]() -> cudaError_t {
                if (so == run_so)
                    return cudaSuccess;
                const cudaError_t e = cudaMemcpyAsync((uint8_t *)L.scan.p + run_o, stage + run_so, so - run_so, cudaMemcpyHostToDevice, L.stream);
                run_so = so;
                return e;
            };
            for (int i = i0; i < i1; ++i) {
                if (scan_lens[i] < SMALL_SCAN) {
                    if (so == run_so)
                        run_o = o;
                    memcpy(stage + so, scans[i], scan_lens[i]);
                    so += scan_lens[i] + 2; // the separator's two bytes travel with the run; the kernel below fills them in
                } else {
                    CK(flush_run());
                    CK(cudaMemcpyAsync((uint8_t *)L.scan.p + o, scans[i], scan_lens[i], cudaMemcpyHostToDevice, L.stream));
                }
                o += scan_lens[i];
                ends[i - i0] = o;
                o += 2;
            }
            CK(flush_run());
            CK(cudaMemcpyAsync(L.d_ends.p, ends, (size_t)m * sizeof(uint64_t), cudaMemcpyHostToDevice, L.stream));
            launch_write_separators((uint8_t *)L.scan.p, (const uint64_t *)L.d_ends.p, (uint32_t)m, L.stream);
        }
        mark(ctx, L, KPEG_T_H2D);
        // Copies out: one per run of images whose host buffers follow each other (a caller that decodes into one
        // frame buffer gets ONE copy per chunk)
        std::vector<Copy> d2h;
        for (int i = i0; i < i1;) {
            int j = i + 1;
            while (j < i1 && pixels_out[j] == pixels_out[j - 1] + npix)
                ++j;
            d2h.push_back(Copy{pixels_out[i], (uint8_t *)L.pixels.p + npix * (size_t)(i - i0), npix * (size_t)(j - i)});
            i = j;
        }
        TRY(job_enqueue(ctx, li, plan, (const uint8_t *)L.scan.p, total, (uint32_t)m, (uint8_t *)L.pixels.p, std::move(d2h)));
    }
    return KPEG_OK;
}

// Host-pointer batch, complete on return: a submission followed by a wait of its own.
extern "C" int kpeg_cuda_decode_batch(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *const *scans,
                                      const size_t *scan_lens, uint8_t *const *pixels_out, kpeg_stats *stats)
{
    if (!ctx || !plan || n <= 0 || !scans || !scan_lens || !pixels_out)
        return KPEG_ERR_ARG;
    zero_stats(stats);
    finish_all_deferred(ctx);
    const DeferredOutcomeSaved saved(ctx);
    const int rc = kpeg_cuda_submit_batch(ctx, plan, n, scans, scan_lens, pixels_out);
    const int wrc = kpeg_cuda_wait(ctx, stats);
    return rc != KPEG_OK ? rc : wrc;
}

// One band of a tiled decode whose frame lives on another GPU: decode here, then one peer copy of the band's rows
// (NVLink where peer access exists, staged by the driver otherwise).  With dst_device == this context's device the
// kernels write straight into the frame.
extern "C" int kpeg_cuda_decode_to_peer(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len, int dst_device,
                                        uint8_t *d_dst, kpeg_stats *stats)
{
    if (!ctx || !plan || !scan || !d_dst || dst_device < 0)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    Lane &L = idle_lane0(ctx);
    const size_t npix = out_of(plan).bytes();
    const bool local = dst_device == ctx->device && (reinterpret_cast<uintptr_t>(d_dst) & 7u) == 0;
    if (!local) {
        TRY(ensure(ctx, L.stream, L.pixels, npix + 64));
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, ctx->device, dst_device) == cudaSuccess && can) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(dst_device, 0);
            if (e != cudaSuccess) // already enabled is fine; anything else leaves the staged path
                cudaGetLastError();
        } else {
            cudaGetLastError();
        }
    }
    std::vector<Copy> out;
    if (!local) {
        Copy c{d_dst, L.pixels.p, npix};
        c.peer = dst_device;
        out.push_back(c);
    }
    return decode_host_scan(ctx, plan, scan, scan_len, local ? d_dst : (uint8_t *)L.pixels.p, std::move(out), nullptr, stats);
}

// GPU-side PPM writer: the bytes Image::dumpRawData puts into <name>.ppm (reference src/Image.cpp:108-140: the P6
// header of Image.cpp:124-127, then the R,G,B rows) assembled in device memory, so a consumer that stores or ships the
// file from the GPU never sees a separate header/payload pair.  The payload is written by K3 itself; only the header
// (about a hundred bytes) is copied in.  The file occupies d_out[*ppm_off, *ppm_off + *ppm_len): the offset (< 16)
// keeps the payload 16-byte aligned for K3's vector stores.  One-component images are expanded to R = G = B
// (SURVEY A.8), as kpeg::JPEGDecoder::dumpRawData does on the host.
extern "C" int kpeg_cuda_decode_ppm_device(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *d_scan, size_t scan_len,
                                           uint8_t *d_out, size_t cap, size_t *ppm_off, size_t *ppm_len, kpeg_stats *stats)
{
    if (!ctx || !plan || !d_scan || !d_out || !ppm_off || !ppm_len)
        return KPEG_ERR_ARG;
    if (reinterpret_cast<uintptr_t>(d_out) & 15u)
        return fail(ctx, KPEG_ERR_ARG, "PPM buffer must be 16-byte aligned");
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    Lane &L = idle_lane0(ctx);
    char header[160];
    const OutGeom o = out_of(plan);
    const int hl = kpeg_ppm_header((int)o.width, (int)o.height, header, sizeof header);
    const size_t pad = (16u - (size_t)hl % 16u) % 16u;
    const size_t npx = (size_t)o.width * o.height;
    if (pad + (size_t)hl + npx * 3u > cap)
        return fail(ctx, KPEG_ERR_ARG, "PPM buffer too small");
    TRY(ensure_pinned(ctx, L.stream, L.h_stage, 256));
    memcpy(L.h_stage.p, header, (size_t)hl);
    uint8_t *payload = d_out + pad + (size_t)hl;
    uint8_t *k3_out = payload;
    if (plan->ncomp == 1) {
        TRY(ensure(ctx, L.stream, L.pixels, npx + 64));
        k3_out = (uint8_t *)L.pixels.p;
    }
    mark(ctx, L, -1);
    CK(cudaMemcpyAsync(d_out + pad, L.h_stage.p, (size_t)hl, cudaMemcpyHostToDevice, L.stream));
    TRY(job_enqueue(ctx, 0, plan, d_scan, scan_len, 1, k3_out, {}));
    if (plan->ncomp == 1)
        launch_gray_to_rgb((const uint8_t *)L.pixels.p, payload, npx, L.stream);
    *ppm_off = pad;
    *ppm_len = (size_t)hl + npx * 3u;
    return job_finish(ctx, 0, stats);
}

// Planar writer: interleaved R,G,B rows (K3's output) -> three planes [3][H][W] in device memory.
extern "C" int kpeg_cuda_interleaved_to_planar(kpeg_ctx *ctx, const uint8_t *d_rgb, uint8_t *d_planes, size_t npixels)
{
    if (!ctx || !d_rgb || !d_planes)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    Lane &L = idle_lane0(ctx);
    launch_rgb_to_planar(d_rgb, d_planes, npixels, L.stream);
    CK(cudaStreamSynchronize(L.stream));
    CK(cudaGetLastError());
    return KPEG_OK;
}

// A frame coded one scan per component (T.81 A.2.3).  Every scan is a one-component image with tables of its own: K0,
// K1 and K2 run on it unchanged and leave the component's coefficient tiles (DC prediction and the reference's
// DC-difference rule included: both are per component); one kernel interleaves the three tile sets into MCU order and
// K3 runs as for an interleaved file.  Synchronous, on lane 0; not a throughput path.
extern "C" int kpeg_cuda_decode_scans(kpeg_ctx *ctx, const kpeg_plan *frame, const kpeg_scan *scans, int nscans, const uint8_t *file,
                                      size_t file_len, uint8_t *pixels_out, kpeg_stats *stats)
{
    if (!ctx || !frame || !scans || nscans < 1 || !file || !pixels_out)
        return KPEG_ERR_ARG;
    for (int k = 0; k < nscans; ++k)
        if (scans[k].off > file_len || scans[k].len > file_len - scans[k].off)
            return fail(ctx, KPEG_ERR_ARG, "scan outside the file");
    if (nscans == 1 && scans[0].plan.ncomp == frame->ncomp) {
        kpeg_plan pl = scans[0].plan;
        pl.flags = frame->flags;
        return kpeg_cuda_decode(ctx, &pl, file + scans[0].off, scans[0].len, pixels_out, stats);
    }
    if (frame->ncomp != 3 || nscans != 3)
        return fail(ctx, KPEG_ERR_UNSUPPORTED, "a frame is one interleaved scan or one scan per component");
    bool seen[3] = {false, false, false};
    for (int k = 0; k < 3; ++k) {
        if (scans[k].plan.ncomp != 1 || scans[k].comp[0] > 2 || seen[scans[k].comp[0]] || scans[k].plan.width != frame->width ||
            scans[k].plan.height != frame->height)
            return fail(ctx, KPEG_ERR_ARG, "scans do not cover the frame's components once each");
        seen[scans[k].comp[0]] = true;
    }
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    finish_all_deferred(ctx);
    Lane &L = ctx->lane[0];
    cudaStream_t s = L.stream;
    JobGeom g3;
    const char *why = nullptr;
    const int grc = make_job_geom(frame, 1, ctx->sub_bits, &g3, &why);
    if (grc != KPEG_OK)
        return fail(ctx, grc, why);
    const uint32_t nstrips = (g3.mcus_per_image + IDCT_MCUS_PER_CTA - 1) / IDCT_MCUS_PER_CTA;
    const uint32_t nmcu_padded = nstrips * IDCT_MCUS_PER_CTA;
    TRY(entropy_decode_component_scans(ctx, scans, file, frame->flags, nmcu_padded, stats));
    uint32_t launches = 0;
    // the frame's tables (quantisers of the three components) for K3
    kpeg_plan fp = *frame;
    for (int c = 0; c < 3; ++c) { // K3 needs no Huffman tables, but the device tables are built from a whole plan
        fp.comp_td[c] = scans[0].plan.comp_td[0];
        fp.comp_ta[c] = scans[0].plan.comp_ta[0];
    }
    memcpy(fp.ht, scans[0].plan.ht, sizeof fp.ht);
    memcpy(fp.ht_present, scans[0].plan.ht_present, sizeof fp.ht_present);
    TRY(upload_plan(ctx, &fp));
    const OutGeom o = out_of(frame);
    const size_t npix = o.bytes();
    TRY(ensure(ctx, s, L.tiles, (size_t)nmcu_padded * 3u * 128u + 256u));
    TRY(ensure(ctx, s, L.pixels, npix + 64));
    TRY(ensure(ctx, s, L.tie_rec, (size_t)nstrips * IDCT_TIE_LIST_CAP * sizeof(uint4)));
    TRY(ensure(ctx, s, L.tie_cnt, (size_t)nstrips * sizeof(uint32_t)));
    DevMeta *d_meta = (DevMeta *)L.meta.p, *h_meta = (DevMeta *)L.h_meta.p;
    CK(cudaMemsetAsync(d_meta, 0, sizeof(DevMeta), s));
    mark(ctx, L, -1);
    launch_interleave_tiles(ctx->scan_tiles[0].p, ctx->scan_tiles[1].p, ctx->scan_tiles[2].p, L.tiles.p, nmcu_padded, s, &launches);
    CK(launch_idct(idct_args(ctx, L, g3, nstrips, L.tiles.p, (uint8_t *)L.pixels.p), s, &launches));
    mark(ctx, L, KPEG_T_IDCT);
    CK(cudaMemcpyAsync(pixels_out, L.pixels.p, npix, cudaMemcpyDeviceToHost, s));
    mark(ctx, L, KPEG_T_D2H);
    CK(cudaMemcpyAsync(h_meta, d_meta, sizeof(DevMeta), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    if (ctx->guard)
        TRY(check_guards(ctx));
    ctx->last_lane = 0;
    ctx->last_g = g3; // kpeg_cuda_read_coefficients: the interleaved tiles
    if (stats) {
        stats->width = o.width;
        stats->height = o.height;
        stats->ncomp = 3;
        stats->exact_samples += h_meta->exact_samples;
        stats->kernel_launches += launches;
        add_times(ctx, L, stats);
    }
    return KPEG_OK;
}

extern "C" int kpeg_cuda_decode_file(kpeg_ctx *ctx, const uint8_t *file, size_t len, uint32_t flags, uint8_t *pixels_out,
                                     size_t cap, kpeg_plan *plan_out, kpeg_stats *stats)
{
    if (!ctx || !file || !pixels_out)
        return KPEG_ERR_ARG;
    kpeg_plan frame;
    kpeg_scan scans[KPEG_MAX_SCANS];
    int nscans = 0;
    const int prc = kpeg_parse_jfif_scans(file, len, &frame, scans, KPEG_MAX_SCANS, &nscans);
    if (prc != KPEG_OK)
        return fail(ctx, prc, prc == KPEG_ERR_UNSUPPORTED ? "unsupported JPEG coding" : "malformed JFIF container");
    frame.flags = flags;
    if (plan_out)
        *plan_out = frame;
    if (out_of(&frame).bytes() > cap)
        return fail(ctx, KPEG_ERR_ARG, "pixel buffer too small");
    return kpeg_cuda_decode_scans(ctx, &frame, scans, nscans, file, len, pixels_out, stats);
}

// Any mix of files.  Files with identical plans (dimensions, tables, restart interval) travel together as ONE batch --
// one kernel sequence for the group -- and the groups overlap on the lanes; only when a group fails are its files
// decoded one by one, to find out which of them it was.
extern "C" int kpeg_cuda_decode_files(kpeg_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, uint32_t flags,
                                      uint8_t *const *pixels_out, const size_t *caps, kpeg_plan *plans_out, int *results,
                                      kpeg_stats *stats)
{
    if (!ctx || n <= 0 || !files || !lens || !pixels_out || !caps)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    struct File {
        kpeg_plan frame;
        kpeg_scan scans[KPEG_MAX_SCANS];
        int nscans = 0, rc = KPEG_OK, group = -1;
    };
    struct Group {
        kpeg_plan plan;
        std::vector<int> members;
        std::vector<const uint8_t *> scans;
        std::vector<size_t> lens;
        std::vector<uint8_t *> outs;
    };
    std::vector<File> fl((size_t)n);
    std::vector<Group> groups;
    std::string first_err;
    int first_rc = KPEG_OK;
    auto note = [&](int i, int rc, const char *what) {
        fl[(size_t)i].rc = rc;
        if (rc != KPEG_OK && first_rc == KPEG_OK) {
            first_rc = rc;
            first_err = std::string("file ") + std::to_string(i) + ": " + what;
        }
    };
    for (int i = 0; i < n; ++i) {
        File &f = fl[(size_t)i];
        if (!files[i] || !pixels_out[i]) {
            note(i, KPEG_ERR_ARG, "null pointer");
            continue;
        }
        const int prc = kpeg_parse_jfif_scans(files[i], lens[i], &f.frame, f.scans, KPEG_MAX_SCANS, &f.nscans);
        if (prc != KPEG_OK) {
            note(i, prc, prc == KPEG_ERR_UNSUPPORTED ? "unsupported JPEG coding" : "malformed JFIF container");
            continue;
        }
        f.frame.flags = flags;
        if (plans_out)
            plans_out[i] = f.frame;
        if (out_of(&f.frame).bytes() > caps[i]) {
            note(i, KPEG_ERR_ARG, "pixel buffer too small");
            continue;
        }
        if (f.nscans != 1)
            continue; // one scan per component: decoded on its own below
        kpeg_plan pl = f.scans[0].plan;
        pl.flags = flags;
        // a plan whose padding can decode as a symbol has no batches (job_enqueue): such files are one job each
        const bool alone = restart_padding_decodes(&pl);
        size_t g = alone ? groups.size() : 0;
        while (g < groups.size() && memcmp(&groups[g].plan, &pl, sizeof pl) != 0)
            ++g;
        if (g == groups.size()) {
            groups.emplace_back();
            groups.back().plan = pl;
        }
        f.group = (int)g;
        groups[g].members.push_back(i);
        groups[g].scans.push_back(files[i] + f.scans[0].off);
        groups[g].lens.push_back(f.scans[0].len);
        groups[g].outs.push_back(pixels_out[i]);
    }
    finish_all_deferred(ctx);
    const DeferredOutcomeSaved saved(ctx);
    // every group is submitted, then ONE wait: the groups overlap on the lanes like consecutive batches do
    int all_rc = KPEG_OK;
    for (Group &g : groups) {
        const int rc = kpeg_cuda_submit_batch(ctx, &g.plan, (int)g.members.size(), g.scans.data(), g.lens.data(), g.outs.data());
        if (all_rc == KPEG_OK)
            all_rc = rc;
    }
    {
        kpeg_stats part = {};
        const int wrc = kpeg_cuda_wait(ctx, &part);
        if (all_rc == KPEG_OK)
            all_rc = wrc;
        if (stats)
            add_stats(*stats, part);
    }
    if (all_rc != KPEG_OK) {
        // something failed, and a deferred failure does not say where: group by group, then file by file
        for (Group &g : groups) {
            reset_deferred(ctx);
            int rc = kpeg_cuda_submit_batch(ctx, &g.plan, (int)g.members.size(), g.scans.data(), g.lens.data(), g.outs.data());
            kpeg_stats part;
            const int wrc = kpeg_cuda_wait(ctx, &part);
            if (rc == KPEG_OK)
                rc = wrc;
            if (rc == KPEG_OK)
                continue;
            if (g.members.size() == 1) {
                note(g.members[0], rc, ctx->err.c_str());
                continue;
            }
            for (size_t k = 0; k < g.members.size(); ++k) {
                const int one = kpeg_cuda_decode(ctx, &g.plan, g.scans[k], g.lens[k], g.outs[k], &part);
                if (one != KPEG_OK)
                    note(g.members[k], one, ctx->err.c_str());
            }
        }
    }
    for (int i = 0; i < n; ++i) {
        File &f = fl[(size_t)i];
        if (f.rc != KPEG_OK || f.nscans == 1)
            continue;
        kpeg_stats part = {};
        const int rc = kpeg_cuda_decode_scans(ctx, &f.frame, f.scans, f.nscans, files[i], lens[i], pixels_out[i], &part);
        if (stats)
            add_stats(*stats, part);
        if (rc != KPEG_OK)
            note(i, rc, ctx->err.c_str());
    }
    if (stats) { // no stage times: the groups' jobs overlap on the lanes, so their sum is no time of this call
        memset(stats->ms, 0, sizeof stats->ms);
        stats->ms_total = 0.0f;
    }
    if (results)
        for (int i = 0; i < n; ++i)
            results[i] = fl[(size_t)i].rc;
    if (first_rc != KPEG_OK)
        ctx->err = first_err;
    return first_rc;
}

extern "C" int kpeg_cuda_read_coefficients(kpeg_ctx *ctx, int16_t *out, size_t cap)
{
    if (!ctx || !out)
        return KPEG_ERR_ARG;
    if (ctx->last_lane < 0)
        return fail(ctx, KPEG_ERR_ARG, "no decode has run on this context");
    CK(cudaSetDevice(ctx->device));
    Lane &L = ctx->lane[ctx->last_lane];
    if (L.job.active)
        return fail(ctx, KPEG_ERR_ARG, "the lane of the last decode is busy with a deferred submission");
    const size_t n = (size_t)ctx->last_g.total_blocks * 64u;
    if (cap < n)
        return fail(ctx, KPEG_ERR_ARG, "coefficient buffer too small");
    TRY(ensure(ctx, L.stream, ctx->merged, n * 2u));
    // the coefficient tiles of the lane's last job are still resident: un-bias and un-swizzle them
    launch_matrix_from_tiles(L.tiles.p, (int16_t *)ctx->merged.p, ctx->last_g.total_blocks, L.stream);
    CK(cudaMemcpyAsync(out, ctx->merged.p, n * 2u, cudaMemcpyDeviceToHost, L.stream));
    CK(cudaStreamSynchronize(L.stream));
    CK(cudaGetLastError());
    return KPEG_OK;
}

// ==================================================================================================
// Encode (csrc/encode.cu)
// ==================================================================================================

namespace {

bool encode_params_ok(const kpeg_encode_params *p)
{
    return p && p->width >= 1 && p->height >= 1 && (p->ncomp == 1 || p->ncomp == 3) && p->quality >= 1 && p->quality <= 100 &&
           (p->flags & ~(KPEG_FLAG_REF_PARITY | KPEG_FLAG_OPTIMIZE_HUFFMAN)) == 0u;
}

void enc_mark(void *user, int stage)
{
    kpeg_ctx *ctx = (kpeg_ctx *)user;
    mark(ctx, ctx->lane[0], stage);
}

bool encode_optimized(const kpeg_encode_params *p) { return (p->flags & KPEG_FLAG_OPTIMIZE_HUFFMAN) != 0u; }

// What the host writes before the kernels: the whole header with the Annex K tables, or only SOI..SOF0 when the
// optimised tables are built (and the rest of the header written) on the device.
std::vector<uint8_t> encode_host_header(const kpeg_encode_params *p)
{
    return encode_optimized(p) ? enc::file_prefix(p->width, p->height, p->ncomp, p->quality)
                               : enc::file_header(p->width, p->height, p->ncomp, p->quality, p->restart_interval);
}

// The cached encoder tables (Annex K codes, the quantisers and cosines of `quality`), rebuilt when the quality changes.
int encode_tables(kpeg_ctx *ctx, int quality)
{
    EncScratch &E = ctx->enc;
    cudaStream_t s = ctx->lane[0].stream;
    if (E.quality == quality)
        return KPEG_OK;
    CK(cudaStreamSynchronize(s)); // nothing may still read the old tables or their staging copy
    TRY(ensure_pinned(ctx, s, E.h_tables, sizeof(enc::EncTables)));
    TRY(ensure(ctx, s, E.tables, sizeof(enc::EncTables)));
    enc::build_tables(quality, (enc::EncTables *)E.h_tables.p);
    CK(cudaMemcpyAsync(E.tables.p, E.h_tables.p, sizeof(enc::EncTables), cudaMemcpyHostToDevice, s));
    E.quality = quality;
    return KPEG_OK;
}

// The encoder's scratch for geometry g, and b's pointers into it (all but pixels and the output).
int encode_scratch(kpeg_ctx *ctx, const enc::EncGeom &g, enc::EncBufs *bp)
{
    EncScratch &E = ctx->enc;
    cudaStream_t s = ctx->lane[0].stream;
    size_t sz[enc::BUF_COUNT];
    enc::scratch_sizes(g, sz);
    for (int i = 0; i < enc::BUF_COUNT; ++i)
        TRY(ensure(ctx, s, E.buf[i], sz[i] + 16));
    TRY(ensure(ctx, s, E.meta, sizeof(enc::EncMeta)));
    TRY(ensure_pinned(ctx, s, E.h_meta, sizeof(enc::EncMeta)));
    if (g.flags & KPEG_FLAG_OPTIMIZE_HUFFMAN) {
        TRY(ensure(ctx, s, E.opt_tables, sizeof(enc::EncTables)));
        TRY(ensure(ctx, s, E.hist, 4u * huff::NSYM * sizeof(uint64_t)));
    }
    enc::EncBufs &b = *bp;
    b = enc::EncBufs();
    b.tables = (const enc::EncTables *)E.tables.p;
    b.opt_tables = (enc::EncTables *)E.opt_tables.p;
    b.hist = (uint64_t *)E.hist.p;
    b.coef = (int16_t *)E.buf[enc::BUF_COEF].p;
    b.raw = (int16_t *)E.buf[enc::BUF_RAW].p;
    b.dc = (int16_t *)E.buf[enc::BUF_DC].p;
    b.has_ac = (uint8_t *)E.buf[enc::BUF_HAS_AC].p;
    b.bits = (uint32_t *)E.buf[enc::BUF_BITS].p;
    b.off = (uint64_t *)E.buf[enc::BUF_OFF].p;
    b.seg_byte = (uint64_t *)E.buf[enc::BUF_SEG].p;
    b.words = (uint32_t *)E.buf[enc::BUF_WORDS].p;
    b.agg = E.buf[enc::BUF_AGG].p;
    b.tile_ff = (uint64_t *)E.buf[enc::BUF_TILE_FF].p;
    b.meta = (enc::EncMeta *)E.meta.p;
    return KPEG_OK;
}

// Tables (per quality) and scratch, then E1..E5 on lane 0 and the read-back of the length words into h_meta.
// d_out / out_cap: the file and how many bytes may be written there; hdr_len: bytes of it the host has written.
int encode_enqueue(kpeg_ctx *ctx, int quality, const enc::EncGeom &g, const uint8_t *d_pixels, uint8_t *d_out, uint64_t out_cap,
                   uint64_t hdr_len, uint32_t *launches)
{
    EncScratch &E = ctx->enc;
    cudaStream_t s = ctx->lane[0].stream;
    TRY(encode_tables(ctx, quality));
    enc::EncBufs b;
    TRY(encode_scratch(ctx, g, &b));
    b.pixels = d_pixels;
    b.out = d_out;
    b.out_cap = out_cap;
    b.hdr_len = hdr_len;
    CK(enc::launch_encode(g, b, s, launches, enc_mark, ctx));
    CK(cudaMemcpyAsync(E.h_meta.p, E.meta.p, sizeof(enc::EncMeta), cudaMemcpyDeviceToHost, s));
    return KPEG_OK;
}

// the encoder's figures for the file of geometry g that lane 0 has coded (h_meta read back)
void encode_stats(kpeg_ctx *ctx, const enc::EncGeom &g, uint32_t launches, kpeg_stats *stats)
{
    if (!stats)
        return;
    const enc::EncMeta *m = (const enc::EncMeta *)ctx->enc.h_meta.p;
    stats->width = g.width;
    stats->height = g.height;
    stats->ncomp = g.ncomp;
    stats->scan_bytes = m->scan_len;
    stats->unstuffed_bytes = m->unstuffed;
    stats->segments = (uint32_t)g.nseg;
    stats->kernel_launches += launches;
    add_times(ctx, ctx->lane[0], stats);
}

// The end of an encode into host memory, once the coded stages are enqueued on lane 0 (h_meta's read-back included):
// *len = the file's size; when it fits in cap, the part of the header the host wrote (the whole Annex K header, or the
// prefix up to SOF0) and the rest from the device (optimised mode: the header's tail, then the scan) go to out.  Then the
// guard check and the figures; KPEG_ERR_NOMEM with too_small when the file does not fit.
int finish_encoded_file(kpeg_ctx *ctx, const std::vector<uint8_t> &hdr, const enc::EncGeom &g, uint32_t launches, uint8_t *out,
                        size_t cap, size_t *len, kpeg_stats *stats, const char *too_small)
{
    Lane &L = ctx->lane[0];
    CK(cudaStreamSynchronize(L.stream));
    CK(cudaGetLastError());
    const enc::EncMeta *m = (const enc::EncMeta *)ctx->enc.h_meta.p;
    *len = m->hdr_len + m->scan_len;
    const bool fits = *len <= cap;
    if (fits) {
        memcpy(out, hdr.data(), hdr.size());
        CK(cudaMemcpyAsync(out + hdr.size(), (const uint8_t *)ctx->enc.out.p + hdr.size(), *len - hdr.size(), cudaMemcpyDeviceToHost,
                           L.stream));
        mark(ctx, L, KPEG_T_D2H);
        CK(cudaStreamSynchronize(L.stream));
    }
    if (ctx->guard)
        TRY(check_guards(ctx));
    encode_stats(ctx, g, launches, stats);
    return fits ? KPEG_OK : fail(ctx, KPEG_ERR_NOMEM, too_small);
}

} // namespace

extern "C" size_t kpeg_encode_bound(const kpeg_encode_params *p)
{
    if (!encode_params_ok(p))
        return 0;
    return (size_t)enc::encode_bound(p->width, p->height, p->ncomp, p->quality, p->restart_interval, p->flags);
}

extern "C" int kpeg_cuda_encode(kpeg_ctx *ctx, const kpeg_encode_params *p, const uint8_t *pixels, uint8_t *jpeg_out, size_t cap,
                                size_t *jpeg_len, kpeg_stats *stats)
{
    if (!ctx || !encode_params_ok(p) || !pixels || !jpeg_out || !jpeg_len)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    finish_all_deferred(ctx);
    Lane &L = ctx->lane[0];
    EncScratch &E = ctx->enc;
    const size_t npix = (size_t)p->width * p->height * p->ncomp;
    const std::vector<uint8_t> hdr = encode_host_header(p);
    const size_t bound = (size_t)enc::encode_bound(p->width, p->height, p->ncomp, p->quality, p->restart_interval, p->flags);
    const size_t out_cap = std::min(cap, bound);
    const enc::EncGeom g = enc::geometry(p->width, p->height, p->ncomp, p->restart_interval, p->flags);
    TRY(ensure(ctx, L.stream, E.pixels, npix + 64));
    TRY(ensure(ctx, L.stream, E.out, out_cap + 64));
    mark(ctx, L, -1);
    CK(cudaMemcpyAsync(E.pixels.p, pixels, npix, cudaMemcpyHostToDevice, L.stream));
    mark(ctx, L, KPEG_T_H2D);
    uint32_t launches = 0;
    TRY(encode_enqueue(ctx, p->quality, g, (const uint8_t *)E.pixels.p, (uint8_t *)E.out.p, out_cap, hdr.size(), &launches));
    return finish_encoded_file(ctx, hdr, g, launches, jpeg_out, cap, jpeg_len, stats,
                               "output buffer smaller than the encoded file (*jpeg_len = the size needed)");
}

extern "C" int kpeg_cuda_encode_device(kpeg_ctx *ctx, const kpeg_encode_params *p, const uint8_t *d_pixels, uint8_t *d_out, size_t cap,
                                       size_t *jpeg_len, kpeg_stats *stats)
{
    if (!ctx || !encode_params_ok(p) || !d_pixels || !d_out || !jpeg_len)
        return KPEG_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    finish_all_deferred(ctx);
    Lane &L = ctx->lane[0];
    const std::vector<uint8_t> hdr = encode_host_header(p);
    const enc::EncGeom g = enc::geometry(p->width, p->height, p->ncomp, p->restart_interval, p->flags);
    mark(ctx, L, -1);
    if (cap)
        CK(cudaMemcpyAsync(d_out, hdr.data(), std::min(cap, hdr.size()), cudaMemcpyHostToDevice, L.stream));
    uint32_t launches = 0;
    TRY(encode_enqueue(ctx, p->quality, g, d_pixels, d_out, cap, hdr.size(), &launches));
    CK(cudaStreamSynchronize(L.stream));
    CK(cudaGetLastError());
    if (ctx->guard)
        TRY(check_guards(ctx));
    encode_stats(ctx, g, launches, stats);
    const enc::EncMeta *m = (const enc::EncMeta *)ctx->enc.h_meta.p;
    *jpeg_len = m->hdr_len + m->scan_len;
    if (*jpeg_len > cap)
        return fail(ctx, KPEG_ERR_NOMEM, "output buffer smaller than the encoded file (*jpeg_len = the size needed)");
    return KPEG_OK;
}

// ==================================================================================================
// Lossless transcode (csrc/transcode.cu, then the encoder's coded stages)
// ==================================================================================================

namespace {

// What the output takes from the input: size, components, each component's quantiser id and the table in force when its
// scan began, and the first scan's restart interval.  Two components that name one id with different tables (a DQT
// redefined between the scans of a frame coded one scan per component) cannot share one DQT: KPEG_ERR_UNSUPPORTED.
int transcode_input(const kpeg_plan &frame, const kpeg_scan *scans, int nscans, tc::TcInput &in, const char **why)
{
    memset(&in, 0, sizeof in);
    in.width = frame.width;
    in.height = frame.height;
    in.ncomp = frame.ncomp;
    in.restart = scans[0].plan.restart_interval;
    bool have[4] = {false, false, false, false};
    for (int k = 0; k < nscans; ++k)
        for (int j = 0; j < scans[k].plan.ncomp; ++j) {
            const int id = scans[k].plan.comp_tq[j];
            uint8_t q[64];
            for (int i = 0; i < 64; ++i)
                q[i] = (uint8_t)scans[k].plan.qt[id][i]; // 8-bit tables: the parser rejects Pq != 0
            if (have[id] && memcmp(in.qzz[id], q, 64) != 0) {
                *why = "two components use one quantiser id with different tables";
                return KPEG_ERR_UNSUPPORTED;
            }
            memcpy(in.qzz[id], q, 64);
            have[id] = true;
            in.tq[scans[k].comp[j]] = (uint8_t)id;
        }
    return KPEG_OK;
}

// parse + transcode_input + tc::plan
int transcode_plan(const uint8_t *file, size_t len, const kpeg_transcode_params *p, kpeg_plan *frame, kpeg_scan *scans, int *nscans,
                   tc::TcPlan *pl, const char **why)
{
    const int prc = kpeg_parse_jfif_scans(file, len, frame, scans, KPEG_MAX_SCANS, nscans);
    if (prc != KPEG_OK) {
        *why = prc == KPEG_ERR_UNSUPPORTED ? "unsupported JPEG coding" : "malformed JFIF container";
        return prc;
    }
    tc::TcInput in;
    TRY(transcode_input(*frame, scans, *nscans, in, why));
    return tc::plan(in, *p, *pl, why);
}

// every stage of the re-encode is reported in the slot of a decode's reconstruction
void tc_mark(void *user, int)
{
    kpeg_ctx *ctx = (kpeg_ctx *)user;
    mark(ctx, ctx->lane[0], KPEG_T_IDCT);
}

} // namespace

extern "C" size_t kpeg_transcode_bound(const uint8_t *file, size_t len, const kpeg_transcode_params *p)
{
    if (!file || !p)
        return 0;
    kpeg_plan frame;
    kpeg_scan scans[KPEG_MAX_SCANS];
    int nscans = 0;
    tc::TcPlan pl;
    const char *why = nullptr;
    if (transcode_plan(file, len, p, &frame, scans, &nscans, &pl, &why) != KPEG_OK)
        return 0;
    return (size_t)tc::bound(pl);
}

// K0..K2 in T.81 mode into lane 0's tiles (one scan per component: into the components' tiles, then interleaved), TG
// into the encoder's coefficient buffers, the range flag read back, then the encoder's coded stages and the copy-out.
extern "C" int kpeg_cuda_transcode(kpeg_ctx *ctx, const uint8_t *file, size_t len, const kpeg_transcode_params *p, uint8_t *out,
                                   size_t cap, size_t *out_len, kpeg_stats *stats)
{
    if (!ctx || !file || !p || !out || !out_len)
        return KPEG_ERR_ARG;
    kpeg_plan frame;
    kpeg_scan scans[KPEG_MAX_SCANS];
    int nscans = 0;
    tc::TcPlan pl;
    const char *why = nullptr;
    const int prc = transcode_plan(file, len, p, &frame, scans, &nscans, &pl, &why);
    if (prc != KPEG_OK)
        return fail(ctx, prc, why);
    CK(cudaSetDevice(ctx->device));
    zero_stats(stats);
    finish_all_deferred(ctx);
    Lane &L = ctx->lane[0];
    cudaStream_t s = L.stream;
    const enc::EncGeom &g = pl.g.out;
    // decode to coefficient tiles, T.81 (no F1 rule)
    const uint32_t nmcu = (uint32_t)((frame.width + 7u) / 8u) * ((frame.height + 7u) / 8u);
    const uint32_t nmcu_padded = (nmcu + IDCT_MCUS_PER_CTA - 1) / IDCT_MCUS_PER_CTA * IDCT_MCUS_PER_CTA;
    TRY(ensure(ctx, s, L.tiles, (size_t)nmcu_padded * frame.ncomp * 128u + 256u)); // job_enqueue's size: no regrowth there
    uint32_t launches = 0;
    if (nscans == 1) {
        kpeg_plan dp = scans[0].plan;
        dp.flags = 0;
        TRY(decode_host_scan(ctx, &dp, file + scans[0].off, scans[0].len, nullptr, {}, L.tiles.p, stats));
    } else {
        TRY(entropy_decode_component_scans(ctx, scans, file, 0u, nmcu_padded, stats));
        mark(ctx, L, -1);
        launch_interleave_tiles(ctx->scan_tiles[0].p, ctx->scan_tiles[1].p, ctx->scan_tiles[2].p, L.tiles.p, nmcu_padded, s, &launches);
        mark(ctx, L, KPEG_T_ENTROPY_WRITE);
        add_times(ctx, L, stats);
    }
    // TG, and the range rules checked before anything is coded
    EncScratch &E = ctx->enc;
    if (E.quality < 0)
        TRY(encode_tables(ctx, 90)); // only the Annex K codes are read, and they do not depend on the quality
    enc::EncBufs b;
    TRY(encode_scratch(ctx, g, &b));
    const bool opt = (p->flags & KPEG_FLAG_OPTIMIZE_HUFFMAN) != 0u;
    const std::vector<uint8_t> hdr = tc::header(pl, opt);
    const size_t out_cap = std::min<size_t>(cap, (size_t)tc::bound(pl));
    TRY(ensure(ctx, s, E.out, out_cap + 64));
    enc::EncMeta *d_meta = (enc::EncMeta *)E.meta.p, *h_meta = (enc::EncMeta *)E.h_meta.p;
    mark(ctx, L, -1);
    CK(cudaMemsetAsync(d_meta, 0, sizeof(enc::EncMeta), s));
    tc::launch_gather(pl.g, L.tiles.p, b.coef, b.dc, &d_meta->range_fail, s, &launches);
    mark(ctx, L, KPEG_T_IDCT);
    CK(cudaMemcpyAsync(&h_meta->range_fail, &d_meta->range_fail, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    add_times(ctx, L, stats);
    if (h_meta->range_fail)
        return fail(ctx, KPEG_ERR_UNSUPPORTED, "a DC difference or an AC coefficient of the output is beyond what baseline tables code");
    b.out = (uint8_t *)E.out.p;
    b.out_cap = out_cap;
    b.hdr_len = hdr.size();
    mark(ctx, L, -1);
    CK(enc::launch_coded_stages(g, b, b.dc, s, &launches, tc_mark, ctx));
    CK(cudaMemcpyAsync(h_meta, d_meta, sizeof(enc::EncMeta), cudaMemcpyDeviceToHost, s));
    return finish_encoded_file(ctx, hdr, g, launches, out, cap, out_len, stats,
                               "output buffer smaller than the transcoded file (*out_len = the size needed)");
}
