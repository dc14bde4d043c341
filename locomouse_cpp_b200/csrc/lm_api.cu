// lm_api.cu — the C ABI of include/locomouse_b200.h: context, per-video state, the sub-batch
// pipeline (H2D of sub-batch k+1 overlaps the kernels of sub-batch k; results return through pinned
// staging), timing and debug fetches.  No CPU fallback: every entry point needs a CUDA device.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "ffv1_format.h"
#include "mjpeg_format.h"
#include "mpeg4_format.h"
#include "lm_internal.h"

namespace {
std::string g_create_error;     // last lm_create failure (lm_last_error(NULL)); guarded by g_mutex
std::mutex g_mutex;

// Every entry point runs on its context's device and leaves the caller's current device as it found it.
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};
}

struct lm_ctx {
    int device = 0;
    static constexpr int NSLOT = 8;   // scratch sets / compute streams: sub-batch k runs in slot k % (option streams)
    cudaStream_t stream = nullptr, stream_more[NSLOT - 1] = {}, copy_stream = nullptr;
    cudaStream_t stream_hi = nullptr; // highest priority: the tensor-core screen kernels of all slots (option screen_priority)
    cudaStream_t stream_back[NSLOT] = {};  // medium priority, per slot: everything after k_prep (option back_priority)
    int opt_screen_priority = 1;
    int opt_back_priority = 0;        // 1: a sub-batch's sparse / tail / NMS / pairing / D2H outrank the min-max / crop kernels of younger sub-batches
    int opt_screen_stages = 2;        // deepest window-tile ring of k_screen2 (2..4): fewer stages leave shared memory for co-resident CTAs
    lm_config cfg{};
    bool configured = false, model_set = false, bkg_set = false, calib_set = false;
    LmGeom geom{};
    std::string err;

    // One device allocation of the context (alloc_device).  In guard mode it sits between two 4 kB regions filled with a
    // pattern, and [req, cap) holds the pattern too: an overrun is caught at the end of what was asked for.
    struct Buf {
        uint8_t *base = nullptr;      // cudaMalloc result (the leading guard region in guard mode)
        uint8_t *p = nullptr;         // usable bytes [p, p + cap)
        size_t cap = 0;
        size_t req = 0;               // bytes of the buffer placed in it
        template <typename T>
        T *as() const { return reinterpret_cast<T *>(p); }
    };
    // Context-lifetime buffers, by role: grow-only (grow()), kept across re-configuration until lm_destroy.  The folded
    // calibration (k_fold_calib: the map with the mirror folded in, the background seen through it, k_prep's run flags) is
    // rebuilt when fold_dirty is set.  lm_decode_ffv1 shares the PNG staging, offset, status and header buffers, lm_decode_mjpeg
    // and lm_decode_mpeg4 the PNG scratch (their coefficients), staging, offset and status buffers; the three
    // pass-1 entry points share their scratch, as do the two cost builders.
    enum {
        BKG, CALIB, TMPL, FOLD_CALIB = TMPL + 6, FOLD_BKG, FOLD_RUN,
        PNG_SCRATCH, PNG_STAGE0, PNG_STAGE1, PNG_OFFS, PNG_STATUS, PNG_HDR, FFV1_REC, FFV1_INIT, FFV1_SOFF, FFV1_SLEN, FFV1_CHAINS,
        FFV1_WORK0, FFV1_WORK1, MJPEG_HDR, MPEG4_VOP, MPEG4_INFO, MPEG4_LINES, MPEG4_PLANES, MPEG4_SEGS,
        P1_MINMAX, P1_LUT, P1_STAGE, P1_HIST, P1_PRED, P1_DIFF, P1_BITS0, P1_BITS1, P1_CC, P1_VMAP, P1_VMASK, P1_SLOW, P1_RUNS,
        P1_LMASK, P1_DISK, P1_BBX, P1_LIMS, P1_SUMS,
        COST_CAND, COST_NCAND, COST_PRIOR, COST_OUT, COST_JC, COST_NNZ, COST_OFFS, COST_IR, COST_PR,
        GUARD_COUNT, NBUF
    };
    Buf buf[NBUF];
    bool fold_dirty = true;
    std::vector<float> h_tmpl[2][3];  // host copies (the screen's quantisation is derived from them)
    int opt_screen = 2;               // 0: dense exact kernel only, 1: tensor-core screen, one CTA per tile, 2: CTA pairs
    int opt_subbatch = 1024;
    int opt_screen_layout = 3;        // k_screen2 job layout: bit 0 = tail shares the paw + snout job (N = 192), bit 1 = stacked y tiles
    int opt_streams = 4;              // n > 1: n consecutive sub-batches in flight on n streams, 1: strictly serial kernels
    LmScreenHost scr_info[2][3] = {};
    int t_rows[2][3] = {}, t_cols[2][3] = {};
    double t_rho[2][3] = {};

    // sub-batch scratch
    int Bcap = 0;
    LmBatch bt{};                     // config-derived fields + scratch pointers (scratch set 0)
    LmBatch bt_more[NSLOT - 1] = {};  // the same with scratch sets 1..: consecutive sub-batches overlap on their own streams
    int nsets = 0;                    // scratch sets allocated by prepare()
    int last_Bsub = 0;                // sub-batch size of the last lm_detect_batch call
    int hint_B = 0, hint_sets = 0;    // scratch capacity of the last prepare(): a re-configured context asks for at least as much
    // Scratch blocks of the sub-batch pipeline.  They outlive re-configuration: release_scratch() only marks them free and the
    // next prepare() takes, for each request, the smallest free block that is large enough (a video of the same geometry reuses
    // every block; cudaMalloc and cudaFree wait for the whole device, i.e. for every other context's work too).  Blocks that
    // stay free after a prepare() that had to allocate are returned to the driver.
    struct Block : Buf {
        bool used = false;
    };
    std::vector<Block> blocks;
    int64_t device_allocs = 0;        // cudaMalloc calls so far (lm_get_info("device_allocs"))
    // Guard mode (environment variable LM_GUARD=1 when the context is created; compute-sanitizer is not available on the pool):
    // every block and buffer sits between two 4 kB regions filled with a pattern, lm_get_info("guard_violations") counts the
    // bytes of those regions that no longer hold it, i.e. out-of-bounds WRITES of any kernel since the allocation.
    bool guard = false;
    uint8_t *d_stage[2] = {};         // staged raw frames (Bcap + 1 each) when frames come from the host
    uint32_t *d_bb[10] = {};           // [3][Bcap] per ring set
    // result staging
    struct ResOff {
        size_t n_bottom, n_side, bottom, side, match_n, match_y, match_s, tail, flags, total;
    } ro{};
    uint8_t *d_res[NSLOT] = {};       // device results for one sub-batch, per scratch set
    // Result staging, box arrays and events are kept per "ring set" (sub-batch index mod NRES), scratch and streams per slot
    // (index mod the number of slots in use): the host queues as many sub-batches ahead of the one it is copying out as
    // there are slots, so the device always has several sub-batches to overlap while the host copies results out.
    static constexpr int NRES = 10;    // > the deepest lookahead (= number of slots in use)
    uint8_t *h_res[NRES] = {};        // pinned, h_res_bytes each (grow-only)
    size_t h_res_bytes = 0;
    cudaEvent_t ev_h2d[NRES] = {}, ev_done[NRES] = {};
    cudaEvent_t ev_stage[NRES][8] = {};
    cudaEvent_t ev_call[2] = {};      // first kernel / last D2H of a whole lm_detect_batch call
    cudaEvent_t ev_mid[NRES] = {};    // between k_screen and k_corr_sparse
    cudaEvent_t ev_go[NRES] = {};     // before k_screen (hand-over to the high-priority stream)
    cudaEvent_t ev_sstart[NRES] = {}; // on the screen's stream right before k_screen2 (device timeline only)
    float ms_screen = 0.f;            // k_screen alone, summed over the sub-batches of the last call
    long long screen_macs = 0;        // int8 MACs of the last k_screen2 launch
    float ms[7] = {};
    std::vector<float> timeline;     // [sub-batch][9]: ms from the start of the last call to its stage events 0..7 and to the end of the screen kernel
    int64_t launches = 0;
    cudaEvent_t ev_png_copy[2] = {}, ev_png_done[2] = {};
    float ms_decode = 0.f;            // decode kernels of the last lm_decode_png / lm_decode_ffv1 / lm_decode_mjpeg / lm_decode_mpeg4 call
    int last_B = 0;                   // size of the last sub-batch (for lm_debug_fetch)
    int last_slot = 0;
    int64_t last_s0 = 0;
    // the last chunk of the last pass-1 call (lm_debug_fetch items 4 .. 6): method (LM_P1_*, 0: none), its frames
    // [p1_s0, p1_s0 + p1_B) of the call, bit-image rows / words per row / width, int32 sums per frame
    struct {
        int method = 0, B = 0, rows = 0, wpr = 0, width = 0, nsums = 0;
        int64_t s0 = 0;
    } p1;
};

namespace {

int fail(lm_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c)
        c->err = buf;
    else {
        std::lock_guard<std::mutex> lock(g_mutex);
        g_create_error = buf;
    }
    return code;
}

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return fail(ctx, LM_ERR_RUNTIME, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                        __LINE__);                                                                      \
    } while (0)

int ceil_half(int v) { return (int)std::ceil((double)v / 2.0); }

// LocoMouse_Model ctor (class.cpp:3157-3161) + move-assignment quirk (3172-3173, SURVEY Q11) +
// initializeFeatureLoop (672-682)
void make_geom(lm_ctx *c) {
    LmGeom &g = c->geom;
    int mbw = std::max(c->t_cols[0][0], c->t_cols[0][1]) - 1, mbh = std::max(c->t_rows[0][0], c->t_rows[0][1]) - 1;
    int msw = std::max(c->t_cols[1][0], c->t_cols[1][1]) - 1, msh = std::max(c->t_rows[1][0], c->t_rows[1][1]) - 1;
    g.spre_b_w = ceil_half(mbw);
    g.spre_b_h = ceil_half(mbh);
    g.spre_s_w = ceil_half(msw);
    g.spre_s_h = ceil_half(msh);
    g.spost_s_w = msw / 2;
    g.spost_s_h = msh / 2;
    g.spost_b_w = g.spre_b_w;
    g.spost_b_h = g.spre_b_h;
    g.pad_pre_rows = std::max(c->cfg.bb_h_side, std::max(g.spre_s_h, g.spre_b_h));
    g.pad_post_rows = std::max(g.spost_b_h, g.spost_s_h);
    g.pad_pre_cols = std::max(c->cfg.bb_w, std::max(g.spre_s_w, g.spre_b_w));
    g.pad_post_cols = std::max(g.spost_b_w, g.spost_s_w);
}

// cropBoundingBox (class.cpp:1422-1423, 1457-1458) + the cv::Mat ROI assertion the reference relies on
bool roi_ok(const lm_ctx *c, uint32_t bbx, uint32_t bbys, uint32_t bbyb) {
    const LmGeom &g = c->geom;
    const lm_config &k = c->cfg;
    const int64_t cols = (int64_t)g.pad_pre_cols + k.n_cols + g.pad_post_cols;
    const int64_t rows = (int64_t)g.pad_pre_rows + k.n_rows + g.pad_post_rows;
    {
        int64_t W = g.spre_b_w + k.bb_w + g.spost_b_w, H = g.spre_b_h + k.bb_h_bottom + g.spost_b_h;
        int64_t x = (int32_t)(bbx + (uint32_t)g.pad_pre_cols - (uint32_t)(W - g.spost_b_w) + 1u);
        int64_t y = (int32_t)(bbyb + (uint32_t)g.pad_pre_rows - (uint32_t)(H - g.spost_b_h) + 1u);
        if (x < 0 || y < 0 || x + W > cols || y + H > rows) return false;
    }
    {
        int64_t W = g.spre_s_w + k.bb_w + g.spost_s_w, H = g.spre_s_h + k.bb_h_side + g.spost_s_h;
        int64_t x = (int32_t)(bbx + (uint32_t)g.pad_pre_cols - (uint32_t)(W - g.spost_s_w) + 1u);
        int64_t y = (int32_t)(bbys + (uint32_t)g.pad_pre_rows - (uint32_t)(H - g.spost_s_h) + 1u);
        if (x < 0 || y < 0 || x + W > cols || y + H > rows) return false;
    }
    return true;
}

// Waits for this context's own work only (cudaDeviceSynchronize would wait for every other context on the device too).
cudaError_t sync_streams(lm_ctx *c) {
    cudaError_t e = cudaSuccess, x;
    auto one = [&](cudaStream_t s) {
        if (s && (x = cudaStreamSynchronize(s)) != cudaSuccess && e == cudaSuccess) e = x;
    };
    one(c->copy_stream);
    one(c->stream);
    for (cudaStream_t s : c->stream_more) one(s);
    one(c->stream_hi);
    for (cudaStream_t s : c->stream_back) one(s);
    return e;
}

// Runs an entry point's body on the context's device.  After a failure (other than an overflow, whose call completed) nothing
// of the call may stay in flight: the caller's buffers and the context's scratch would still be in use.
template <typename F>
int entry(lm_ctx *ctx, F &&body) {
    if (!ctx) return LM_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    const int rc = body();
    if (rc != LM_OK && rc != LM_ERR_OVERFLOW) {
        sync_streams(ctx);
        cudaGetLastError();
    }
    return rc;
}

// Marks every scratch block free (the streams have been drained) and forgets the derived layout; prepare() re-derives it.
void release_scratch(lm_ctx *c) {
    for (auto &b : c->blocks) b.used = false;
    for (int s = 0; s < 2; ++s) c->d_stage[s] = nullptr;
    c->fold_dirty = true;
    for (int s = 0; s < lm_ctx::NRES; ++s) c->d_bb[s] = nullptr;
    for (int s = 0; s < lm_ctx::NSLOT; ++s) c->d_res[s] = nullptr;
    c->bt = LmBatch{};
    for (auto &b : c->bt_more) b = LmBatch{};
    c->nsets = 0;
    c->Bcap = 0;
}

// Returns the free scratch blocks to the driver (all of them after release_scratch).
void trim_scratch(lm_ctx *c) {
    std::vector<lm_ctx::Block> keep;
    for (auto &b : c->blocks)
        if (b.used) keep.push_back(b);
        else cudaFree(b.base);
    c->blocks.swap(keep);
}

constexpr size_t LM_GUARD_BYTES = 4096;
constexpr int LM_GUARD_PATTERN = 0xA5;

// The one cudaMalloc of context memory: `bytes` usable bytes (between two pattern-filled guard regions in guard mode), counted
// in device_allocs.  When the device is out of memory, the free scratch blocks go back to the driver and the allocation is
// tried once more.
int alloc_device(lm_ctx *ctx, lm_ctx::Buf &b, size_t bytes) {
    const size_t g = ctx->guard ? LM_GUARD_BYTES : 0;
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, bytes + 2 * g);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        trim_scratch(ctx);
        e = cudaMalloc(&q, bytes + 2 * g);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, LM_ERR_RUNTIME, "cannot allocate %zu bytes of device memory: %s", bytes, cudaGetErrorString(e));
    }
    ++ctx->device_allocs;
    b.base = static_cast<uint8_t *>(q);
    b.p = b.base + g;
    b.cap = b.req = bytes;
    if (g) {
        CK(cudaMemsetAsync(b.base, LM_GUARD_PATTERN, g, ctx->stream));
        CK(cudaMemsetAsync(b.p + bytes, LM_GUARD_PATTERN, g, ctx->stream));
    }
    return LM_OK;
}

// Everything the context owns on the device and in page-locked memory (lm_destroy).
void free_all(lm_ctx *c) {
    release_scratch(c);
    trim_scratch(c);
    for (auto &b : c->buf) cudaFree(b.base);
    for (int s = 0; s < lm_ctx::NRES; ++s) {
        if (c->h_res[s]) cudaFreeHost(c->h_res[s]);
        c->h_res[s] = nullptr;
    }
    c->h_res_bytes = 0;
}

// One scratch buffer of `count` T, zero-filled: a free block that is large enough (the smallest such), else a new one.
template <typename T>
int dalloc(lm_ctx *ctx, T **p, size_t count) {
    const size_t bytes = std::max<size_t>(count * sizeof(T), 256);
    lm_ctx::Block *best = nullptr;
    for (auto &b : ctx->blocks)
        if (!b.used && b.cap >= bytes && (!best || b.cap < best->cap)) best = &b;
    if (!best) {
        lm_ctx::Block nb;
        if (int rc = alloc_device(ctx, nb, bytes)) return rc;
        ctx->blocks.push_back(nb);
        best = &ctx->blocks.back();
    }
    best->used = true;
    best->req = bytes;
    // guard mode: the slack of a larger reused block is guarded like the region behind it (an overrun into it is counted)
    if (ctx->guard && best->cap > bytes) CK(cudaMemsetAsync(best->p + bytes, LM_GUARD_PATTERN, best->cap - bytes, ctx->stream));
    // fresh or reused (a reused block holds the previous video's data), every buffer starts zero-filled: results never depend
    // on whether a context was re-configured
    CK(cudaMemsetAsync(best->p, 0, bytes, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    *p = best->as<T>();
    return LM_OK;
}

// Grows a context buffer to at least `bytes` (contents are not kept; a new allocation starts zero-filled).  Growing waits for
// the context's streams, since the old allocation may still be in use.
int grow(lm_ctx *ctx, lm_ctx::Buf &b, size_t bytes) {
    bytes = std::max<size_t>(bytes, 256);
    if (b.cap >= bytes && !(ctx->guard && bytes < b.req)) {
        b.req = bytes;
        return LM_OK;
    }
    if (b.cap < bytes) {
        CK(sync_streams(ctx));
        cudaFree(b.base);
        b = lm_ctx::Buf{};
        if (int rc = alloc_device(ctx, b, bytes)) return rc;
        CK(cudaMemsetAsync(b.p, 0, bytes, ctx->stream));
    } else {  // guard mode: the bytes no longer asked for are guarded like the region behind the allocation
        CK(cudaMemsetAsync(b.p + bytes, LM_GUARD_PATTERN, b.req - bytes, ctx->stream));
        b.req = bytes;
    }
    CK(cudaStreamSynchronize(ctx->stream));  // the memsets are done before another stream writes the buffer
    return LM_OK;
}

// The folded calibration of the current background, calibration and mirror (k_fold_calib), rebuilt when fold_dirty is set;
// detection and lm_bounding_box_tm_de read it.  Every stream of the context is idle.
int fold_calib(lm_ctx *ctx) {
    if (!ctx->fold_dirty) return LM_OK;
    const lm_config &k = ctx->cfg;
    const size_t px = (size_t)k.n_rows * k.n_cols;
    auto &B = ctx->buf;
    using L = lm_ctx;
    if (int rc = grow(ctx, B[L::FOLD_CALIB], px * sizeof(int32_t))) return rc;
    if (int rc = grow(ctx, B[L::FOLD_BKG], px + 32)) return rc;  // + padding: word loads past the last pixel
    if (int rc = grow(ctx, B[L::FOLD_RUN], px)) return rc;
    CK(cudaMemsetAsync(B[L::FOLD_BKG].p + px, 0, 32, ctx->stream));  // the buffer may have held a larger image
    if (lm_launch_fold_calib(B[L::CALIB].as<int32_t>(), B[L::BKG].p, k.n_rows, k.n_cols, k.flip, B[L::FOLD_CALIB].as<int32_t>(), B[L::FOLD_BKG].p,
                             B[L::FOLD_RUN].p, ctx->stream) < 0)
        return fail(ctx, LM_ERR_RUNTIME, "calibration fold launch failed");
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->fold_dirty = false;
    return LM_OK;
}

void use_fold(const lm_ctx *ctx, LmBatch &b) {
    b.calib_flip = ctx->buf[lm_ctx::FOLD_CALIB].as<int32_t>();
    b.bkg_warp = ctx->buf[lm_ctx::FOLD_BKG].p;
    b.run_mode = ctx->buf[lm_ctx::FOLD_RUN].p;
}

__global__ void k_guard_check(const uint8_t *p, size_t n, unsigned long long *bad) {
    unsigned int c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) c += p[i] != (uint8_t)LM_GUARD_PATTERN;
    if (c) atomicAdd(bad, (unsigned long long)c);
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Builds everything the screen kernels need for the current model / geometry.  Mode 2 (CTA pairs, k_screen2) is
// tried first when requested, then mode 1 (k_screen); if neither fits the dense kernel stays in charge.
int prepare_screen(lm_ctx *ctx, LmBatch &b, int want, size_t B) {
    b.scr = LmScreen{};
    const lm_config &k = ctx->cfg;
    const size_t smem_limit = 220 * 1024;
    if (want <= 0 || k.bb_w > 1024 || std::max(k.bb_h_bottom, k.bb_h_side) > 512 || B > ((size_t)1 << 16)) return LM_OK;  // task word: frame << 16 | patch_row << 8 | patch_col
    const int nfeat = k.tail_w > 0 ? 3 : 2;
    // 1. quantisation + thresholds of every template
    for (int v = 0; v < 2; ++v)
        for (int f = 0; f < nfeat; ++f) {
            const LmTemplateDev &T = b.tmpl[v][f];
            LmScreenHost &H = ctx->scr_info[v][f];
            H = LmScreenHost{};
            if (!lm_screen_quantize(ctx->h_tmpl[v][f].data(), T.kh, T.kw, T.init, &H)) return LM_OK;
            H.dx = b.view[v].halo_x - T.ax;
            H.dy = b.view[v].halo_y - T.ay;
            if (H.dx < 0 || H.dy < 0) return LM_OK;
        }
    // 2a. CTA-pair jobs.  A spec lists, per CTA rank, the planes (template slot, digit) of its B image.
    struct Spec {
        int ntmpl, f[3];
        int nplanes;                 // planes per rank (nhalf = 32 * nplanes)
        int pl_t[2][3], pl_d[2][3];  // [rank][plane]: template slot, digit (0 hi / 1 lo)
        int narrow;                  // 1: the tail planes are last and x tiles right of the tail box skip them
        int KH, ks, rows, stages;
    };
    const Spec SPEC_PST{3, {LM_PAW, LM_SNOUT, LM_TAIL}, 3, {{0, 0, 2}, {1, 1, 2}}, {{0, 1, 0}, {0, 1, 1}}, 1, 0, 0, 0, 0};
    const Spec SPEC_PS{2, {LM_PAW, LM_SNOUT, 0}, 2, {{0, 0, 0}, {1, 1, 0}}, {{0, 1, 0}, {0, 1, 0}}, 0, 0, 0, 0, 0};
    auto single = [](int f) { return Spec{1, {f, 0, 0}, 1, {{0, 0, 0}, {0, 0, 0}}, {{0, 0, 0}, {1, 0, 0}}, 0, 0, 0, 0, 0}; };
    Spec spec[2][3] = {};
    std::vector<int8_t> img2[2][3][2];
    bool have2 = want >= 2;
    auto fit = [&](Spec &S, int v) {  // common geometry of the job's templates + the deepest ring that fits
        S.KH = 0;
        S.ks = 0;
        for (int t = 0; t < S.ntmpl; ++t) {
            const LmScreenHost &H = ctx->scr_info[v][S.f[t]];
            S.KH = std::max(S.KH, H.dy + b.tmpl[v][S.f[t]].kh);
            S.ks = std::max(S.ks, (31 + H.dx + b.tmpl[v][S.f[t]].kw + 31) / 32);
        }
        S.rows = (128 + S.KH - 1 + 7) & ~7;
        for (S.stages = std::max(2, std::min(4, ctx->opt_screen_stages)); S.stages >= 2; --S.stages)
            if (lm_screen2_smem_bytes(S.KH, S.ks, S.rows, 32 * S.nplanes, S.stages) <= smem_limit) return true;
        return false;
    };
    // cost of one tile in tensor-pipe cycles: KH * ks instructions of N/2 cycles each
    auto icost = [](int N) { return std::max(43.0, N / 2.0); };   // cycles per pair instruction (tools/umma_pair_probe.cu)
    const int nxt_box = (k.bb_w + 31) / 32, nxt_tail = (k.tail_w + 31) / 32;
    for (int v = 0; v < 2 && have2; ++v) {
        Spec ps = SPEC_PS, pst = SPEC_PST, tl = single(LM_TAIL);
        const bool ok_ps = fit(ps, v);
        const bool ok_tl = nfeat == 3 && fit(tl, v);
        bool merged = false;
        if (nfeat == 3 && (ctx->opt_screen_layout & 1) && ok_ps && ok_tl && fit(pst, v)) {
            const double sep = (double)nxt_box * ps.KH * ps.ks * icost(128) + (double)nxt_tail * tl.KH * tl.ks * icost(64);
            const double mrg = (double)pst.KH * pst.ks * (nxt_tail * icost(192) + std::max(0, nxt_box - nxt_tail) * icost(128));
            merged = mrg < sep;
        }
        if (merged) {
            spec[v][0] = pst;
        } else {
            if (ok_ps) {
                spec[v][0] = ps;
            } else {  // one template per job, hi digits in CTA 0, lo digits in CTA 1
                Spec p1 = single(LM_PAW), s1 = single(LM_SNOUT);
                if (!fit(p1, v) || !fit(s1, v)) have2 = false;
                spec[v][0] = p1;
                spec[v][2] = s1;
            }
            if (nfeat == 3) {
                if (!ok_tl) have2 = false;
                spec[v][1] = tl;
            }
        }
        for (int q = 0; q < 3 && have2; ++q) {
            const Spec &S = spec[v][q];
            if (!S.ntmpl) continue;
            for (int r = 0; r < 2 && have2; ++r) {
                img2[v][q][r].assign((size_t)S.KH * 2 * S.ks * S.nplanes * 512, 0);
                for (int g = 0; g < S.nplanes && have2; ++g) {
                    const int f = S.f[S.pl_t[r][g]];
                    const LmScreenHost &H = ctx->scr_info[v][f];
                    LmScreenHost tmp{};
                    have2 = lm_screen_build_plane(ctx->h_tmpl[v][f].data(), b.tmpl[v][f].kh, b.tmpl[v][f].kw, b.tmpl[v][f].init, H.dx, H.dy,
                                                  S.KH, S.ks, S.pl_d[r][g], g, S.nplanes, &tmp, &img2[v][q][r]);
                    if (have2 && (tmp.t_lo != H.t_lo || tmp.t_hi != H.t_hi)) have2 = false;
                }
            }
        }
    }
    // 2b. single-CTA images
    bool have1 = false;
    std::vector<int8_t> img1[2][3];
    if (!have2) {
        have1 = true;
        for (int v = 0; v < 2 && have1; ++v)
            for (int f = 0; f < nfeat && have1; ++f) {
                LmScreenHost tmp{};
                const LmTemplateDev &T = b.tmpl[v][f];
                have1 = lm_screen_build(ctx->h_tmpl[v][f].data(), T.kh, T.kw, T.init, b.view[v].halo_x, b.view[v].halo_y, k.fma_mode, &tmp,
                                        &img1[v][f]);
                if (have1) {
                    ctx->scr_info[v][f].kh = tmp.kh;
                    ctx->scr_info[v][f].ks = tmp.ks;
                    ctx->scr_info[v][f].rows = tmp.rows;
                }
            }
    }
    if (!have1 && !have2) return LM_OK;
    // 3. what k_corr_sparse needs, for both modes (the task lists belong to the scratch sets: alloc_set)
    int rc;
    for (int v = 0; v < 2; ++v)
        for (int f = 0; f < nfeat; ++f) {
            const LmScreenHost &H = ctx->scr_info[v][f];
            LmScreenJob &J = b.scr.job[v][f];
            J.kh = H.kh;
            J.ks = H.ks;
            J.dx = H.dx;
            J.dy = H.dy;
            J.rows = H.rows;
            J.t_lo = H.t_lo;
            J.t_hi = H.t_hi;
            const int ow = (f == LM_TAIL) ? k.tail_w : k.bb_w;
            J.task_cap = (int)std::min<size_t>((size_t)1 << 30, B * (size_t)((b.bb_h[v] + 1) / 2) * (size_t)((ow + 3) / 4));  // every 2x4 patch undecided
            if (have1) {
                int8_t *dimg = nullptr;
                if ((rc = dalloc(ctx, &dimg, img1[v][f].size()))) return rc;
                CK(cudaMemcpyAsync(dimg, img1[v][f].data(), img1[v][f].size(), cudaMemcpyHostToDevice, ctx->stream));
                CK(cudaStreamSynchronize(ctx->stream));
                J.Bimg = dimg;
            }
        }
    if (have2)
        for (int v = 0; v < 2; ++v)
            for (int q = 0; q < 3; ++q) {
                const Spec &S = spec[v][q];
                if (!S.ntmpl) continue;
                LmScreen2Job &J2 = b.scr.job2[v][q];
                for (int r = 0; r < 2; ++r) {
                    int8_t *dimg = nullptr;
                    if ((rc = dalloc(ctx, &dimg, img2[v][q][r].size()))) return rc;
                    CK(cudaMemcpyAsync(dimg, img2[v][q][r].data(), img2[v][q][r].size(), cudaMemcpyHostToDevice, ctx->stream));
                    CK(cudaStreamSynchronize(ctx->stream));
                    J2.Bimg[r] = dimg;
                }
                J2.view = v;
                J2.ntmpl = S.ntmpl;
                J2.KH = S.KH;
                J2.ks = S.ks;
                J2.rows = S.rows;
                J2.nhalf = 32 * S.nplanes;
                J2.stages = S.stages;
                // narrow instruction: without the trailing tail planes, for x tiles right of the tail box
                J2.nhalf_narrow = S.narrow ? 32 * (S.nplanes - 1) : J2.nhalf;
                J2.narrow_x0 = S.narrow ? ((k.tail_w + 31) / 32) * 32 : INT_MAX;
                J2.ntmpl_narrow = S.narrow ? S.ntmpl - 1 : S.ntmpl;
                for (int r = 0; r < 2; ++r)
                    for (int g = 0; g < S.nplanes; ++g) {
                        const int t = S.pl_t[r][g];
                        (S.pl_d[r][g] ? J2.col_lo : J2.col_hi)[0][t] = r * J2.nhalf + 32 * g;
                        (S.pl_d[r][g] ? J2.col_lo : J2.col_hi)[1][t] = r * J2.nhalf_narrow + 32 * g;
                    }
                // stacked y tiles when the window height wastes less of a 256-row tile pair than whole tiles per frame do
                {
                    const int nytp = ((b.bb_h[v] + 127) / 128 + 1) / 2;
                    J2.stacked = (ctx->opt_screen_layout & 2) && (b.view[v].win_h % 4 == 0) && b.view[v].win_h < 256 * nytp;
                }
                for (int t = 0; t < S.ntmpl; ++t) {
                    const int f = S.f[t];
                    J2.feat[t] = f;
                    J2.t_lo[t] = b.scr.job[v][f].t_lo;
                    J2.t_hi[t] = b.scr.job[v][f].t_hi;
                    J2.task_cap[t] = b.scr.job[v][f].task_cap;
                }
            }
    b.scr.enabled = have2 ? 2 : 1;
    return LM_OK;
}

// derive window geometry + allocate scratch for sub-batches of Bcap frames
// Scratch for sub-batches of up to `want_B` frames in `want_sets` rotating sets (0: the configured sub-batch size / stream
// count).  Grows on demand and never shrinks: a short first video does not pay for (or wait for the allocation of) the
// ~2.5 GB per set that a long one uses, and a re-configured context keeps the capacity of its last videos.
int prepare_impl(lm_ctx *ctx, int want_B, int want_sets);
int alloc_set(lm_ctx *ctx, LmBatch &x, int set, size_t B);
int prepare(lm_ctx *ctx, int want_B = 0, int want_sets = 0) {
    int cap_B = ctx->opt_subbatch;
    if (const char *e = getenv("LM_SUBBATCH")) cap_B = std::max(1, atoi(e));
    const int cap_sets = std::max(2, std::min(ctx->opt_streams, (int)lm_ctx::NSLOT));
    want_B = want_B <= 0 ? cap_B : std::min(want_B, cap_B);
    want_sets = want_sets <= 0 ? cap_sets : std::max(2, std::min(want_sets, cap_sets));
    if (ctx->Bcap >= want_B && ctx->nsets >= want_sets) return LM_OK;
    // too small for this call (every stream was drained when the previous call returned), or re-derived after re-configuration
    want_B = std::min(cap_B, std::max({want_B, ctx->Bcap, ctx->hint_B}));
    want_sets = std::min(cap_sets, std::max({want_sets, ctx->nsets, ctx->hint_sets}));
    release_scratch(ctx);
    const int64_t allocs = ctx->device_allocs;
    const int rc = prepare_impl(ctx, want_B, want_sets);
    if (rc != LM_OK) return rc;
    ctx->hint_B = ctx->Bcap;
    ctx->hint_sets = ctx->nsets;
    if (ctx->device_allocs != allocs) trim_scratch(ctx);  // the geometry grew: blocks too small for it go back to the driver
    return LM_OK;
}

int prepare_impl(lm_ctx *ctx, int want_B, int want_sets) {
    const lm_config &k = ctx->cfg;
    LmBatch &b = ctx->bt;
    b = LmBatch{};
    b.vid_rows = k.vid_rows;
    b.vid_cols = k.vid_cols;
    b.n_rows = k.n_rows;
    b.n_cols = k.n_cols;
    b.frame_bytes = (int64_t)k.vid_rows * k.vid_cols;
    b.bb_w = k.bb_w;
    b.bb_h[LM_BOTTOM] = k.bb_h_bottom;
    b.bb_h[LM_SIDE] = k.bb_h_side;
    b.tail_w = k.tail_w;
    b.tail_pitch = std::max(32, (k.tail_w + 31) & ~31);  // rows start 32-byte aligned (k_tail packs 32 px per word)
    b.flip = k.flip;
    b.imadjust = k.imadjust;
    b.conn = k.conn;
    b.n_tail_points = k.n_tail_points;
    b.fma_mode = k.fma_mode;
    b.cand_cap = k.cand_cap;
    b.det_cap = k.det_cap;
    b.match_cap = k.match_cap;
    b.bkg = ctx->buf[lm_ctx::BKG].p;
    b.calib = ctx->buf[lm_ctx::CALIB].as<int32_t>();
    for (int f = 0; f < 2; ++f) b.ovlp[f] = (int)((double)ctx->t_cols[LM_BOTTOM][f] * (1 - k.min_overlap));
    for (int v = 0; v < 2; ++v) {
        LmView &V = b.view[v];
        V.box_w = k.bb_w;
        V.box_h = b.bb_h[v];
        int hx = 0, hy = 0, px = 0, py = 0;
        for (int f = 0; f < 3; ++f) {
            LmTemplateDev &T = b.tmpl[v][f];
            T.w = ctx->buf[lm_ctx::TMPL + v * 3 + f].as<float>();
            T.kh = ctx->t_rows[v][f];
            T.kw = ctx->t_cols[v][f];
            T.kwp = T.kw;
            T.ax = T.kw / 2;
            T.ay = T.kh / 2;
            T.init = (float)(-ctx->t_rho[v][f]);
            if (lm_corr_kwp(T.kw) < 0)
                return fail(ctx, LM_ERR_INVALID, "template wider than %d columns is not supported", LM_MAX_KW);
            hx = std::max(hx, T.ax);
            hy = std::max(hy, T.ay);
            px = std::max(px, T.kw - 1 - T.ax);
            py = std::max(py, T.kh - 1 - T.ay);
        }
        V.halo_x = hx;
        V.halo_y = hy;
        V.win_w = V.box_w + hx + px;
        V.win_h = (V.box_h + hy + py + 3) & ~3;  // multiple of 4: stacked y tiles of k_screen2 keep 4-row patches inside one frame
        V.win_pitch = (V.win_w + 15) & ~15;
        V.win_stride = (int64_t)V.win_pitch * V.win_h;
    }
    int dev_smem = 0;
    CK(cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    for (int v = 0; v < 2; ++v)
        for (int f = 0; f < 3; ++f) {
            size_t need = lm_corr_smem_bytes(b, v, f);
            if (need > (size_t)dev_smem)
                return fail(ctx, LM_ERR_INVALID, "box %d px wide with a %dx%d template needs %zu B of shared memory",
                            k.bb_w, ctx->t_rows[v][f], ctx->t_cols[v][f], need);
        }

    const int Bcap = want_B;
    const size_t B = (size_t)Bcap;
    int rc;
    b.cc_stride = (int64_t)std::max(b.bb_h[0], b.bb_h[1]) * std::max(b.tail_w, 1);
    for (int s = 0; s < lm_ctx::NRES; ++s)
        if ((rc = dalloc(ctx, &ctx->d_bb[s], 3 * B))) return rc;
    // results: one device block + two pinned host blocks, same sub-array order
    lm_ctx::ResOff &o = ctx->ro;
    size_t off = 0;
    o.n_bottom = off; off = align256(off + B * 2 * 4);
    o.n_side = off;   off = align256(off + B * 2 * 4);
    o.bottom = off;   off = align256(off + B * 2 * k.cand_cap * sizeof(lm_cand));
    o.side = off;     off = align256(off + B * 2 * k.cand_cap * sizeof(lm_cand));
    o.match_n = off;  off = align256(off + B * 2 * k.cand_cap * 4);
    o.match_y = off;  off = align256(off + B * 2 * k.match_cap * 4);
    o.match_s = off;  off = align256(off + B * 2 * k.match_cap * 8);
    o.tail = off;     off = align256(off + B * 3 * k.n_tail_points * 4);
    o.flags = off;    off = align256(off + B * 4);
    o.total = off;
    if (ctx->h_res_bytes < o.total) {
        for (int s = 0; s < lm_ctx::NRES; ++s) {
            if (ctx->h_res[s]) cudaFreeHost(ctx->h_res[s]);
            ctx->h_res[s] = nullptr;
        }
        ctx->h_res_bytes = 0;
        for (int s = 0; s < lm_ctx::NRES; ++s) CK(cudaMallocHost((void **)&ctx->h_res[s], o.total));
        ctx->h_res_bytes = o.total;
    }
    // ---- tensor-core screen: operand images, thresholds (falls back to the dense kernel) ----------------------
    {
        int want_screen = ctx->opt_screen;
        if (const char *e = getenv("LM_SCREEN")) want_screen = atoi(e);
        if ((rc = prepare_screen(ctx, b, want_screen, B))) return rc;
    }
    // ---- scratch sets: same geometry and operands, their own mutable buffers --------------------------------------
    ctx->nsets = want_sets;
    for (int set = 0; set < ctx->nsets; ++set) {
        LmBatch &x = set ? ctx->bt_more[set - 1] : b;
        if (set) x = b;
        if ((rc = alloc_set(ctx, x, set, B))) return rc;
    }
    ctx->Bcap = Bcap;
    return LM_OK;
}

// The mutable buffers of scratch set `set` for sub-batches of B frames (x holds the geometry and the screen's operands).
int alloc_set(lm_ctx *ctx, LmBatch &x, int set, size_t B) {
    const lm_config &k = ctx->cfg;
    int rc;
    if ((rc = dalloc(ctx, &x.minmax, (B + 1) * 2))) return rc;
    if ((rc = dalloc(ctx, &x.lut, (B + 1) * 256))) return rc;
    for (int v = 0; v < 2; ++v) {
        if ((rc = dalloc(ctx, &x.win[v], B * x.view[v].win_stride + 512))) return rc;  // slack: k_corr_sparse reads whole words past a row end
        if ((rc = dalloc(ctx, &x.tailbin[v], B * x.bb_h[v] * x.tail_pitch))) return rc;
    }
    if ((rc = dalloc(ctx, &x.tailmask, B * x.bb_h[LM_BOTTOM] * x.tail_pitch))) return rc;
    if ((rc = dalloc(ctx, &x.sidemask, B * x.bb_h[LM_SIDE] * x.tail_pitch))) return rc;
    if ((rc = dalloc(ctx, &x.cc, B * 3 * x.cc_stride))) return rc;
    if ((rc = dalloc(ctx, &x.cc_flag, B))) return rc;
    if ((rc = dalloc(ctx, &x.det, B * 4 * (size_t)k.det_cap))) return rc;
    if ((rc = dalloc(ctx, &x.det_count, B * 4))) return rc;
    if ((rc = dalloc(ctx, &x.nms_scratch, B * 2 * lm_nms_scratch_bytes(k.det_cap)))) return rc;
    // results: same sub-array order as the page-locked staging
    if ((rc = dalloc(ctx, &ctx->d_res[set], ctx->ro.total))) return rc;
    const lm_ctx::ResOff &o = ctx->ro;
    uint8_t *r = ctx->d_res[set];
    x.n_bottom = (int32_t *)(r + o.n_bottom);
    x.n_side = (int32_t *)(r + o.n_side);
    x.bottom = (lm_cand *)(r + o.bottom);
    x.side = (lm_cand *)(r + o.side);
    x.match_n = (int32_t *)(r + o.match_n);
    x.match_y = (int32_t *)(r + o.match_y);
    x.match_s = (double *)(r + o.match_s);
    x.tail = (int32_t *)(r + o.tail);
    x.flags = (uint32_t *)(r + o.flags);
    if (!x.scr.enabled) return LM_OK;
    // the screen's task lists: [view][feat] for k_screen, bound to the template slots of the CTA-pair jobs
    if ((rc = dalloc(ctx, &x.scr.ntasks, 16))) return rc;
    for (int v = 0; v < 2; ++v)
        for (int f = 0; f < 3; ++f)
            if (x.scr.job[v][f].task_cap && (rc = dalloc(ctx, &x.scr.job[v][f].tasks, (size_t)x.scr.job[v][f].task_cap))) return rc;
    for (int v = 0; v < 2; ++v)
        for (int q = 0; q < 3; ++q) {
            LmScreen2Job &J2 = x.scr.job2[v][q];
            for (int t = 0; t < J2.ntmpl; ++t) {
                J2.tasks[t] = x.scr.job[v][J2.feat[t]].tasks;
                J2.ntasks[t] = x.scr.ntasks + (v * 3 + J2.feat[t]);
            }
        }
    return LM_OK;
}

int ensure_stage(lm_ctx *ctx) {
    if (ctx->d_stage[0]) return LM_OK;
    for (int s = 0; s < 2; ++s) {
        int rc = dalloc(ctx, &ctx->d_stage[s], (size_t)(ctx->Bcap + 1) * ctx->bt.frame_bytes);
        if (rc) return rc;
    }
    return LM_OK;
}

}  // namespace

extern "C" {

int lm_abi_version(void) { return LM_ABI_VERSION; }

const char *lm_last_error(const lm_ctx *ctx) {
    if (ctx) return ctx->err.c_str();
    static thread_local std::string copy;  // the global may be rewritten by a concurrent lm_create
    std::lock_guard<std::mutex> lock(g_mutex);
    copy = g_create_error;
    return copy.c_str();
}

int lm_create(lm_ctx **out, int device) {
    lm_ctx *ctx = nullptr;
    if (!out) return fail(nullptr, LM_ERR_INVALID, "lm_create: null output pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(nullptr, LM_ERR_RUNTIME, "no CUDA device: %s (this library has no CPU fallback)",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(nullptr, LM_ERR_INVALID, "device %d out of range (%d devices)", device, n);
    DeviceGuard guard(device);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, LM_ERR_RUNTIME, "cudaSetDevice: %s", cudaGetErrorString(e));
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major != 10)
        return fail(nullptr, LM_ERR_RUNTIME, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    ctx = new lm_ctx();
    ctx->device = device;
    if (const char *g = getenv("LM_GUARD")) ctx->guard = atoi(g) != 0;
    bool streams_ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess &&
                      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int s = 0; s < lm_ctx::NSLOT - 1; ++s)
        streams_ok = streams_ok && cudaStreamCreateWithFlags(&ctx->stream_more[s], cudaStreamNonBlocking) == cudaSuccess;
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi is the numerically lowest = highest priority
        streams_ok = streams_ok && cudaStreamCreateWithPriority(&ctx->stream_hi, cudaStreamNonBlocking, hi) == cudaSuccess;
        const int mid = hi < lo ? std::min(lo, hi + (lo - hi + 1) / 2) : lo;  // between the default (lo) and the screen's (hi)
        for (int s = 0; s < lm_ctx::NSLOT; ++s)
            streams_ok = streams_ok && cudaStreamCreateWithPriority(&ctx->stream_back[s], cudaStreamNonBlocking, mid) == cudaSuccess;
    }
    if (!streams_ok) {
        delete ctx;
        return fail(nullptr, LM_ERR_RUNTIME, "cudaStreamCreate failed");
    }
    for (int s = 0; s < 2; ++s) cudaEventCreate(&ctx->ev_call[s]);
    for (int s = 0; s < lm_ctx::NRES; ++s) {
        cudaEventCreateWithFlags(&ctx->ev_h2d[s], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ctx->ev_done[s], cudaEventDisableTiming);
        for (int q = 0; q < 8; ++q) cudaEventCreate(&ctx->ev_stage[s][q]);
        cudaEventCreate(&ctx->ev_mid[s]);
        cudaEventCreateWithFlags(&ctx->ev_go[s], cudaEventDisableTiming);
        cudaEventCreate(&ctx->ev_sstart[s]);
    }
    *out = ctx;
    return LM_OK;
}

int lm_destroy(lm_ctx *ctx) {
    if (!ctx) return LM_OK;
    DeviceGuard guard(ctx->device);
    sync_streams(ctx);
    free_all(ctx);
    for (int s = 0; s < 2; ++s) cudaEventDestroy(ctx->ev_call[s]);
    for (int s = 0; s < lm_ctx::NRES; ++s) {
        cudaEventDestroy(ctx->ev_h2d[s]);
        cudaEventDestroy(ctx->ev_done[s]);
        for (int q = 0; q < 8; ++q) cudaEventDestroy(ctx->ev_stage[s][q]);
        cudaEventDestroy(ctx->ev_mid[s]);
        cudaEventDestroy(ctx->ev_go[s]);
        cudaEventDestroy(ctx->ev_sstart[s]);
    }
    cudaStreamDestroy(ctx->stream);
    for (int s = 0; s < lm_ctx::NSLOT - 1; ++s) cudaStreamDestroy(ctx->stream_more[s]);
    cudaStreamDestroy(ctx->stream_hi);
    for (int s = 0; s < lm_ctx::NSLOT; ++s) cudaStreamDestroy(ctx->stream_back[s]);
    cudaStreamDestroy(ctx->copy_stream);
    for (int s = 0; s < 2; ++s) {
        if (ctx->ev_png_copy[s]) cudaEventDestroy(ctx->ev_png_copy[s]);
        if (ctx->ev_png_done[s]) cudaEventDestroy(ctx->ev_png_done[s]);
    }
    delete ctx;
    return LM_OK;
}

int lm_configure(lm_ctx *ctx, const lm_config *cfg) {
    if (!ctx) return LM_ERR_INVALID;
    if (!cfg) return fail(ctx, LM_ERR_INVALID, "lm_configure: null config");
    const lm_config &k = *cfg;
    if (k.vid_rows <= 0 || k.vid_cols <= 0 || k.n_rows <= 0 || k.n_cols <= 0)
        return fail(ctx, LM_ERR_INVALID, "image sizes must be positive");
    if (k.bb_w <= 0 || k.bb_h_bottom <= 0 || k.bb_h_side <= 0) return fail(ctx, LM_ERR_INVALID, "box sizes must be positive");
    if (k.tail_w < 0 || k.tail_w > k.bb_w) return fail(ctx, LM_ERR_INVALID, "tail_w must be in [0, bb_w]");
    if (k.conn != 4 && k.conn != 8) return fail(ctx, LM_ERR_INVALID, "conn_comp_connectivity must be 4 or 8");
    if (k.n_tail_points <= 0 || k.n_tail_points > 256) return fail(ctx, LM_ERR_INVALID, "n_tail_points out of range");
    if (k.cand_cap <= 0 || k.cand_cap > 1024 || k.match_cap <= 0 || k.det_cap <= 0 || k.det_cap > 8192)
        return fail(ctx, LM_ERR_INVALID, "capacities: 0 < cand_cap <= 1024, 0 < det_cap <= 8192, match_cap > 0");
    if ((int64_t)k.bb_w * std::max(k.bb_h_bottom, k.bb_h_side) >= (1 << 21))
        return fail(ctx, LM_ERR_INVALID, "box too large for the connected-component key packing");
    DeviceGuard guard(ctx->device);
    CK(sync_streams(ctx));
    release_scratch(ctx);  // the allocations stay for the next video; the layout follows the new geometry
    ctx->bkg_set = ctx->calib_set = false;
    ctx->cfg = k;
    ctx->configured = true;
    if (ctx->model_set) make_geom(ctx);  // pads / canvas depend on the box sizes: a new configuration keeps the model
    return LM_OK;
}

int lm_set_model(lm_ctx *ctx, const lm_template t[2][3]) {
    if (!ctx) return LM_ERR_INVALID;
    if (!ctx->configured) return fail(ctx, LM_ERR_STATE, "lm_set_model before lm_configure");
    if (!t) return fail(ctx, LM_ERR_INVALID, "null model");
    DeviceGuard guard(ctx->device);
    CK(sync_streams(ctx));
    release_scratch(ctx);
    ctx->model_set = false;  // a failure below must not leave a half-updated model in use
    for (int v = 0; v < 2; ++v)
        for (int f = 0; f < 3; ++f) {
            const lm_template &T = t[v][f];
            if (!T.w || T.rows <= 0 || T.cols <= 0) return fail(ctx, LM_ERR_INVALID, "template [%d][%d] is empty", v, f);
            if (T.cols > LM_MAX_KW) return fail(ctx, LM_ERR_INVALID, "template [%d][%d] has %d columns (max %d)", v, f, T.cols, LM_MAX_KW);
            const size_t bytes = (size_t)T.rows * T.cols * sizeof(float);
            lm_ctx::Buf &d = ctx->buf[lm_ctx::TMPL + v * 3 + f];
            if (int rc = grow(ctx, d, bytes)) return rc;
            CK(cudaMemcpyAsync(d.p, T.w, bytes, cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            ctx->h_tmpl[v][f].assign(T.w, T.w + (size_t)T.rows * T.cols);
            ctx->t_rows[v][f] = T.rows;
            ctx->t_cols[v][f] = T.cols;
            ctx->t_rho[v][f] = T.rho;
        }
    ctx->model_set = true;
    make_geom(ctx);
    return LM_OK;
}

int lm_set_background(lm_ctx *ctx, const uint8_t *bkg) {
    if (!ctx) return LM_ERR_INVALID;
    if (!ctx->configured) return fail(ctx, LM_ERR_STATE, "lm_set_background before lm_configure");
    if (!bkg) return fail(ctx, LM_ERR_INVALID, "null background");
    DeviceGuard guard(ctx->device);
    const size_t n = (size_t)ctx->cfg.vid_rows * ctx->cfg.vid_cols;
    CK(sync_streams(ctx));
    lm_ctx::Buf &d = ctx->buf[lm_ctx::BKG];
    if (int rc = grow(ctx, d, n)) return rc;
    CK(cudaMemcpyAsync(d.p, bkg, n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->bt.bkg = d.p;
    ctx->bkg_set = true;
    ctx->fold_dirty = true;
    return LM_OK;
}

int lm_set_calibration(lm_ctx *ctx, const int32_t *map) {
    if (!ctx) return LM_ERR_INVALID;
    if (!ctx->configured) return fail(ctx, LM_ERR_STATE, "lm_set_calibration before lm_configure");
    if (!map) return fail(ctx, LM_ERR_INVALID, "null calibration map");
    const size_t n = (size_t)ctx->cfg.n_rows * ctx->cfg.n_cols;
    const int64_t lim = (int64_t)ctx->cfg.vid_rows * ctx->cfg.vid_cols;
    // validateImageVideoSize (class.cpp:512-515): indices must address the raw frame
    for (size_t i = 0; i < n; ++i)
        if (map[i] < 0 || map[i] >= lim)
            return fail(ctx, LM_ERR_RUNTIME, "Calibration mapping indices out of range (index %zu = %d, frame has %lld pixels)",
                        i, map[i], (long long)lim);
    DeviceGuard guard(ctx->device);
    CK(sync_streams(ctx));
    lm_ctx::Buf &d = ctx->buf[lm_ctx::CALIB];
    if (int rc = grow(ctx, d, n * sizeof(int32_t))) return rc;
    CK(cudaMemcpyAsync(d.p, map, n * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->bt.calib = d.as<int32_t>();
    ctx->calib_set = true;
    ctx->fold_dirty = true;
    return LM_OK;
}

int lm_get_geometry(const lm_ctx *ctx, int32_t pads[8], int32_t canvas[4]) {
    if (!ctx || !ctx->model_set) return LM_ERR_STATE;
    const LmGeom &g = ctx->geom;
    if (pads) {
        int32_t p[8] = {g.spre_b_w, g.spre_b_h, g.spost_b_w, g.spost_b_h, g.spre_s_w, g.spre_s_h, g.spost_s_w, g.spost_s_h};
        memcpy(pads, p, sizeof p);
    }
    if (canvas) {
        int32_t c[4] = {g.pad_pre_cols, g.pad_pre_rows, g.pad_post_cols, g.pad_post_rows};
        memcpy(canvas, c, sizeof c);
    }
    return LM_OK;
}

static int detect_batch_impl(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, const uint8_t *prev_frame, int64_t n,
                             int64_t first_frame_index, const uint32_t *bb_x, const uint32_t *bb_y_side,
                             const uint32_t *bb_y_bottom, lm_results *out);

int lm_detect_batch(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, const uint8_t *prev_frame, int64_t n,
                    int64_t first_frame_index, const uint32_t *bb_x, const uint32_t *bb_y_side,
                    const uint32_t *bb_y_bottom, lm_results *out) {
    return entry(ctx, [&] {
        return detect_batch_impl(ctx, frames, frames_on_device, prev_frame, n, first_frame_index, bb_x, bb_y_side, bb_y_bottom, out);
    });
}

static int detect_batch_impl(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, const uint8_t *prev_frame, int64_t n,
                             int64_t first_frame_index, const uint32_t *bb_x, const uint32_t *bb_y_side,
                             const uint32_t *bb_y_bottom, lm_results *out) {
    if (!ctx->configured || !ctx->model_set || !ctx->bkg_set || !ctx->calib_set)
        return fail(ctx, LM_ERR_STATE, "lm_detect_batch needs lm_configure, lm_set_model, lm_set_background and lm_set_calibration first");
    if (n < 0 || first_frame_index < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count or index");
    if (n == 0) return LM_OK;
    if (!frames || !bb_x || !bb_y_side || !bb_y_bottom || !out) return fail(ctx, LM_ERR_INVALID, "null argument");
    if (first_frame_index > 0 && !prev_frame)
        return fail(ctx, LM_ERR_INVALID, "prev_frame is required when first_frame_index > 0 (previous image of the velocity check)");
    const lm_config &k = ctx->cfg;
    if (out->n_frames < n || out->cand_cap != k.cand_cap || out->match_cap != k.match_cap ||
        out->n_tail_points != k.n_tail_points)
        return fail(ctx, LM_ERR_INVALID, "result buffers do not match the configuration");
    if (!out->n_bottom || !out->n_side || !out->bottom || !out->side || !out->match_n || !out->match_y || !out->match_s || !out->tail || !out->flags)
        return fail(ctx, LM_ERR_INVALID, "every array of lm_results must be allocated");
    for (int64_t f = 0; f < n; ++f)
        if (!roi_ok(ctx, bb_x[f], bb_y_side[f], bb_y_bottom[f]))
            return fail(ctx, LM_ERR_ROI, "frame %lld: bounding box (x=%u, y_side=%u, y_bottom=%u) leaves the padded image",
                        (long long)(first_frame_index + f), bb_x[f], bb_y_side[f], bb_y_bottom[f]);
    CK(cudaSetDevice(ctx->device));
    // Sub-batch size of this call.  Frames in HOST memory: the path is bound by the PCIe link, so half the configured size
    // (the first kernels start after half as many bytes, the last ones finish sooner).  A short video is cut in (at least) two
    // so that sub-batches overlap on the streams (and the second half's copy runs under the first half's kernels).
    int Bsub;
    {
        int cap = ctx->opt_subbatch;
        if (const char *e = getenv("LM_SUBBATCH")) cap = std::max(1, atoi(e));
        Bsub = cap;
        if (!frames_on_device && cap >= 128) Bsub = (cap / 2 + 63) / 64 * 64;
        if (n < 2 * (int64_t)Bsub) Bsub = (int)std::min<int64_t>(Bsub, std::max<int64_t>(64, ((n + 1) / 2 + 63) / 64 * 64));
        Bsub = std::min(Bsub, cap);
    }
    ctx->last_Bsub = Bsub;
    int rc = prepare(ctx, Bsub, (int)std::min<int64_t>(lm_ctx::NSLOT, (n + Bsub - 1) / Bsub));
    if (rc == LM_OK && !frames_on_device) rc = ensure_stage(ctx);
    if (rc) {  // a half-built scratch set (device or pinned memory ran out) is released, not leaked
        release_scratch(ctx);
        trim_scratch(ctx);
        return rc;
    }
    if ((rc = fold_calib(ctx))) return rc;  // per-video constants of k_prep / k_pair

    const int Bcap = ctx->Bcap;
    const int64_t fsz = ctx->bt.frame_bytes;
    const int64_t nsub = (n + Bsub - 1) / Bsub;
    const bool has_prev0 = first_frame_index > 0;
    for (int q = 0; q < 7; ++q) ctx->ms[q] = 0.f;
    ctx->ms_screen = 0.f;
    ctx->launches = 0;
    ctx->timeline.assign((size_t)nsub * 10, -1.f);
    const lm_ctx::ResOff &o = ctx->ro;
    const int nslot = ctx->nsets;  // scratch sets in rotation; with option streams = 1 they share one stream (strictly serial kernels)
    cudaStream_t streams[lm_ctx::NSLOT];
    for (int q = 0; q < lm_ctx::NSLOT; ++q) streams[q] = (q == 0 || ctx->opt_streams == 1) ? ctx->stream : ctx->stream_more[q - 1];
    const int lookahead = nslot;

    auto issue_h2d = [&](int64_t sub) -> int {
        const int slot = (int)(sub & 1);   // frame staging slot
        const int64_t s0 = sub * Bsub;
        const int B = (int)std::min<int64_t>(Bsub, n - s0);
        uint32_t *bb = ctx->d_bb[sub % lm_ctx::NRES];   // its last user (sub - NRES) has been drained
        CK(cudaMemcpyAsync(bb, bb_x + s0, (size_t)B * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaMemcpyAsync(bb + Bcap, bb_y_side + s0, (size_t)B * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaMemcpyAsync(bb + 2 * Bcap, bb_y_bottom + s0, (size_t)B * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        if (!frames_on_device) {
            uint8_t *stg = ctx->d_stage[slot];
            // the frame staging slot is free once the sub-batch that last used it has finished on the device
            if (sub >= 2) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_done[(sub - 2) % lm_ctx::NRES], 0));
            if (s0 > 0)  // halo = last frame of the previous sub-batch, contiguous in the caller's array
                CK(cudaMemcpyAsync(stg, frames + (s0 - 1) * fsz, (size_t)(B + 1) * fsz, cudaMemcpyHostToDevice, ctx->copy_stream));
            else {
                if (has_prev0) CK(cudaMemcpyAsync(stg, prev_frame, (size_t)fsz, cudaMemcpyHostToDevice, ctx->copy_stream));
                CK(cudaMemcpyAsync(stg + fsz, frames, (size_t)B * fsz, cudaMemcpyHostToDevice, ctx->copy_stream));
            }
        }
        CK(cudaEventRecord(ctx->ev_h2d[sub % lm_ctx::NRES], ctx->copy_stream));
        return LM_OK;
    };

    // result arrays in page-locked memory receive the D2H copies directly (no staging, no host memcpy)
    bool direct = true;
    {
        const void *arrs[9] = {out->n_bottom, out->n_side, out->bottom, out->side, out->match_n, out->match_y, out->match_s, out->tail, out->flags};
        for (const void *a : arrs) {
            cudaPointerAttributes at{};
            if (cudaPointerGetAttributes(&at, a) != cudaSuccess || at.type != cudaMemoryTypeHost) direct = false;
        }
        cudaGetLastError();
    }
    int overflow = 0;
    auto drain = [&](int64_t sub) -> int {  // wait for sub-batch `sub` and copy its results to the caller
        const int slot = (int)(sub % lm_ctx::NRES);
        const int64_t s0 = sub * Bsub;
        const int B = (int)std::min<int64_t>(Bsub, n - s0);
        CK(cudaEventSynchronize(ctx->ev_done[slot]));
        const uint8_t *h = ctx->h_res[slot];
        if (!direct) {
            memcpy(out->n_bottom + s0 * 2, h + o.n_bottom, (size_t)B * 2 * 4);
            memcpy(out->n_side + s0 * 2, h + o.n_side, (size_t)B * 2 * 4);
            memcpy(out->bottom + s0 * 2 * k.cand_cap, h + o.bottom, (size_t)B * 2 * k.cand_cap * sizeof(lm_cand));
            memcpy(out->side + s0 * 2 * k.cand_cap, h + o.side, (size_t)B * 2 * k.cand_cap * sizeof(lm_cand));
            memcpy(out->match_n + s0 * 2 * k.cand_cap, h + o.match_n, (size_t)B * 2 * k.cand_cap * 4);
            memcpy(out->match_y + s0 * 2 * k.match_cap, h + o.match_y, (size_t)B * 2 * k.match_cap * 4);
            memcpy(out->match_s + s0 * 2 * k.match_cap, h + o.match_s, (size_t)B * 2 * k.match_cap * 8);
            memcpy(out->tail + s0 * 3 * k.n_tail_points, h + o.tail, (size_t)B * 3 * k.n_tail_points * 4);
            memcpy(out->flags + s0, h + o.flags, (size_t)B * 4);
        }
        for (int i = 0; i < B; ++i)
            if (out->flags[s0 + i]) overflow = 1;
        float t;
        for (int q = 0; q < 6; ++q)
            if (cudaEventElapsedTime(&t, ctx->ev_stage[slot][q], ctx->ev_stage[slot][q + 1]) == cudaSuccess) ctx->ms[q] += t;
        if (ctx->bt.scr.enabled && cudaEventElapsedTime(&t, ctx->ev_stage[slot][2], ctx->ev_mid[slot]) == cudaSuccess) ctx->ms_screen += t;
        for (int q = 0; q < 10; ++q) {
            t = -1.f;
            if (cudaEventElapsedTime(&t, ctx->ev_call[0], q < 8 ? ctx->ev_stage[slot][q] : (q == 8 ? ctx->ev_mid[slot] : ctx->ev_sstart[slot])) != cudaSuccess) t = -1.f;
            ctx->timeline[(size_t)sub * 10 + q] = t;
        }
        cudaGetLastError();
        return LM_OK;
    };

    CK(cudaEventRecord(ctx->ev_call[0], streams[0]));
    auto issue_chain = [&](int64_t sub) -> int {  // every kernel of sub-batch `sub` + the D2H of its results
        int rc = LM_OK;
        const int slot = (int)(sub % nslot), ring = (int)(sub % lm_ctx::NRES), stg = (int)(sub & 1);
        const int64_t s0 = sub * Bsub;
        const int B = (int)std::min<int64_t>(Bsub, n - s0);
        cudaStream_t stf = streams[slot];   // front: min/max, LUT, crop
        const bool split = ctx->opt_streams > 1 && ctx->opt_back_priority;
        cudaStream_t st = split ? ctx->stream_back[slot] : stf;   // back: screen hand-over, sparse pass, tail, NMS, pairing, D2H
        LmBatch b = slot ? ctx->bt_more[slot - 1] : ctx->bt;
        use_fold(ctx, b);
        b.B = B;
        b.first_index = first_frame_index + s0;
        if (frames_on_device) {
            b.frames = frames + s0 * fsz;
            b.prev = s0 > 0 ? frames + (s0 - 1) * fsz : (has_prev0 ? prev_frame : nullptr);
        } else {
            b.frames = ctx->d_stage[stg] + fsz;
            b.prev = (s0 > 0 || has_prev0) ? ctx->d_stage[stg] : nullptr;
        }
        b.bb_x = ctx->d_bb[ring];
        b.bb_y_side = ctx->d_bb[ring] + Bcap;
        b.bb_y_bottom = ctx->d_bb[ring] + 2 * Bcap;
        b.ev_screen_done = ctx->ev_mid[ring];
        b.screen_stream = (ctx->opt_streams > 1 && ctx->opt_screen_priority) ? ctx->stream_hi : nullptr;
        b.ev_screen_go = ctx->ev_go[ring];
        b.ev_screen_start = ctx->ev_sstart[ring];
        b.screen_macs = &ctx->screen_macs;
        cudaEvent_t *ev = ctx->ev_stage[ring];
        CK(cudaStreamWaitEvent(stf, ctx->ev_h2d[ring], 0));
        // with the back phase on its own stream the slot's scratch is no longer protected by stream order alone
        if (split && sub >= nslot) CK(cudaStreamWaitEvent(stf, ctx->ev_done[(sub - nslot) % lm_ctx::NRES], 0));
        CK(cudaMemsetAsync(b.minmax, 0, (size_t)(B + 1) * 2 * 4, stf));
        CK(cudaMemsetAsync(b.det_count, 0, (size_t)B * 4 * 4, stf));
        CK(cudaMemsetAsync(b.flags, 0, (size_t)B * 4, stf));
        CK(cudaEventRecord(ev[0], stf));
        int nl;
        const int skip = lm_whatif_skip();  // timing experiments only (0 in production)
        if ((nl = (skip & 1) ? 0 : lm_launch_minmax(b, stf)) < 0) return fail(ctx, LM_ERR_RUNTIME, "minmax launch failed");
        ctx->launches += nl;
        CK(cudaEventRecord(ev[1], stf));
        if ((nl = (skip & 2) ? 0 : lm_launch_prep(b, stf)) < 0) return fail(ctx, LM_ERR_RUNTIME, "prep launch failed");
        ctx->launches += nl;
        CK(cudaEventRecord(ev[2], stf));
        if (split) CK(cudaStreamWaitEvent(st, ev[2], 0));
        nl = b.scr.enabled ? lm_launch_screen(b, st) : lm_launch_corr(b, st);
        if (nl < 0) return fail(ctx, LM_ERR_RUNTIME, "correlation launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        ctx->launches += nl;
        CK(cudaEventRecord(ev[3], st));
        if ((nl = (skip & 16) ? 0 : lm_launch_tail(b, st)) < 0) return fail(ctx, LM_ERR_RUNTIME, "tail launch failed");
        ctx->launches += nl;
        CK(cudaEventRecord(ev[4], st));
        if ((nl = (skip & 32) ? 0 : lm_launch_nms(b, st)) < 0) return fail(ctx, LM_ERR_RUNTIME, "nms launch failed");
        ctx->launches += nl;
        CK(cudaEventRecord(ev[5], st));
        if ((nl = (skip & 64) ? 0 : lm_launch_pair(b, st)) < 0) return fail(ctx, LM_ERR_RUNTIME, "pair launch failed");
        ctx->launches += nl;
        CK(cudaEventRecord(ev[6], st));
        CK(cudaGetLastError());
        if (direct) {
            const uint8_t *d = ctx->d_res[slot];
            const cudaMemcpyKind D2H = cudaMemcpyDeviceToHost;
            CK(cudaMemcpyAsync(out->n_bottom + s0 * 2, d + o.n_bottom, (size_t)B * 2 * 4, D2H, st));
            CK(cudaMemcpyAsync(out->n_side + s0 * 2, d + o.n_side, (size_t)B * 2 * 4, D2H, st));
            CK(cudaMemcpyAsync(out->bottom + s0 * 2 * k.cand_cap, d + o.bottom, (size_t)B * 2 * k.cand_cap * sizeof(lm_cand), D2H, st));
            CK(cudaMemcpyAsync(out->side + s0 * 2 * k.cand_cap, d + o.side, (size_t)B * 2 * k.cand_cap * sizeof(lm_cand), D2H, st));
            CK(cudaMemcpyAsync(out->match_n + s0 * 2 * k.cand_cap, d + o.match_n, (size_t)B * 2 * k.cand_cap * 4, D2H, st));
            CK(cudaMemcpyAsync(out->match_y + s0 * 2 * k.match_cap, d + o.match_y, (size_t)B * 2 * k.match_cap * 4, D2H, st));
            CK(cudaMemcpyAsync(out->match_s + s0 * 2 * k.match_cap, d + o.match_s, (size_t)B * 2 * k.match_cap * 8, D2H, st));
            CK(cudaMemcpyAsync(out->tail + s0 * 3 * k.n_tail_points, d + o.tail, (size_t)B * 3 * k.n_tail_points * 4, D2H, st));
            CK(cudaMemcpyAsync(out->flags + s0, d + o.flags, (size_t)B * 4, D2H, st));
        } else {
            CK(cudaMemcpyAsync(ctx->h_res[ring], ctx->d_res[slot], o.total, cudaMemcpyDeviceToHost, st));
        }
        CK(cudaEventRecord(ev[7], st));
        CK(cudaEventRecord(ctx->ev_done[ring], st));
        ctx->last_B = B;
        ctx->last_s0 = s0;
        ctx->last_slot = slot;
        return rc;
    };
    // sub-batches are queued `lookahead` ahead of the one being copied out; ring set (sub % NRES) was last drained at sub - NRES
    int64_t issued = 0;
    for (int64_t sub = 0; sub < nsub; ++sub) {
        for (; issued < nsub && issued <= sub + lookahead; ++issued) {
            if ((rc = issue_h2d(issued))) return rc;
            if ((rc = issue_chain(issued))) return rc;
        }
        if ((rc = drain(sub))) return rc;
    }
    for (int q = 1; q < nslot; ++q) CK(cudaStreamSynchronize(streams[q]));
    for (int q = 0; q < nslot; ++q) CK(cudaStreamSynchronize(ctx->stream_back[q]));
    CK(cudaEventRecord(ctx->ev_call[1], streams[0]));  // both streams are idle here: end of the whole call
    CK(cudaStreamSynchronize(streams[0]));
    {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, ctx->ev_call[0], ctx->ev_call[1]) == cudaSuccess) ctx->ms[6] = t;
    }
    if (overflow) return fail(ctx, LM_ERR_OVERFLOW, "a fixed-capacity list overflowed (see lm_results.flags); raise det_cap / cand_cap / match_cap");
    return LM_OK;
}

int lm_set_option(lm_ctx *ctx, const char *name, int64_t value) {
    if (!ctx) return LM_ERR_INVALID;
    if (!name) return fail(ctx, LM_ERR_INVALID, "lm_set_option: null name");
    DeviceGuard guard(ctx->device);
    if (!strcmp(name, "screen")) {
        if (value < 0 || value > 2) return fail(ctx, LM_ERR_INVALID, "option screen must be 0, 1 or 2");
        ctx->opt_screen = (int)value;
    } else if (!strcmp(name, "screen_layout")) {
        if (value < 0 || value > 3) return fail(ctx, LM_ERR_INVALID, "option screen_layout must be in [0, 3]");
        ctx->opt_screen_layout = (int)value;
    } else if (!strcmp(name, "screen_stages")) {
        if (value < 2 || value > 4) return fail(ctx, LM_ERR_INVALID, "option screen_stages must be in [2, 4]");
        ctx->opt_screen_stages = (int)value;
    } else if (!strcmp(name, "back_priority")) {
        ctx->opt_back_priority = value != 0;
    } else if (!strcmp(name, "screen_priority")) {
        ctx->opt_screen_priority = value != 0;
    } else if (!strcmp(name, "streams")) {
        if (value < 1 || value > lm_ctx::NSLOT) return fail(ctx, LM_ERR_INVALID, "option streams must be in [1, %d]", (int)lm_ctx::NSLOT);
        ctx->opt_streams = (int)value;
    } else if (!strcmp(name, "subbatch")) {
        if (value < 1 || value > 4096) return fail(ctx, LM_ERR_INVALID, "option subbatch must be in [1, 4096]");
        ctx->opt_subbatch = (int)value;
    } else {
        return fail(ctx, LM_ERR_INVALID, "unknown option '%s'", name);
    }
    CK(sync_streams(ctx));
    release_scratch(ctx);  // re-derived by the next lm_detect_batch
    return LM_OK;
}

int lm_get_info(const lm_ctx *ctx, const char *name, double *value) {
    if (!ctx || !name || !value) return LM_ERR_INVALID;
    if (!strcmp(name, "screen_active")) {
        *value = ctx->Bcap ? (double)ctx->bt.scr.enabled : -1.0;  // -1: not prepared yet
        return LM_OK;
    }
    if (!strncmp(name, "screen_eps_", 11) || !strncmp(name, "screen_scale_", 13)) {
        const bool eps = name[7] == 'e';
        const char *q = name + (eps ? 11 : 13);
        const int v = q[0] - '0', f = q[1] - '0';
        if (v < 0 || v > 1 || f < 0 || f > 2 || q[2]) return LM_ERR_INVALID;
        *value = eps ? ctx->scr_info[v][f].eps : ctx->scr_info[v][f].scale;
        return LM_OK;
    }
    if (!strncmp(name, "stage_t_", 8) && name[8] >= '0' && name[8] <= '1' && name[9] == '_' && name[10] >= '0' && name[10] <= '7' && !name[11]) {
        // device timeline of the last call: ms from the start of the call to stage event k of the LAST sub-batch that ran in slot s
        float t = -1.f;
        if (cudaEventElapsedTime(&t, ctx->ev_call[0], ctx->ev_stage[name[8] - '0'][name[10] - '0']) != cudaSuccess) t = -1.f;
        *value = (double)t;
        return LM_OK;
    }
    if (!strcmp(name, "screen2_merged") || !strcmp(name, "screen2_stacked")) {  // bit v: view v's pair job shares the tail / is stacked
        int m = 0;
        for (int v = 0; v < 2; ++v) {
            const LmScreen2Job &J = ctx->bt.scr.job2[v][0];
            if (ctx->Bcap && ctx->bt.scr.enabled == 2 && J.Bimg[0] && (name[8] == 'm' ? J.ntmpl == 3 : J.stacked)) m |= 1 << v;
        }
        *value = (double)m;
        return LM_OK;
    }
    if (!strncmp(name, "tl_", 3)) {  // tl_<sub>_<k>: device timeline of the last call (ms since its start), k = 0..7 stage events, 8 = screen end, 9 = screen start
        int sub = -1, q = -1;
        if (sscanf(name + 3, "%d_%d", &sub, &q) != 2 || sub < 0 || q < 0 || q > 9 || (size_t)sub * 10 + q >= ctx->timeline.size()) return LM_ERR_INVALID;
        *value = (double)ctx->timeline[(size_t)sub * 10 + q];
        return LM_OK;
    }
    if (!strcmp(name, "ms_decode")) {  // device time of the decode kernels in the last lm_decode_png / ffv1 / mjpeg / mpeg4 call
        *value = (double)ctx->ms_decode;
        return LM_OK;
    }
    if (!strcmp(name, "ms_screen")) {  // device time of k_screen alone in the last lm_detect_batch call
        *value = (double)ctx->ms_screen;
        return LM_OK;
    }
    if (!strcmp(name, "streams")) {
        *value = (double)ctx->opt_streams;
        return LM_OK;
    }
    if (!strcmp(name, "screen_macs")) {  // int8 MACs the last k_screen2 launch (one sub-batch) issued to the tensor cores
        *value = (double)ctx->screen_macs;
        return LM_OK;
    }
    if (!strcmp(name, "subbatch")) {   // frames per sub-batch of the last lm_detect_batch call (before the first: the configured size)
        *value = (double)(ctx->last_Bsub > 0 ? ctx->last_Bsub : ctx->opt_subbatch);
        return LM_OK;
    }
    if (!strcmp(name, "scratch_subbatch")) {   // capacity the scratch sets are allocated for (grows on demand)
        *value = (double)ctx->Bcap;
        return LM_OK;
    }
    if (!strcmp(name, "device_allocs")) {   // cudaMalloc calls of this context so far (each waits for the whole device)
        *value = (double)ctx->device_allocs;
        return LM_OK;
    }
    if (!strcmp(name, "guard_regions")) {
        size_t k = ctx->blocks.size();
        for (const auto &b : ctx->buf) k += b.base ? 1 : 0;
        *value = ctx->guard ? 2.0 * (double)k : 0.0;
        return LM_OK;
    }
    const bool selftest = !strcmp(name, "guard_selftest");   // positive control: three guard bytes are overwritten, counted, restored
    if (!strcmp(name, "guard_violations") || selftest) {   // bytes of the guard regions overwritten so far (-1: guard mode is off)
        if (!ctx->guard || (selftest && ctx->blocks.empty())) {
            *value = -1.0;
            return LM_OK;
        }
        DeviceGuard dg(ctx->device);
        lm_ctx *c = const_cast<lm_ctx *>(ctx);  // only its streams are used
        cudaStream_t st = c->stream;
        unsigned long long h = 0;
        if (sync_streams(c) != cudaSuccess || grow(c, c->buf[lm_ctx::GUARD_COUNT], sizeof h) != LM_OK) return LM_ERR_RUNTIME;
        unsigned long long *bad = c->buf[lm_ctx::GUARD_COUNT].as<unsigned long long>();
        uint8_t *probe = selftest ? ctx->blocks.back().p + ctx->blocks.back().req + 7 : nullptr;  // trailing guard
        cudaMemsetAsync(bad, 0, sizeof *bad, st);
        if (selftest) cudaMemsetAsync(probe, 0, 3, st);
        auto check = [&](const lm_ctx::Buf &b) {
            if (!b.base) return;
            k_guard_check<<<4, 256, 0, st>>>(b.base, LM_GUARD_BYTES, bad);
            k_guard_check<<<4, 256, 0, st>>>(b.p + b.req, b.cap - b.req + LM_GUARD_BYTES, bad);
        };
        for (const auto &b : ctx->blocks) check(b);  // retained blocks (free until the next prepare) keep their guards too
        for (const auto &b : ctx->buf) check(b);
        cudaError_t e = cudaMemcpyAsync(&h, bad, sizeof h, cudaMemcpyDeviceToHost, st);
        if (selftest) cudaMemsetAsync(probe, LM_GUARD_PATTERN, 3, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) e = cudaErrorUnknown;
        if (e != cudaSuccess) return LM_ERR_RUNTIME;
        *value = (double)h;
        return LM_OK;
    }
    // diagnostics of the sub-batch that last ran in scratch set 0 (all streams drained when lm_detect_batch returns):
    // "sparse_tasks" = 4x8 patches handed to the exact pass, "positives" = entries of the positive-pixel lists
    if (!strcmp(name, "sparse_tasks") || !strcmp(name, "positives")) {
        if (!ctx->Bcap) return LM_ERR_INVALID;
        const LmBatch &b = ctx->bt;
        DeviceGuard dg(ctx->device);
        cudaStream_t st = ctx->stream;
        auto fetch = [st](void *dst, const void *src, size_t n) {
            return cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToHost, st) == cudaSuccess && cudaStreamSynchronize(st) == cudaSuccess;
        };
        double tot = 0.0;
        if (name[0] == 's') {
            int32_t nt[8] = {};
            if (!b.scr.ntasks || !fetch(nt, b.scr.ntasks, sizeof nt)) return LM_ERR_RUNTIME;
            for (int i = 0; i < 6; ++i) tot += nt[i];
        } else {
            std::vector<int32_t> c((size_t)ctx->Bcap * 4);
            if (!fetch(c.data(), b.det_count, c.size() * sizeof(int32_t))) return LM_ERR_RUNTIME;
            for (int32_t x : c) tot += x;
        }
        *value = tot;
        return LM_OK;
    }
    return LM_ERR_INVALID;
}

// ---- pass 1 (SURVEY 8f-1): per-frame boxes, in chunks of frames ------------------------------------------------------
namespace {
int grow_bufs(lm_ctx *ctx, std::initializer_list<std::pair<int, size_t>> want) {
    for (const auto &w : want)
        if (int rc = grow(ctx, ctx->buf[w.first], w.second)) return rc;
    return LM_OK;
}

// Scratch of every pass-1 entry point for chunks of `cap` frames: min / max, the normalisation LUTs and, for frames in host
// memory, the staging buffer.
int pass1_scratch(lm_ctx *ctx, int cap, int frames_on_device) {
    using L = lm_ctx;
    ctx->p1.method = 0;  // the buffers are about to be overwritten: nothing to fetch until this call finishes
    const int64_t fsz = (int64_t)ctx->cfg.vid_rows * ctx->cfg.vid_cols;
    if (int rc = grow_bufs(ctx, {{L::P1_MINMAX, (size_t)(cap + 1) * 2 * sizeof(int32_t)}, {L::P1_LUT, (size_t)(cap + 1) * 256}})) return rc;
    return frames_on_device ? LM_OK : grow(ctx, ctx->buf[L::P1_STAGE], (size_t)cap * fsz);
}

// Frames [s0, s0 + B) of a pass-1 call as one chunk: the base class's readFrame (no imadjust: LocoMouse_TM_DE.cpp:36,
// LocoMouse_class.cpp:622, LocoMouse_TM.cpp:138) on the caller's device frames or on a copy of its host frames (the staging
// buffer is reused: stream order makes the copy wait for the previous chunk's kernels).
int pass1_chunk(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, int64_t s0, int B, LmBatch &b) {
    const lm_config &k = ctx->cfg;
    const int64_t fsz = (int64_t)k.vid_rows * k.vid_cols;
    b = LmBatch{};
    b.B = B;
    b.frame_bytes = fsz;
    b.bkg = ctx->buf[lm_ctx::BKG].p;
    b.calib = ctx->buf[lm_ctx::CALIB].as<int32_t>();
    b.n_rows = k.n_rows;
    b.n_cols = k.n_cols;
    b.vid_rows = k.vid_rows;
    b.vid_cols = k.vid_cols;
    b.flip = k.flip;
    b.conn = k.conn;
    b.imadjust = 0;
    b.minmax = ctx->buf[lm_ctx::P1_MINMAX].as<int32_t>();
    b.lut = ctx->buf[lm_ctx::P1_LUT].p;
    if (frames_on_device) {
        b.frames = frames + s0 * fsz;
    } else {
        uint8_t *stage = ctx->buf[lm_ctx::P1_STAGE].p;
        CK(cudaMemcpyAsync(stage, frames + s0 * fsz, (size_t)B * fsz, cudaMemcpyHostToDevice, ctx->stream));
        b.frames = stage;
    }
    return LM_OK;
}

// The per-frame sums only lm_debug_fetch reads: kept for the last chunk of a call (the only one it can address), so the
// earlier chunks of a long video skip the stores (measured on a B200: storing every chunk cost pass 1 about 0.7 %).
int32_t *last_chunk_sums(lm_ctx *ctx, int64_t s0, int cap, int64_t n) { return s0 + cap >= n ? ctx->buf[lm_ctx::P1_SUMS].as<int32_t>() : nullptr; }

// Records the last chunk of a finished pass-1 call of n frames in chunks of `cap` for lm_debug_fetch items 4 .. 6.
void set_p1(lm_ctx *ctx, int method, int64_t n, int cap, int rows, int wpr, int width, int nsums) {
    auto &q = ctx->p1;
    q.method = method;
    q.s0 = (n - 1) / cap * cap;
    q.B = (int)(n - q.s0);
    q.rows = rows;
    q.wpr = wpr;
    q.width = width;
    q.nsums = nsums;
}
}  // namespace

int lm_bounding_box_tm_de(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, int64_t n, const lm_bb_de_params *p,
                          double *bb_x_raw, int32_t *lims) {
    return entry(ctx, [&]() -> int {
        if (!ctx->configured || !ctx->bkg_set || !ctx->calib_set)
            return fail(ctx, LM_ERR_STATE, "lm_bounding_box_tm_de needs lm_configure, lm_set_background and lm_set_calibration first");
        if (n < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count");
        if (n == 0) return LM_OK;
        if (!frames || !p || !bb_x_raw) return fail(ctx, LM_ERR_INVALID, "null argument");
        const lm_config &k = ctx->cfg;
        if (p->side_x < 0 || p->side_y < 0 || p->side_w <= 0 || p->side_h <= 0 || p->side_x + p->side_w > k.n_cols ||
            p->side_y + p->side_h > k.n_rows)
            return fail(ctx, LM_ERR_INVALID, "side view box (%d, %d, %d x %d) leaves the calibrated image", p->side_x, p->side_y, p->side_w,
                        p->side_h);
        if ((int64_t)p->side_w * p->side_h >= (1 << 24))
            return fail(ctx, LM_ERR_INVALID, "side view too large for the float histogram scan of imadjust_default");
        using L = lm_ctx;
        auto &S = ctx->buf;
        const int cap = 1024;  // frames per chunk: large enough that launch gaps do not matter, small scratch (1.3 MB)
        int rc;
        if ((rc = pass1_scratch(ctx, cap, frames_on_device))) return rc;
        // the side view's raw differences of one chunk (one gather instead of two; see k_bb_hist); the results of the whole
        // call stay on the device until the end: chunks run back to back without a host sync
        if ((rc = grow_bufs(ctx, {{L::P1_PRED, (size_t)cap * 256}, {L::P1_HIST, (size_t)cap * 256 * sizeof(uint32_t)},
                                  {L::P1_DIFF, (size_t)cap * p->side_w * p->side_h}, {L::P1_BBX, (size_t)n * sizeof(double)},
                                  {L::P1_LIMS, (size_t)n * 2 * sizeof(int32_t)}, {L::P1_SUMS, (size_t)cap * p->side_w * sizeof(int32_t)}})))
            return rc;
        if ((rc = fold_calib(ctx))) return rc;  // k_prep's vector tier, used by k_bb_hist16
        cudaStream_t st = ctx->stream;
        double *d_bbx = S[L::P1_BBX].as<double>();
        int32_t *d_lims = S[L::P1_LIMS].as<int32_t>();
        for (int64_t s0 = 0; s0 < n; s0 += cap) {
            const int B = (int)std::min<int64_t>(cap, n - s0);
            LmBatch b;
            if ((rc = pass1_chunk(ctx, frames, frames_on_device, s0, B, b))) return rc;
            use_fold(ctx, b);
            if (lm_launch_bbox_tm_de(b, *p, S[L::P1_HIST].as<uint32_t>(), S[L::P1_PRED].p, d_bbx + s0, d_lims + s0 * 2, last_chunk_sums(ctx, s0, cap, n), st,
                                     S[L::P1_DIFF].p) < 0)
                return fail(ctx, LM_ERR_RUNTIME, "bounding-box launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        if (cudaMemcpyAsync(bb_x_raw, d_bbx, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess)
            return fail(ctx, LM_ERR_RUNTIME, "D2H copy failed");
        if (lims && cudaMemcpyAsync(lims, d_lims, (size_t)n * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess)
            return fail(ctx, LM_ERR_RUNTIME, "D2H copy failed");
        if (cudaStreamSynchronize(st) != cudaSuccess)
            return fail(ctx, LM_ERR_RUNTIME, "pass 1 failed on the device: %s", cudaGetErrorString(cudaGetLastError()));
        set_p1(ctx, LM_P1_TM_DE, n, cap, 0, 0, p->side_w, p->side_w);
        return LM_OK;
    });
}

// Pass 1 of the base class, per frame (LocoMouse_class.cpp:579-631, 921-997); see include/locomouse_b200.h.
int lm_bounding_box_base(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, int64_t n, const lm_bb_base_params *p, double *box,
                         int32_t *lims) {
    return entry(ctx, [&]() -> int {
        if (!ctx->configured || !ctx->bkg_set || !ctx->calib_set)
            return fail(ctx, LM_ERR_STATE, "lm_bounding_box_base needs lm_configure, lm_set_background and lm_set_calibration first");
        if (n < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count");
        if (n == 0) return LM_OK;
        if (!frames || !p || !box) return fail(ctx, LM_ERR_INVALID, "null argument");
        const lm_config &k = ctx->cfg;
        auto inside = [&](int x, int y, int w, int h) { return x >= 0 && y >= 0 && w > 0 && h > 0 && x + w <= k.n_cols && y + h <= k.n_rows; };
        if (!inside(p->side_x, p->side_y, p->side_w, p->side_h) || !inside(p->bottom_x, p->bottom_y, p->bottom_w, p->bottom_h))
            return fail(ctx, LM_ERR_INVALID, "view boxes must lie inside the calibrated image");
        if (p->median_filter_size < 1 || !(p->median_filter_size & 1) || p->median_filter_size > 31)
            return fail(ctx, LM_ERR_INVALID, "median_filter_size must be odd and at most 31. Was %d.", p->median_filter_size);
        if (p->min_pixel_visible < 0) return fail(ctx, LM_ERR_INVALID, "min_pixel_visible must be non-negative. Was %d.", p->min_pixel_visible);
        if ((int64_t)p->side_w * p->side_h >= (1 << 21) || (int64_t)p->bottom_w * p->bottom_h >= (1 << 21) || p->side_w > 65535 || p->bottom_w > 65535)
            return fail(ctx, LM_ERR_INVALID, "view too large for the connected-component key packing");
        using L = lm_ctx;
        auto &S = ctx->buf;
        const int cap = 256;  // frames per chunk: two bit images of the whole calibrated image per frame
        const size_t slow = lm_bbox_base_slow_ints(*p), bits = lm_bbox_base_bits_bytes(k.n_rows, k.n_cols, cap);
        int rc;
        if ((rc = pass1_scratch(ctx, cap, frames_on_device))) return rc;
        if ((rc = grow_bufs(ctx, {{L::P1_BITS0, bits}, {L::P1_BITS1, bits}, {L::P1_CC, (size_t)LM_BBOX_SLOW_SLOTS * 3 * slow * sizeof(int32_t)},
                                  {L::P1_VMAP, (size_t)LM_BBOX_SLOW_SLOTS * slow}, {L::P1_VMASK, (size_t)LM_BBOX_SLOW_SLOTS * slow},
                                  {L::P1_SLOW, (size_t)cap * 2 * sizeof(int)}, {L::P1_LIMS, (size_t)n * 8 * sizeof(int32_t)},
                                  {L::P1_SUMS, (size_t)cap * lm_bbox_base_sums(*p) * sizeof(int32_t)}})))
            return rc;
        cudaStream_t st = ctx->stream;
        int32_t *d_lims = S[L::P1_LIMS].as<int32_t>();
        for (int64_t s0 = 0; s0 < n; s0 += cap) {
            const int B = (int)std::min<int64_t>(cap, n - s0);
            LmBatch b;
            if ((rc = pass1_chunk(ctx, frames, frames_on_device, s0, B, b))) return rc;
            if (lm_launch_bbox_base(b, *p, S[L::P1_BITS0].as<uint32_t>(), S[L::P1_BITS1].as<uint32_t>(), S[L::P1_CC].as<int32_t>(), S[L::P1_VMAP].p,
                                    S[L::P1_VMASK].p, S[L::P1_SLOW].as<int>(), d_lims + s0 * 8, last_chunk_sums(ctx, s0, cap, n), st) < 0)
                return fail(ctx, LM_ERR_RUNTIME, "bounding-box launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        std::vector<int32_t> h_lims((size_t)n * 8);
        CK(cudaMemcpyAsync(h_lims.data(), d_lims, h_lims.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        set_p1(ctx, LM_P1_BASE, n, cap, k.n_rows, (k.n_cols + 31) / 32, k.n_cols, lm_bbox_base_sums(*p));
        for (int64_t f = 0; f < n; ++f) {  // computeMouseBox's last lines (class.cpp:981-993) + the caller's offset (628)
            const int32_t *rs = &h_lims[(size_t)f * 8], *rb = rs + 2, *cs = rs + 4, *cb = rs + 6;
            double *o = box + f * 6;
            o[0] = rb[1] > rs[1] ? (double)rb[1] : (double)rs[1];
            o[1] = (double)cb[1] + (double)p->bottom_y;
            o[2] = (double)cs[1];
            const unsigned int wt = (unsigned int)(rs[1] - rs[0]), wb = (unsigned int)(rb[1] - rb[0]);
            o[3] = wt > wb ? (double)wt : (double)wb;
            o[4] = (double)(cb[1] - cb[0]);
            o[5] = (double)(cs[1] - cs[0]);
        }
        if (lims) memcpy(lims, h_lims.data(), h_lims.size() * sizeof(int32_t));
        return LM_OK;
    });
}

// Pass 1 of LocoMouse_TM, per frame (LocoMouse_TM.cpp:115-269); see include/locomouse_b200.h.
int lm_bounding_box_tm(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, int64_t n, const lm_bb_tm_params *p, double *bb_x_raw,
                       int32_t *lims) {
    return entry(ctx, [&]() -> int {
        if (!ctx->configured || !ctx->bkg_set || !ctx->calib_set)
            return fail(ctx, LM_ERR_STATE, "lm_bounding_box_tm needs lm_configure, lm_set_background and lm_set_calibration first");
        if (n < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count");
        if (n == 0) return LM_OK;
        if (!frames || !p || !bb_x_raw || !p->disk) return fail(ctx, LM_ERR_INVALID, "null argument");
        const lm_config &k = ctx->cfg;
        // what the reference's own checks and OpenCV's range assertions would reject (LocoMouse_TM.cpp:20-36, 203-206)
        if (p->side_x != 0 || p->side_w != k.n_cols || p->side_y < 0 || p->side_h <= 0 || p->side_y + p->side_h > k.n_rows)
            return fail(ctx, LM_ERR_INVALID, "the side view must span the image width and lie inside the calibrated image");
        if (p->side_threshold < 0 || p->side_threshold > 255) return fail(ctx, LM_ERR_INVALID, "bw_threshold_side must belong to [0, 255].");
        if (p->min_pixel_count < 1) return fail(ctx, LM_ERR_INVALID, "Min pixel count must be at least 1.");
        if (p->min_pixel_visible < 0) return fail(ctx, LM_ERR_INVALID, "min_pixel_visible must be non-negative. Was %d.", p->min_pixel_visible);
        if (p->zero_col_pre < 0 || p->zero_col_post < 0 || p->zero_row_pre < 0 || p->zero_row_post < 0 || p->zero_col_pre > p->side_w ||
            p->zero_col_post > k.n_cols || p->zero_row_pre > p->side_h || p->zero_row_post > p->side_h)
            return fail(ctx, LM_ERR_INVALID, "zero_*_* parameters range from 0 to the relevant size of the image.");
        if (p->disk_size < 1 || p->disk_size > 63) return fail(ctx, LM_ERR_INVALID, "disk_size must be in [1, 63]. Was %d.", p->disk_size);
        if (p->side_w > 65535 || p->side_h > 65535) return fail(ctx, LM_ERR_INVALID, "side view too large for 16-bit run coordinates");
        {
            // the device keeps the filtered image as bits: its values must be 0 or 1, i.e. no sum of taps may round above 1
            double pos = 0.0;
            for (int i = 0; i < p->disk_size * p->disk_size; ++i) {
                if (!std::isfinite(p->disk[i])) return fail(ctx, LM_ERR_INVALID, "DISK_FILTER has a non-finite entry");
                if (p->disk[i] > 0.f) pos += (double)p->disk[i];
            }
            if (pos >= 1.499) return fail(ctx, LM_ERR_INVALID, "DISK_FILTER must be a normalised smoothing kernel (its positive taps sum to %.4f, limit 1.499)", pos);
        }
        using L = lm_ctx;
        auto &S = ctx->buf;
        const int cap = 256;
        const int cap_tm = (int)std::min<int64_t>(cap, n);   // run-array slots of the global-memory labelling: one per frame of a chunk
        const size_t bits = lm_bbox_tm_bits_bytes(*p, cap), disk = (size_t)p->disk_size * p->disk_size * sizeof(float);
        int rc;
        if ((rc = pass1_scratch(ctx, cap, frames_on_device))) return rc;
        if ((rc = grow_bufs(ctx, {{L::P1_HIST, (size_t)cap * 256 * sizeof(uint32_t)}, {L::P1_PRED, (size_t)cap * 256}, {L::P1_BITS0, bits},
                                  {L::P1_BITS1, bits}, {L::P1_SLOW, (size_t)cap * 2 * sizeof(int)},
                                  {L::P1_RUNS, (size_t)cap_tm * lm_bbox_tm_slow_runs(*p) * 14 + 64}, {L::P1_LMASK, 512 * sizeof(uint32_t)},
                                  {L::P1_DISK, disk}, {L::P1_BBX, (size_t)n * sizeof(double)}, {L::P1_LIMS, (size_t)n * 2 * sizeof(int32_t)},
                                  {L::P1_SUMS, (size_t)cap * p->side_w * sizeof(int32_t)}})))
            return rc;
        cudaStream_t st = ctx->stream;
        double *d_bbx = S[L::P1_BBX].as<double>();
        int32_t *d_lims = S[L::P1_LIMS].as<int32_t>();
        CK(cudaMemcpyAsync(S[L::P1_DISK].p, p->disk, disk, cudaMemcpyHostToDevice, st));
        for (int64_t s0 = 0; s0 < n; s0 += cap) {
            const int B = (int)std::min<int64_t>(cap, n - s0);
            LmBatch b;
            if ((rc = pass1_chunk(ctx, frames, frames_on_device, s0, B, b))) return rc;
            rc = lm_launch_bbox_tm(b, *p, S[L::P1_DISK].as<float>(), S[L::P1_HIST].as<uint32_t>(), S[L::P1_PRED].p, S[L::P1_BITS0].as<uint32_t>(),
                                   S[L::P1_BITS1].as<uint32_t>(), S[L::P1_SLOW].as<int>(), S[L::P1_RUNS].as<unsigned char>(), cap_tm,
                                   S[L::P1_LMASK].as<uint32_t>(), d_bbx + s0, d_lims + s0 * 2, last_chunk_sums(ctx, s0, cap, n), st);
            if (rc == -2) return fail(ctx, LM_ERR_INVALID, "side view of %d x %d pixels does not fit the shared-memory bit image", p->side_w, p->side_h);
            if (rc < 0) return fail(ctx, LM_ERR_RUNTIME, "bounding-box launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        CK(cudaMemcpyAsync(bb_x_raw, d_bbx, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (lims) CK(cudaMemcpyAsync(lims, d_lims, (size_t)n * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        set_p1(ctx, LM_P1_TM, n, cap, p->side_h, (p->side_w + 31) / 32, p->side_w, p->side_w);
        return LM_OK;
    });
}

// computeMouseBoxSize (LocoMouse_class.cpp:1481-1506): per series min(median + 3 std, max).  medianvec sorts the series
// and, for an odd count, returns the element below the middle; stdvec is the sample standard deviation (1515-1556).
int lm_mouse_box_size(double *bb_w, double *bb_hb, double *bb_hs, int64_t n, int32_t size[3]) {
    if (!bb_w || !bb_hb || !bb_hs || !size || n < 1) return LM_ERR_INVALID;
    double *series[3] = {bb_w, bb_hb, bb_hs};
    for (int q = 0; q < 3; ++q) {
        double *v = series[q];
        double med = v[0], sd = 0.0;
        if (n > 1) {
            std::sort(v, v + n);
            const int64_t half = n / 2;
            med = (n % 2 == 0) ? (v[half - 1] + v[half]) / 2 : v[half - 1];
            double sum = 0.0;
            for (int64_t i = 0; i < n; ++i) sum += v[i];
            const double mean = sum / (double)n;
            double sq = 0.0;
            for (int64_t i = 0; i < n; ++i) sq += (v[i] - mean) * (v[i] - mean);
            sd = std::sqrt(sq / (double)(n - 1));
        }
        const uint32_t m3 = (uint32_t)(int64_t)(med + 3 * sd);
        const double last = v[n - 1];
        size[q] = (int32_t)(uint32_t)(int64_t)((double)m3 < last ? (double)m3 : last);
    }
    return LM_OK;
}

// vecmovingaverage (LocoMouse_class.cpp:1559-1608).  (uint32_t)double of a negative value is undefined in C++; like
// the reference built for x86-64 this converts through int64 and keeps the low 32 bits.
int lm_moving_average(const double *v, int64_t n, int32_t window, uint32_t *out) {
    if (!v || !out || n < 0 || window <= 0) return LM_ERR_INVALID;
    auto u32 = [](double x) { return (uint32_t)(int64_t)x; };
    if ((int64_t)window >= n) {
        for (int64_t i = 0; i < n; ++i) out[i] = u32(v[i]);
        return LM_OK;
    }
    const int half = window / 2;
    double cur = 0;
    for (int i = 0; i < half; ++i) out[i] = u32(v[i]);
    for (int i = 0; i < window; ++i) cur += v[i];
    out[half] = u32(std::floor(cur / window));
    for (int64_t i = 0; i < n - window; ++i) {
        cur = cur - v[i] + v[i + window];
        out[half + 1 + i] = u32(std::floor(cur / window));
    }
    for (int64_t i = n - half - 1; i < n; ++i) out[i] = u32(v[i]);
    return LM_OK;
}

// ---- cost builders of the host tracker (SURVEY 8f-2): candidates up, cost matrices down -------------------------------
int lm_unary_costs(lm_ctx *ctx, const lm_results *res, int64_t n, int32_t feat, int32_t bb_w, int32_t bb_h, const lm_location_prior *priors,
                   int32_t n_priors, double *out) {
    return entry(ctx, [&]() -> int {
        if (!res || !priors || !out || n < 0 || n > res->n_frames || feat < 0 || feat > 1 || bb_w < 1 || bb_h < 1 || n_priors < 1 || res->cand_cap < 1)
            return fail(ctx, LM_ERR_INVALID, "lm_unary_costs: bad argument");
        if (n == 0) return LM_OK;
        using L = lm_ctx;
        auto &D = ctx->buf;
        const size_t cap = (size_t)res->cand_cap;
        const size_t cand = (size_t)n * 2 * cap * sizeof(lm_cand), ncand = (size_t)n * 2 * 4, pri = (size_t)n_priors * sizeof(lm_location_prior),
                     nout = (size_t)n * n_priors * cap * 8;
        cudaStream_t st = ctx->stream;
        if (int rc = grow_bufs(ctx, {{L::COST_CAND, cand}, {L::COST_NCAND, ncand}, {L::COST_PRIOR, pri}, {L::COST_OUT, nout}})) return rc;
        CK(cudaMemcpyAsync(D[L::COST_CAND].p, res->bottom, cand, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(D[L::COST_NCAND].p, res->n_bottom, ncand, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(D[L::COST_PRIOR].p, priors, pri, cudaMemcpyHostToDevice, st));
        if (lm_launch_unary(D[L::COST_CAND].as<lm_cand>(), D[L::COST_NCAND].as<int32_t>(), n, (int)cap, feat, bb_w, bb_h, D[L::COST_PRIOR].as<lm_location_prior>(),
                            n_priors, D[L::COST_OUT].as<double>(), st) < 0)
            return fail(ctx, LM_ERR_RUNTIME, "unary cost launch failed");
        CK(cudaMemcpyAsync(out, D[L::COST_OUT].p, nout, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return LM_OK;
    });
}

int lm_pairwise_costs(lm_ctx *ctx, const lm_results *res, int64_t n, int32_t feat, const lm_pairwise_params *p, int64_t *offs, int32_t *jc,
                      int32_t *ir, double *pr, int64_t cap, int64_t *total) {
    return entry(ctx, [&]() -> int {
        if (!res || !p || !offs || !jc || !total || n < 0 || n > res->n_frames || feat < 0 || feat > 1 || cap < 0 || (cap > 0 && (!ir || !pr)) ||
            p->ong_w < 1 || p->ong_h < 1 || (int64_t)p->ong_w * p->ong_h > (1 << 20) || res->cand_cap < 1)
            return fail(ctx, LM_ERR_INVALID, "lm_pairwise_costs: bad argument");
        *total = 0;
        offs[0] = 0;
        if (n == 0) return LM_OK;
        using L = lm_ctx;
        auto &D = ctx->buf;
        const size_t ccap = (size_t)res->cand_cap;
        const size_t jc_stride = ccap + (size_t)p->ong_w * p->ong_h + 1;
        const size_t cand = (size_t)n * 2 * ccap * sizeof(lm_cand), ncand = (size_t)n * 2 * 4;
        cudaStream_t st = ctx->stream;
        int rc;
        if ((rc = grow_bufs(ctx, {{L::COST_CAND, cand}, {L::COST_NCAND, ncand}, {L::COST_JC, (size_t)n * jc_stride * 4}, {L::COST_NNZ, (size_t)n * 8},
                                  {L::COST_OFFS, (size_t)(n + 1) * 8}})))
            return rc;
        lm_cand *d_cand = D[L::COST_CAND].as<lm_cand>();
        int32_t *d_ncand = D[L::COST_NCAND].as<int32_t>(), *d_jc = D[L::COST_JC].as<int32_t>();
        int64_t *d_nnz = D[L::COST_NNZ].as<int64_t>(), *d_offs = D[L::COST_OFFS].as<int64_t>();
        CK(cudaMemcpyAsync(d_cand, res->bottom, cand, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_ncand, res->n_bottom, ncand, cudaMemcpyHostToDevice, st));
        if (lm_launch_pairwise(d_cand, d_ncand, n, (int)ccap, feat, *p, d_jc, d_nnz, d_offs, nullptr, nullptr, 0, 0, st) < 0)
            return fail(ctx, LM_ERR_RUNTIME, "pairwise cost launch failed");
        CK(cudaMemcpyAsync(offs, d_offs, (size_t)(n + 1) * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(jc, d_jc, (size_t)n * jc_stride * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        *total = offs[n];
        if (*total > cap) return fail(ctx, LM_ERR_OVERFLOW, "lm_pairwise_costs: %lld stored entries, capacity %lld", (long long)*total, (long long)cap);
        if (*total == 0) return LM_OK;
        if ((rc = grow_bufs(ctx, {{L::COST_IR, (size_t)*total * 4}, {L::COST_PR, (size_t)*total * 8}}))) return rc;
        if (lm_launch_pairwise(d_cand, d_ncand, n, (int)ccap, feat, *p, d_jc, d_nnz, d_offs, D[L::COST_IR].as<int32_t>(), D[L::COST_PR].as<double>(),
                               *total, 1, st) < 0)
            return fail(ctx, LM_ERR_RUNTIME, "pairwise cost launch failed");
        CK(cudaMemcpyAsync(ir, D[L::COST_IR].p, (size_t)*total * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(pr, D[L::COST_PR].p, (size_t)*total * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return LM_OK;
    });
}

int lm_debug_nms(lm_ctx *ctx, int view, int feat, const float *scores, lm_cand *out) {
    if (!ctx) return LM_ERR_INVALID;
    if (!ctx->configured || !ctx->model_set) return fail(ctx, LM_ERR_STATE, "lm_debug_nms needs lm_configure and lm_set_model first");
    if (view < 0 || view > 1 || feat < 0 || feat > 1 || !scores || !out) return fail(ctx, LM_ERR_INVALID, "lm_debug_nms: bad argument");
    DeviceGuard guard(ctx->device);
    int rc = prepare(ctx, 64, 2);   // one frame's lists: the smallest scratch set will do (grows later if a detection call needs more)
    if (rc) {
        release_scratch(ctx);
        trim_scratch(ctx);
        return rc;
    }
    LmBatch b = ctx->bt;
    b.B = 1;
    const lm_config &k = ctx->cfg;
    const int bw = k.bb_w, bh = b.bb_h[view];
    std::vector<LmDet> det;
    for (int y = 0; y < bh; ++y)
        for (int x = 0; x < bw; ++x) {
            const float v = scores[(size_t)y * bw + x];
            if (v > 0.f) det.push_back(LmDet{(uint32_t)(y * bw + x), v});
        }
    if ((int)det.size() > k.det_cap) return fail(ctx, LM_ERR_OVERFLOW, "lm_debug_nms: %zu positives exceed det_cap", det.size());
    cudaStream_t st = ctx->stream;
    CK(cudaStreamSynchronize(st));
    const int list = (0 * 2 + feat) * 2 + view;
    int32_t counts[4] = {0, 0, 0, 0};
    counts[list] = (int32_t)det.size();
    if (view == LM_SIDE) {
        // peakClustering only runs for a feature whose bottom list is non-empty (class.cpp:820, 828): give it one detection
        const int blist = (0 * 2 + feat) * 2 + LM_BOTTOM;
        const LmDet one{0u, 1.0f};
        counts[blist] = 1;
        CK(cudaMemcpyAsync(b.det + (size_t)blist * k.det_cap, &one, sizeof one, cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemcpyAsync(b.det_count, counts, sizeof counts, cudaMemcpyHostToDevice, st));
    if (!det.empty())
        CK(cudaMemcpyAsync(b.det + (size_t)list * k.det_cap, det.data(), det.size() * sizeof(LmDet), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(b.tailmask, 0, (size_t)b.bb_h[LM_BOTTOM] * b.tail_pitch, st));
    CK(cudaMemsetAsync(b.flags, 0, 4, st));
    if (lm_launch_nms(b, st) < 0) return fail(ctx, LM_ERR_RUNTIME, "nms launch failed");
    int32_t n = 0;
    uint32_t flags = 0;
    const lm_cand *src = (view == LM_BOTTOM ? b.bottom : b.side) + (size_t)feat * k.cand_cap;
    CK(cudaMemcpyAsync(&n, (view == LM_BOTTOM ? b.n_bottom : b.n_side) + feat, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&flags, b.flags, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out, src, (size_t)k.cand_cap * sizeof(lm_cand), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (flags) return fail(ctx, LM_ERR_OVERFLOW, "lm_debug_nms: list overflow (flags %u)", flags);
    return n;
}

int lm_host_alloc(void **ptr, size_t bytes) {
    if (!ptr) return LM_ERR_INVALID;
    *ptr = nullptr;
    return cudaHostAlloc(ptr, std::max<size_t>(bytes, 1), cudaHostAllocPortable) == cudaSuccess ? LM_OK : LM_ERR_RUNTIME;
}

int lm_host_free(void *ptr) {
    if (!ptr) return LM_OK;
    return cudaFreeHost(ptr) == cudaSuccess ? LM_OK : LM_ERR_RUNTIME;
}

int lm_device_alloc(lm_ctx *ctx, void **ptr, size_t bytes) {
    if (!ctx || !ptr) return LM_ERR_INVALID;
    *ptr = nullptr;
    DeviceGuard guard(ctx->device);
    const cudaError_t e = cudaMalloc(ptr, std::max<size_t>(bytes, 1));
    if (e != cudaSuccess) {
        cudaGetLastError();
        *ptr = nullptr;
        return fail(ctx, LM_ERR_RUNTIME, "cannot allocate %zu bytes of device memory: %s", bytes, cudaGetErrorString(e));
    }
    ++ctx->device_allocs;
    return LM_OK;
}

int lm_device_free(lm_ctx *ctx, void *ptr) {
    if (!ctx) return LM_ERR_INVALID;
    if (!ptr) return LM_OK;
    DeviceGuard guard(ctx->device);
    return cudaFree(ptr) == cudaSuccess ? LM_OK : fail(ctx, LM_ERR_RUNTIME, "cudaFree failed");
}

int lm_device_copy(lm_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (!ctx || (bytes && (!dst || !src))) return LM_ERR_INVALID;
    if (!bytes) return LM_OK;
    DeviceGuard guard(ctx->device);
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    return e == cudaSuccess ? LM_OK : fail(ctx, LM_ERR_RUNTIME, "device copy of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
}

// ---- lm_decode_png -----------------------------------------------------------------------------------------------------
namespace {
// Signature and IHDR of one frame (the first LM_PNG_HDR_BYTES bytes, len = the frame's size); bytes per pixel or 0 with `why`.
int png_check_header(const uint8_t *h, int64_t len, int rows, int cols, char *why, size_t why_cap) {
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    auto be32 = [](const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3]; };
    if (len < 45 || memcmp(h, sig, 8)) return snprintf(why, why_cap, "not a PNG file (%lld bytes)", (long long)len), 0;
    if (be32(h + 8) != 13 || memcmp(h + 12, "IHDR", 4)) return snprintf(why, why_cap, "the first chunk is not IHDR"), 0;
    const uint32_t w = be32(h + 16), ht = be32(h + 20);
    if (w != (uint32_t)cols || ht != (uint32_t)rows)
        return snprintf(why, why_cap, "%u x %u pixels, the configured video is %d x %d", w, ht, cols, rows), 0;
    const int depth = h[24], ct = h[25];
    if (depth != 8 || (ct != 0 && ct != 2 && ct != 6))
        return snprintf(why, why_cap, "bit depth %d, colour type %d: only 8-bit grey (0), RGB (2) and RGBA (6) are decoded", depth, ct), 0;
    if (h[26] || h[27]) return snprintf(why, why_cap, "unknown compression or filter method"), 0;
    if (h[28]) return snprintf(why, why_cap, "interlaced frames are not decoded"), 0;
    return ct == 0 ? 1 : ct == 2 ? 3 : 4;
}

int decode_png_impl(lm_ctx *ctx, const uint8_t *payload, int on_dev, const int64_t *offsets, int64_t n, uint8_t *frames) {
    if (!ctx->configured) return fail(ctx, LM_ERR_STATE, "lm_decode_png needs lm_configure first");
    if (n < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count");
    ctx->ms_decode = 0.f;
    if (n == 0) return LM_OK;
    if (!payload || !offsets || !frames) return fail(ctx, LM_ERR_INVALID, "null argument");
    const int rows = ctx->cfg.vid_rows, cols = ctx->cfg.vid_cols;
    for (int64_t i = 0; i < n; ++i)
        if (offsets[i] < 0 || offsets[i + 1] < offsets[i]) return fail(ctx, LM_ERR_INVALID, "frame %lld: offsets must not decrease", (long long)i);
    if ((int64_t)rows * (1 + (int64_t)cols * 4) >= INT32_MAX) return fail(ctx, LM_ERR_INVALID, "frame too large for the PNG decoder");
    cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
    auto &B = ctx->buf;
    if (int rc = grow(ctx, B[lm_ctx::PNG_OFFS], (size_t)(n + 1) * sizeof(int64_t))) return rc;
    if (int rc = grow(ctx, B[lm_ctx::PNG_STATUS], (size_t)n * sizeof(int32_t))) return rc;
    int64_t *d_offs = reinterpret_cast<int64_t *>(B[lm_ctx::PNG_OFFS].p);
    int32_t *d_status = reinterpret_cast<int32_t *>(B[lm_ctx::PNG_STATUS].p);
    CK(cudaMemcpyAsync(d_offs, offsets, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(d_status, 0xff, (size_t)n * sizeof(int32_t), st));  // -1: not decoded

    // every frame's signature and IHDR, checked before anything is decoded
    std::vector<uint8_t> hdr_dev;
    if (on_dev) {
        if (int rc = grow(ctx, B[lm_ctx::PNG_HDR], (size_t)n * LM_PNG_HDR_BYTES)) return rc;
        if (lm_launch_png_headers(payload, d_offs, 0, n, B[lm_ctx::PNG_HDR].p, st) < 0) return fail(ctx, LM_ERR_RUNTIME, "PNG header launch failed");
        hdr_dev.resize((size_t)n * LM_PNG_HDR_BYTES);
        CK(cudaMemcpyAsync(hdr_dev.data(), B[lm_ctx::PNG_HDR].p, hdr_dev.size(), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    std::vector<uint8_t> bpp((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        char why[160];
        const uint8_t *h = on_dev ? hdr_dev.data() + (size_t)i * LM_PNG_HDR_BYTES : payload + offsets[i];
        if (!(bpp[i] = (uint8_t)png_check_header(h, offsets[i + 1] - offsets[i], rows, cols, why, sizeof why)))
            return fail(ctx, LM_ERR_INVALID, "frame %lld: %s", (long long)i, why);
    }

    // Pieces of consecutive frames share one scratch allocation (one filtered stream per frame) and, from the host, one of
    // two compressed staging buffers: the copy of piece k + 1 (copy stream) overlaps the decode of piece k.
    const int64_t max_piece = on_dev ? 8192 : std::max<int64_t>(1024, (n + 3) / 4);
    const size_t scratch_budget = (size_t)4 << 30, stage_budget = (size_t)2 << 30;
    struct Piece {
        int64_t s, e;
        int64_t slot;
    };
    std::vector<Piece> pieces;
    size_t scratch_need = 0, stage_need = 0;
    for (int64_t s = 0; s < n;) {
        int64_t e = s, slot = 0;
        while (e < n && e - s < max_piece) {
            const int64_t sl = std::max<int64_t>(slot, (int64_t)rows * (1 + (int64_t)cols * bpp[e]));
            const size_t comp = (size_t)(offsets[e + 1] - offsets[s]);
            if (e > s && ((size_t)sl * (e + 1 - s) > scratch_budget || (!on_dev && comp > stage_budget))) break;
            slot = sl;
            ++e;
        }
        pieces.push_back({s, e, slot});
        scratch_need = std::max(scratch_need, (size_t)slot * (e - s));
        stage_need = std::max(stage_need, (size_t)(offsets[e] - offsets[s]));
        s = e;
    }
    if (int rc = grow(ctx, B[lm_ctx::PNG_SCRATCH], scratch_need)) return rc;
    if (!on_dev) {
        for (int k = 0; k < 2 && k < (int)pieces.size(); ++k)
            if (int rc = grow(ctx, B[lm_ctx::PNG_STAGE0 + k], stage_need)) return rc;
        for (int k = 0; k < 2; ++k) {
            if (!ctx->ev_png_copy[k]) CK(cudaEventCreateWithFlags(&ctx->ev_png_copy[k], cudaEventDisableTiming));
            if (!ctx->ev_png_done[k]) CK(cudaEventCreateWithFlags(&ctx->ev_png_done[k], cudaEventDisableTiming));
        }
    }
    struct Events {  // start / end of each decode launch, for ms_decode
        std::vector<cudaEvent_t> ev;
        ~Events() {
            for (cudaEvent_t e : ev) cudaEventDestroy(e);
        }
    } T;
    T.ev.resize(2 * pieces.size());
    for (auto &e : T.ev) CK(cudaEventCreate(&e));
    for (size_t k = 0; k < pieces.size(); ++k) {
        const Piece &P = pieces[k];
        const uint8_t *src = payload;
        int64_t base = 0;
        if (!on_dev) {
            uint8_t *stg = B[lm_ctx::PNG_STAGE0 + (k & 1)].p;
            if (k >= 2) CK(cudaStreamWaitEvent(cp, ctx->ev_png_done[k & 1], 0));  // piece k - 2 no longer reads this buffer
            CK(cudaMemcpyAsync(stg, payload + offsets[P.s], (size_t)(offsets[P.e] - offsets[P.s]), cudaMemcpyHostToDevice, cp));
            CK(cudaEventRecord(ctx->ev_png_copy[k & 1], cp));
            CK(cudaStreamWaitEvent(st, ctx->ev_png_copy[k & 1], 0));
            src = stg;
            base = offsets[P.s];
        }
        CK(cudaEventRecord(T.ev[2 * k], st));
        if (lm_launch_png_decode(src, d_offs + P.s, base, (int)(P.e - P.s), rows, cols, B[lm_ctx::PNG_SCRATCH].p, P.slot,
                                 frames + P.s * (int64_t)rows * cols, d_status + P.s, st) < 0)
            return fail(ctx, LM_ERR_RUNTIME, "PNG decode launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        CK(cudaEventRecord(T.ev[2 * k + 1], st));
        if (!on_dev) CK(cudaEventRecord(ctx->ev_png_done[k & 1], st));
    }
    std::vector<int32_t> status((size_t)n);
    CK(cudaMemcpyAsync(status.data(), d_status, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (size_t k = 0; k < pieces.size(); ++k) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, T.ev[2 * k], T.ev[2 * k + 1]) == cudaSuccess) ctx->ms_decode += t;
    }
    for (int64_t i = 0; i < n; ++i)
        if (status[i] != LM_PNG_OK) return fail(ctx, LM_ERR_INVALID, "frame %lld: %s", (long long)i, lm_png_status_text(status[i]));
    return LM_OK;
}
}  // namespace

// ---- lm_decode_ffv1 ----------------------------------------------------------------------------------------------------
namespace {
int decode_ffv1_impl(lm_ctx *ctx, const uint8_t *extradata, int64_t extradata_len, const uint8_t *payload, int on_dev, const int64_t *offsets,
                     int64_t n, uint8_t *frames) {
    if (!ctx->configured) return fail(ctx, LM_ERR_STATE, "lm_decode_ffv1 needs lm_configure first");
    if (n < 0 || extradata_len < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count or record length");
    ctx->ms_decode = 0.f;
    if (n == 0) return LM_OK;
    if (!payload || !offsets || !frames || (extradata_len && !extradata)) return fail(ctx, LM_ERR_INVALID, "null argument");
    const int rows = ctx->cfg.vid_rows, cols = ctx->cfg.vid_cols;
    for (int64_t i = 0; i < n; ++i)
        if (offsets[i] < 0 || offsets[i + 1] < offsets[i]) return fail(ctx, LM_ERR_INVALID, "frame %lld: offsets must not decrease", (long long)i);
    std::unique_ptr<ffv1::Record> rec(new ffv1::Record);
    char why[200];
    int64_t init_bytes = 0;
    if (ffv1::parse_record(extradata, extradata_len, rows, cols, *rec, nullptr, &init_bytes, why, sizeof why))
        return fail(ctx, LM_ERR_INVALID, "FFV1 configuration record: %s", why);
    std::vector<uint8_t> initial((size_t)std::max<int64_t>(init_bytes, 1));
    ffv1::parse_record(extradata, extradata_len, rows, cols, *rec, initial.data(), &init_bytes, why, sizeof why);
    const int S = rec->slices();
    cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
    auto &B = ctx->buf;
    using L = lm_ctx;
    if (int rc = grow(ctx, B[L::PNG_OFFS], (size_t)(n + 1) * sizeof(int64_t))) return rc;
    int64_t *d_offs = reinterpret_cast<int64_t *>(B[L::PNG_OFFS].p);
    CK(cudaMemcpyAsync(d_offs, offsets, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));

    // keyframe flags (each frame's first decision): they cut the video into GOPs, and every (GOP, slice) is a chain
    std::vector<uint8_t> hdr_dev;
    if (on_dev) {
        if (int rc = grow(ctx, B[L::PNG_HDR], (size_t)n * LM_PNG_HDR_BYTES)) return rc;
        if (lm_launch_png_headers(payload, d_offs, 0, n, B[L::PNG_HDR].p, st) < 0) return fail(ctx, LM_ERR_RUNTIME, "FFV1 header launch failed");
        hdr_dev.resize((size_t)n * LM_PNG_HDR_BYTES);
        CK(cudaMemcpyAsync(hdr_dev.data(), B[L::PNG_HDR].p, hdr_dev.size(), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    std::vector<int64_t> gop;  // first frame of every GOP, then n
    for (int64_t i = 0; i < n; ++i) {
        const int64_t len = offsets[i + 1] - offsets[i];
        const bool key = on_dev ? ffv1::keyframe_bit(hdr_dev.data() + (size_t)i * LM_PNG_HDR_BYTES, std::min<int64_t>(len, LM_PNG_HDR_BYTES))
                                : ffv1::keyframe_bit(payload + offsets[i], len);
        if (i == 0 && !key) return fail(ctx, LM_ERR_INVALID, "frame 0: the first FFV1 frame is not a keyframe");
        if (key) gop.push_back(i);
    }
    gop.push_back(n);
    const int64_t ngop = (int64_t)gop.size() - 1;
    std::vector<LmFfv1Chain> chains((size_t)(ngop * S));
    for (int64_t g = 0; g < ngop; ++g)
        for (int s = 0; s < S; ++s) chains[(size_t)(g * S + s)] = LmFfv1Chain{gop[g], (int32_t)(gop[g + 1] - gop[g]), s};

    const int64_t ns = n * S;
    if (int rc = grow(ctx, B[L::PNG_STATUS], (size_t)ns * sizeof(int32_t))) return rc;
    if (int rc = grow(ctx, B[L::FFV1_SOFF], (size_t)ns * sizeof(int64_t))) return rc;
    if (int rc = grow(ctx, B[L::FFV1_SLEN], (size_t)ns * sizeof(int32_t))) return rc;
    if (int rc = grow(ctx, B[L::FFV1_CHAINS], chains.size() * sizeof(LmFfv1Chain))) return rc;
    if (int rc = grow(ctx, B[L::FFV1_REC], sizeof(ffv1::Record))) return rc;
    if (int rc = grow(ctx, B[L::FFV1_INIT], initial.size())) return rc;
    int32_t *d_status = reinterpret_cast<int32_t *>(B[L::PNG_STATUS].p);
    int64_t *d_soff = reinterpret_cast<int64_t *>(B[L::FFV1_SOFF].p);
    int32_t *d_slen = reinterpret_cast<int32_t *>(B[L::FFV1_SLEN].p);
    LmFfv1Chain *d_chains = reinterpret_cast<LmFfv1Chain *>(B[L::FFV1_CHAINS].p);
    const ffv1::Record *d_rec = reinterpret_cast<const ffv1::Record *>(B[L::FFV1_REC].p);
    CK(cudaMemsetAsync(d_status, 0xff, (size_t)ns * sizeof(int32_t), st));  // -1: not decoded
    CK(cudaMemcpyAsync(B[L::FFV1_CHAINS].p, chains.data(), chains.size() * sizeof(LmFfv1Chain), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B[L::FFV1_REC].p, rec.get(), sizeof(ffv1::Record), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B[L::FFV1_INIT].p, initial.data(), initial.size(), cudaMemcpyHostToDevice, st));

    // A host payload goes up in (at most) two pieces of whole GOPs, one per staging buffer: piece 0 is decoded on the
    // library stream while piece 1 is copied, and piece 1 is decoded on the copy stream after its copy, concurrently.
    struct Piece {
        int64_t g0, g1;  // GOPs [g0, g1)
    };
    std::vector<Piece> pieces;
    if (!on_dev && ngop >= 2) {
        int64_t g = 1;
        while (g + 1 < ngop && gop[g] < n / 2) ++g;
        pieces.push_back({0, g});
        pieces.push_back({g, ngop});
    } else {
        pieces.push_back({0, ngop});
    }
    // Chain work memory: in shared memory when the launch still fits in one wave that way, else in global slots
    // (at most 2 GB per piece; more chains run as consecutive launches over the same slots).
    const int64_t wb = (ffv1::work_bytes(*rec, cols) + 15) & ~(int64_t)15;
    int dev_smem = 0, sm_smem = 0, n_sm = 0;
    CK(cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    CK(cudaDeviceGetAttribute(&sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, ctx->device));
    CK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, ctx->device));
    const int64_t smem_cta = (int64_t)lm_ffv1_smem_tables() + LM_FFV1_CHAINS_PER_CTA * wb;
    const int64_t smem_wave = smem_cta <= dev_smem ? (int64_t)(sm_smem / (smem_cta + 1024)) * n_sm * LM_FFV1_CHAINS_PER_CTA : 0;
    const int64_t slot_budget = (int64_t)2 << 30;
    const int64_t batch = std::max<int64_t>(LM_FFV1_CHAINS_PER_CTA, slot_budget / wb / LM_FFV1_CHAINS_PER_CTA * LM_FFV1_CHAINS_PER_CTA);
    if (!on_dev) {
        for (size_t k = 0; k < pieces.size(); ++k) {
            const size_t bytes = (size_t)(offsets[gop[pieces[k].g1]] - offsets[gop[pieces[k].g0]]);
            if (int rc = grow(ctx, B[L::PNG_STAGE0 + k], bytes)) return rc;
        }
        for (int k = 0; k < 2; ++k)
            if (!ctx->ev_png_copy[k]) CK(cudaEventCreateWithFlags(&ctx->ev_png_copy[k], cudaEventDisableTiming));
    }
    std::vector<int> in_smem(pieces.size());
    for (size_t k = 0; k < pieces.size(); ++k) {
        const int64_t nch = (pieces[k].g1 - pieces[k].g0) * S;
        in_smem[k] = nch <= smem_wave;
        if (!in_smem[k])
            if (int rc = grow(ctx, B[L::FFV1_WORK0 + k], (size_t)(std::min(nch, batch) * wb))) return rc;
    }
    struct Events {  // uploads done, decode start, decode end
        cudaEvent_t e[3] = {};
        ~Events() {
            for (cudaEvent_t x : e)
                if (x) cudaEventDestroy(x);
        }
    } T;
    for (auto &e : T.e) CK(cudaEventCreate(&e));
    CK(cudaEventRecord(T.e[0], st));
    for (size_t k = 0; k < pieces.size(); ++k) {
        const Piece &P = pieces[k];
        const int64_t f0 = gop[P.g0], f1 = gop[P.g1];
        cudaStream_t ks = k ? cp : st;
        const uint8_t *src = payload;
        int64_t base = 0;
        if (!on_dev) {
            src = B[L::PNG_STAGE0 + k].p;
            base = offsets[f0];
            CK(cudaMemcpyAsync(B[L::PNG_STAGE0 + k].p, payload + base, (size_t)(offsets[f1] - base), cudaMemcpyHostToDevice, cp));
            if (k == 0) {
                CK(cudaEventRecord(ctx->ev_png_copy[0], cp));
                CK(cudaStreamWaitEvent(st, ctx->ev_png_copy[0], 0));
            } else {
                CK(cudaStreamWaitEvent(cp, T.e[0], 0));  // the offsets, record and chain list are on the device
            }
        }
        if (k == 0) CK(cudaEventRecord(T.e[1], st));
        if (lm_launch_ffv1_locate(src, d_offs + f0, base, f1 - f0, S, rec->ec, d_soff + f0 * S, d_slen + f0 * S, d_status + f0 * S, ks) < 0 ||
            (rec->ec && lm_launch_ffv1_crc(src, d_soff + f0 * S, d_slen + f0 * S, (f1 - f0) * S, d_status + f0 * S, ks) < 0))
            return fail(ctx, LM_ERR_RUNTIME, "FFV1 slice launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        for (int64_t c0 = P.g0 * S; c0 < P.g1 * S; c0 += batch) {  // (slice offsets are relative to src: frames keep their numbers)
            const int nch = (int)std::min<int64_t>(batch, P.g1 * S - c0);
            if (lm_launch_ffv1_decode(d_rec, rec->ac, B[L::FFV1_INIT].p, src, d_soff, d_slen, d_status, frames, rows, cols, d_chains + c0, nch,
                                      B[L::FFV1_WORK0 + k].p, wb, in_smem[k], ks) < 0)
                return fail(ctx, LM_ERR_RUNTIME, "FFV1 decode launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
    }
    if (pieces.size() > 1) {
        CK(cudaEventRecord(ctx->ev_png_copy[1], cp));
        CK(cudaStreamWaitEvent(st, ctx->ev_png_copy[1], 0));
    }
    CK(cudaEventRecord(T.e[2], st));
    std::vector<int32_t> status((size_t)ns);
    CK(cudaMemcpyAsync(status.data(), d_status, (size_t)ns * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float t = 0.f;
    if (cudaEventElapsedTime(&t, T.e[1], T.e[2]) == cudaSuccess) ctx->ms_decode = t;
    for (int64_t i = 0; i < ns; ++i)
        if (status[i] != ffv1::LM_FFV1_OK)
            return fail(ctx, LM_ERR_INVALID, "frame %lld, slice %d: %s", (long long)(i / S), (int)(i % S), ffv1::status_text(status[i]));
    return LM_OK;
}
}  // namespace

// ---- lm_decode_mjpeg ---------------------------------------------------------------------------------------------------
namespace {
int decode_mjpeg_impl(lm_ctx *ctx, const uint8_t *payload, int on_dev, const int64_t *offsets, int64_t n, uint8_t *frames) {
    if (!ctx->configured) return fail(ctx, LM_ERR_STATE, "lm_decode_mjpeg needs lm_configure first");
    if (n < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count");
    ctx->ms_decode = 0.f;
    if (n == 0) return LM_OK;
    if (!payload || !offsets || !frames) return fail(ctx, LM_ERR_INVALID, "null argument");
    const int rows = ctx->cfg.vid_rows, cols = ctx->cfg.vid_cols;
    for (int64_t i = 0; i < n; ++i)
        if (offsets[i] < 0 || offsets[i + 1] < offsets[i]) return fail(ctx, LM_ERR_INVALID, "frame %lld: offsets must not decrease", (long long)i);
    if (rows > 65535 || cols > 65535) return fail(ctx, LM_ERR_INVALID, "a JPEG frame is at most 65535 x 65535 pixels");
    cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
    auto &B = ctx->buf;
    using L = lm_ctx;
    if (int rc = grow(ctx, B[L::PNG_OFFS], (size_t)(n + 1) * sizeof(int64_t))) return rc;
    if (int rc = grow(ctx, B[L::PNG_STATUS], (size_t)(n + 1) * sizeof(int32_t))) return rc;  // + frame 0's DHT tables
    int64_t *d_offs = reinterpret_cast<int64_t *>(B[L::PNG_OFFS].p);
    int32_t *d_status = reinterpret_cast<int32_t *>(B[L::PNG_STATUS].p);
    CK(cudaMemcpyAsync(d_offs, offsets, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(d_status, 0xff, (size_t)n * sizeof(int32_t), st));  // -1: not decoded

    // Pieces of consecutive frames share the coefficient scratch (the widest layout's blocks per frame) and, from the host,
    // one of two staging buffers: the copy of piece k + 1 (copy stream) overlaps the decode of piece k.
    const size_t slot = (size_t)mjpeg::max_blocks(rows, cols) * 64 * sizeof(int16_t);
    const size_t scratch_budget = (size_t)4 << 30, stage_budget = (size_t)2 << 30;
    const int64_t max_piece = std::max<int64_t>(1, std::min<int64_t>(on_dev ? 8192 : std::max<int64_t>(1024, (n + 3) / 4), scratch_budget / slot));
    struct Piece {
        int64_t s, e;
    };
    std::vector<Piece> pieces;
    size_t stage_need = 0;
    int64_t piece_max = 0;
    for (int64_t s = 0; s < n;) {
        int64_t e = s + 1;
        while (e < n && e - s < max_piece && (on_dev || (size_t)(offsets[e + 1] - offsets[s]) <= stage_budget)) ++e;
        pieces.push_back({s, e});
        stage_need = std::max(stage_need, (size_t)(offsets[e] - offsets[s]));
        piece_max = std::max(piece_max, e - s);
        s = e;
    }
    if (int rc = grow(ctx, B[L::PNG_SCRATCH], slot * (size_t)piece_max)) return rc;
    if (int rc = grow(ctx, B[L::MJPEG_HDR], lm_mjpeg_header_bytes() * (size_t)piece_max)) return rc;
    if (!on_dev) {
        for (int k = 0; k < 2 && k < (int)pieces.size(); ++k)
            if (int rc = grow(ctx, B[L::PNG_STAGE0 + k], std::max<size_t>(stage_need, 1))) return rc;
        for (int k = 0; k < 2; ++k) {
            if (!ctx->ev_png_copy[k]) CK(cudaEventCreateWithFlags(&ctx->ev_png_copy[k], cudaEventDisableTiming));
            if (!ctx->ev_png_done[k]) CK(cudaEventCreateWithFlags(&ctx->ev_png_done[k], cudaEventDisableTiming));
        }
    }
    struct Events {  // start / end of each piece's decode launches, for ms_decode
        std::vector<cudaEvent_t> ev;
        ~Events() {
            for (cudaEvent_t e : ev) cudaEventDestroy(e);
        }
    } T;
    T.ev.resize(2 * pieces.size());
    for (auto &e : T.ev) CK(cudaEventCreate(&e));
    for (size_t k = 0; k < pieces.size(); ++k) {
        const Piece &P = pieces[k];
        const uint8_t *src = payload;
        int64_t base = 0;
        if (!on_dev) {
            uint8_t *stg = B[L::PNG_STAGE0 + (k & 1)].p;
            if (k >= 2) CK(cudaStreamWaitEvent(cp, ctx->ev_png_done[k & 1], 0));  // piece k - 2 no longer reads this buffer
            CK(cudaMemcpyAsync(stg, payload + offsets[P.s], (size_t)(offsets[P.e] - offsets[P.s]), cudaMemcpyHostToDevice, cp));
            CK(cudaEventRecord(ctx->ev_png_copy[k & 1], cp));
            CK(cudaStreamWaitEvent(st, ctx->ev_png_copy[k & 1], 0));
            src = stg;
            base = offsets[P.s];
        }
        CK(cudaEventRecord(T.ev[2 * k], st));
        if (lm_launch_mjpeg_decode(src, d_offs + P.s, base, (int)(P.e - P.s), rows, cols, B[L::MJPEG_HDR].p, B[L::PNG_SCRATCH].as<int16_t>(),
                                   d_status + P.s, d_status + n, k == 0, frames + P.s * (int64_t)rows * cols, st) < 0)
            return fail(ctx, LM_ERR_RUNTIME, "Motion-JPEG decode launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        CK(cudaEventRecord(T.ev[2 * k + 1], st));
        if (!on_dev) CK(cudaEventRecord(ctx->ev_png_done[k & 1], st));
    }
    std::vector<int32_t> status((size_t)n);
    CK(cudaMemcpyAsync(status.data(), d_status, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (size_t k = 0; k < pieces.size(); ++k) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, T.ev[2 * k], T.ev[2 * k + 1]) == cudaSuccess) ctx->ms_decode += t;
    }
    for (int64_t i = 0; i < n; ++i)
        if (status[i] != mjpeg::LM_MJPEG_OK) return fail(ctx, LM_ERR_INVALID, "frame %lld: %s", (long long)i, mjpeg::status_text(status[i]));
    return LM_OK;
}
}  // namespace

int lm_decode_mjpeg(lm_ctx *ctx, const uint8_t *payload, int payload_on_device, const int64_t *offsets, int64_t n, uint8_t *frames) {
    return entry(ctx, [&] { return decode_mjpeg_impl(ctx, payload, payload_on_device, offsets, n, frames); });
}

// ---- lm_decode_mpeg4 ---------------------------------------------------------------------------------------------------
namespace {
int decode_mpeg4_impl(lm_ctx *ctx, const uint8_t *extradata, int64_t extradata_len, const uint8_t *payload, int on_dev, const int64_t *offsets,
                      int64_t n, uint8_t *frames) {
    if (!ctx->configured) return fail(ctx, LM_ERR_STATE, "lm_decode_mpeg4 needs lm_configure first");
    if (n < 0) return fail(ctx, LM_ERR_INVALID, "negative frame count");
    ctx->ms_decode = 0.f;
    if (n == 0) return LM_OK;
    if (!payload || !offsets || !frames || extradata_len < 0 || (extradata_len > 0 && !extradata)) return fail(ctx, LM_ERR_INVALID, "null argument");
    if (n > INT32_MAX) return fail(ctx, LM_ERR_INVALID, "too many frames in one call");
    const int rows = ctx->cfg.vid_rows, cols = ctx->cfg.vid_cols;
    for (int64_t i = 0; i < n; ++i)
        if (offsets[i] < 0 || offsets[i + 1] < offsets[i]) return fail(ctx, LM_ERR_INVALID, "frame %lld: offsets must not decrease", (long long)i);
    if (rows > 8191 || cols > 8191) return fail(ctx, LM_ERR_INVALID, "an MPEG-4 frame is at most 8191 x 8191 pixels");
    mpeg4::Vol vol{};
    mpeg4::Vop vop0{};
    if (extradata_len > 0)
        if (int st = mpeg4::parse(extradata, extradata_len, rows, cols, false, vol, vop0))
            return fail(ctx, LM_ERR_INVALID, "MPEG-4 extradata: %s", mpeg4::status_text(st));
    cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
    auto &B = ctx->buf;
    using L = lm_ctx;
    if (int rc = grow(ctx, B[L::PNG_OFFS], (size_t)(n + 1) * sizeof(int64_t))) return rc;
    if (int rc = grow(ctx, B[L::PNG_STATUS], (size_t)n * sizeof(int32_t))) return rc;
    if (int rc = grow(ctx, B[L::MPEG4_VOP], (size_t)n * lm_mpeg4_vop_bytes() + lm_mpeg4_vol_bytes())) return rc;
    int64_t *d_offs = reinterpret_cast<int64_t *>(B[L::PNG_OFFS].p);
    int32_t *d_status = reinterpret_cast<int32_t *>(B[L::PNG_STATUS].p);
    uint8_t *d_vop = B[L::MPEG4_VOP].p, *d_vol = d_vop + (size_t)n * lm_mpeg4_vop_bytes();
    CK(cudaMemcpyAsync(d_offs, offsets, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));

    // Every frame's VOP header, in order: parsed here from a host payload, by k_mpeg4_locate from a device payload
    std::vector<mpeg4::Vop> vops((size_t)n);
    std::vector<int32_t> status((size_t)n, 0);
    if (!on_dev) {
        for (int64_t f = 0; f < n; ++f) {
            int s = mpeg4::parse(payload + offsets[f], offsets[f + 1] - offsets[f], rows, cols, true, vol, vops[(size_t)f]);
            if (s == mpeg4::LM_MPEG4_OK && vops[(size_t)f].type == mpeg4::VOP_N) s = mpeg4::LM_MPEG4_NOT_CODED;
            if (s == mpeg4::LM_MPEG4_OK && f == 0 && vops[0].type != mpeg4::VOP_I) s = mpeg4::LM_MPEG4_FIRST_NOT_I;
            if (s) return fail(ctx, LM_ERR_INVALID, "frame %lld: %s", (long long)f, mpeg4::status_text(s));
        }
        CK(cudaMemcpyAsync(d_vop, vops.data(), (size_t)n * sizeof(mpeg4::Vop), cudaMemcpyHostToDevice, st));
        CK(cudaMemsetAsync(d_status, 0, (size_t)n * sizeof(int32_t), st));
    } else {
        CK(cudaMemcpyAsync(d_vol, &vol, sizeof vol, cudaMemcpyHostToDevice, st));
        if (lm_launch_mpeg4_locate(payload, d_offs, (int)n, rows, cols, d_vol, !vol.valid, d_vop, d_status, st) < 0)
            return fail(ctx, LM_ERR_RUNTIME, "MPEG-4 locate launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        CK(cudaMemcpyAsync(vops.data(), d_vop, (size_t)n * sizeof(mpeg4::Vop), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(status.data(), d_status, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int64_t f = 0; f < n; ++f)
            if (status[(size_t)f]) return fail(ctx, LM_ERR_INVALID, "frame %lld: %s", (long long)f, mpeg4::status_text(status[(size_t)f]));
    }

    // Pieces of consecutive frames share the scratch (coefficients, macroblock records, prediction state) and, from the host,
    // one of two staging buffers: the copy of piece k + 1 (copy stream) overlaps the decode of piece k.  A piece's segments
    // start at its first frame and at each I-VOP; every segment has two reference planes.
    const int mbw = (cols + 15) / 16, mbh = (rows + 15) / 16;
    const int64_t nmb = (int64_t)mbw * mbh, plane = lm_mpeg4_plane_bytes(rows, cols), lines = lm_mpeg4_lines_bytes(cols);
    const size_t per_frame = (size_t)nmb * (mpeg4::BLOCKS_PER_MB * 64 * sizeof(int16_t) + lm_mpeg4_info_bytes()) + (size_t)lines;
    const size_t scratch_budget = (size_t)4 << 30, stage_budget = (size_t)2 << 30;
    constexpr int max_segs = 256;
    const int64_t max_piece = std::max<int64_t>(1, std::min<int64_t>(on_dev ? 2048 : std::max<int64_t>(512, (n + 3) / 4), scratch_budget / per_frame));
    struct Piece {
        int64_t s, e;
        int seg0, nseg, seg_len;  // its segments: entries seg0 .. seg0 + nseg - 1 of segs
    };
    std::vector<Piece> pieces;
    std::vector<int32_t> segs;  // (first frame in the piece, frames) per segment
    size_t stage_need = 0;
    int64_t piece_max = 0;
    int segs_max = 0;
    for (int64_t s = 0; s < n;) {
        Piece P{s, s, (int)(segs.size() / 2), 0, 0};
        for (int64_t e = s; e < n; ++e) {
            const bool starts = e == s || vops[(size_t)e].type == mpeg4::VOP_I;
            if (e > s && (e - s >= max_piece || (starts && P.nseg == max_segs) ||
                          (!on_dev && (size_t)(offsets[e + 1] - offsets[s]) > stage_budget)))
                break;
            if (starts) {
                segs.push_back((int32_t)(e - s));
                segs.push_back(0);
                ++P.nseg;
            }
            ++segs.back();
            P.seg_len = std::max<int>(P.seg_len, segs.back());
            P.e = e + 1;
        }
        pieces.push_back(P);
        stage_need = std::max(stage_need, (size_t)(offsets[P.e] - offsets[P.s]));
        piece_max = std::max(piece_max, P.e - P.s);
        segs_max = std::max(segs_max, P.nseg);
        s = P.e;
    }
    if (int rc = grow(ctx, B[L::PNG_SCRATCH], (size_t)piece_max * nmb * mpeg4::BLOCKS_PER_MB * 64 * sizeof(int16_t))) return rc;
    if (int rc = grow(ctx, B[L::MPEG4_INFO], (size_t)piece_max * nmb * lm_mpeg4_info_bytes())) return rc;
    if (int rc = grow(ctx, B[L::MPEG4_LINES], (size_t)piece_max * lines)) return rc;
    if (int rc = grow(ctx, B[L::MPEG4_PLANES], (size_t)(2 * segs_max + 1) * plane)) return rc;  // + the carried plane
    if (int rc = grow(ctx, B[L::MPEG4_SEGS], segs.size() * sizeof(int32_t))) return rc;
    uint8_t *planes = B[L::MPEG4_PLANES].p, *carry = planes + (size_t)2 * segs_max * plane;
    int32_t *d_segs = reinterpret_cast<int32_t *>(B[L::MPEG4_SEGS].p);
    CK(cudaMemcpyAsync(d_segs, segs.data(), segs.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (!on_dev) {
        for (int k = 0; k < 2 && k < (int)pieces.size(); ++k)
            if (int rc = grow(ctx, B[L::PNG_STAGE0 + k], std::max<size_t>(stage_need, 1))) return rc;
        for (int k = 0; k < 2; ++k) {
            if (!ctx->ev_png_copy[k]) CK(cudaEventCreateWithFlags(&ctx->ev_png_copy[k], cudaEventDisableTiming));
            if (!ctx->ev_png_done[k]) CK(cudaEventCreateWithFlags(&ctx->ev_png_done[k], cudaEventDisableTiming));
        }
    }
    struct Events {  // start / end of each piece's decode launches, for ms_decode
        std::vector<cudaEvent_t> ev;
        ~Events() {
            for (cudaEvent_t e : ev) cudaEventDestroy(e);
        }
    } T;
    T.ev.resize(2 * pieces.size());
    for (auto &e : T.ev) CK(cudaEventCreate(&e));
    for (size_t k = 0; k < pieces.size(); ++k) {
        const Piece &P = pieces[k];
        const uint8_t *src = payload;
        int64_t base = 0;
        if (!on_dev) {
            uint8_t *stg = B[L::PNG_STAGE0 + (k & 1)].p;
            if (k >= 2) CK(cudaStreamWaitEvent(cp, ctx->ev_png_done[k & 1], 0));  // piece k - 2 no longer reads this buffer
            CK(cudaMemcpyAsync(stg, payload + offsets[P.s], (size_t)(offsets[P.e] - offsets[P.s]), cudaMemcpyHostToDevice, cp));
            CK(cudaEventRecord(ctx->ev_png_copy[k & 1], cp));
            CK(cudaStreamWaitEvent(st, ctx->ev_png_copy[k & 1], 0));
            src = stg;
            base = offsets[P.s];
        }
        CK(cudaEventRecord(T.ev[2 * k], st));
        if (lm_launch_mpeg4_decode(src, d_offs + P.s, base, (int)(P.e - P.s), d_vop + P.s * (int64_t)lm_mpeg4_vop_bytes(), rows, cols,
                                   B[L::MPEG4_INFO].p, B[L::PNG_SCRATCH].as<int16_t>(), B[L::MPEG4_LINES].p, d_segs + 2 * P.seg0, P.nseg,
                                   P.seg_len, planes, carry, d_status + P.s, frames + P.s * (int64_t)rows * cols, st) < 0)
            return fail(ctx, LM_ERR_RUNTIME, "MPEG-4 decode launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        // the piece's last frame, which the next piece's first segment may continue
        const int32_t last_len = segs[(size_t)2 * (P.seg0 + P.nseg - 1) + 1];
        CK(cudaMemcpyAsync(carry, planes + (size_t)(2 * (P.nseg - 1) + ((last_len - 1) & 1)) * plane, (size_t)plane, cudaMemcpyDeviceToDevice, st));
        CK(cudaEventRecord(T.ev[2 * k + 1], st));
        if (!on_dev) CK(cudaEventRecord(ctx->ev_png_done[k & 1], st));
    }
    CK(cudaMemcpyAsync(status.data(), d_status, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (size_t k = 0; k < pieces.size(); ++k) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, T.ev[2 * k], T.ev[2 * k + 1]) == cudaSuccess) ctx->ms_decode += t;
    }
    for (int64_t i = 0; i < n; ++i)
        if (status[(size_t)i] != mpeg4::LM_MPEG4_OK) return fail(ctx, LM_ERR_INVALID, "frame %lld: %s", (long long)i, mpeg4::status_text(status[(size_t)i]));
    return LM_OK;
}
}  // namespace

int lm_decode_mpeg4(lm_ctx *ctx, const uint8_t *extradata, int64_t extradata_len, const uint8_t *payload, int payload_on_device,
                    const int64_t *offsets, int64_t n, uint8_t *frames) {
    return entry(ctx, [&] { return decode_mpeg4_impl(ctx, extradata, extradata_len, payload, payload_on_device, offsets, n, frames); });
}

int lm_decode_ffv1(lm_ctx *ctx, const uint8_t *extradata, int64_t extradata_len, const uint8_t *payload, int payload_on_device,
                   const int64_t *offsets, int64_t n, uint8_t *frames) {
    return entry(ctx, [&] { return decode_ffv1_impl(ctx, extradata, extradata_len, payload, payload_on_device, offsets, n, frames); });
}

int lm_decode_png(lm_ctx *ctx, const uint8_t *payload, int payload_on_device, const int64_t *offsets, int64_t n, uint8_t *frames) {
    return entry(ctx, [&] { return decode_png_impl(ctx, payload, payload_on_device, offsets, n, frames); });
}

int lm_last_timing(const lm_ctx *ctx, float ms[7], int64_t *launches) {
    if (!ctx) return LM_ERR_INVALID;
    if (ms) memcpy(ms, ctx->ms, sizeof ctx->ms);
    if (launches) *launches = ctx->launches;
    return LM_OK;
}

// items 4 .. 6: the last chunk of the last pass-1 call
static int64_t debug_fetch_p1(lm_ctx *ctx, int what, int64_t frame, void *dst, int64_t dst_bytes, int32_t dims[4]) {
    const auto &q = ctx->p1;
    if (!q.method) return fail(ctx, LM_ERR_STATE, "no pass-1 call has finished on this context");
    const int64_t i = frame - q.s0;
    if (i < 0 || i >= q.B) return fail(ctx, LM_ERR_INVALID, "frame %lld is not in the last chunk of the last pass-1 call", (long long)frame);
    if (what != 6 && q.method == LM_P1_TM_DE) return fail(ctx, LM_ERR_INVALID, "lm_bounding_box_tm_de keeps no bit images");
    int32_t d[4] = {q.rows, q.wpr, q.width, q.method};
    if (what == 6) d[0] = 1, d[1] = q.nsums;
    const int64_t bytes = (int64_t)d[0] * d[1] * 4;
    const auto &b = ctx->buf[what == 4 ? lm_ctx::P1_BITS0 : what == 5 ? lm_ctx::P1_BITS1 : lm_ctx::P1_SUMS];
    if (dims) memcpy(dims, d, sizeof d);
    if (!dst || dst_bytes < bytes) return fail(ctx, LM_ERR_INVALID, "debug buffer too small (%lld needed)", (long long)bytes);
    DeviceGuard guard(ctx->device);
    cudaError_t e = cudaMemcpyAsync(dst, b.p + i * bytes, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(ctx, LM_ERR_RUNTIME, "cudaMemcpy: %s", cudaGetErrorString(e));
    return bytes;
}

int64_t lm_debug_fetch(lm_ctx *ctx, int what, int64_t frame, void *dst, int64_t dst_bytes, int32_t dims[4]) {
    if (ctx && what >= 4 && what <= 6) return debug_fetch_p1(ctx, what, frame, dst, dst_bytes, dims);
    if (!ctx || !ctx->Bcap) return LM_ERR_STATE;
    const int64_t i = frame - ctx->last_s0;
    if (i < 0 || i >= ctx->last_B) return fail(ctx, LM_ERR_INVALID, "frame %lld is not in the last sub-batch", (long long)frame);
    DeviceGuard guard(ctx->device);
    const LmBatch &b = ctx->last_slot ? ctx->bt_more[ctx->last_slot - 1] : ctx->bt;
    const void *src = nullptr;
    int64_t bytes = 0;
    int32_t d[4] = {0, 0, 0, 0};
    switch (what) {
        case 0:
        case 1: {
            const LmView &V = b.view[what];
            src = b.win[what] + i * V.win_stride;
            bytes = V.win_stride;
            d[0] = V.win_h; d[1] = V.win_pitch; d[2] = V.halo_y; d[3] = V.halo_x;
            break;
        }
        case 2:
            src = b.tailmask + i * b.bb_h[LM_BOTTOM] * b.tail_pitch;
            bytes = (int64_t)b.bb_h[LM_BOTTOM] * b.tail_pitch;
            d[0] = b.bb_h[LM_BOTTOM]; d[1] = b.tail_pitch; d[2] = b.tail_w;
            break;
        case 3:
            src = b.minmax + (i + 1) * 2;
            bytes = 8;
            d[0] = 2;
            break;
        default:
            return fail(ctx, LM_ERR_INVALID, "unknown debug item %d", what);
    }
    if (dims) memcpy(dims, d, sizeof d);
    if (!dst || dst_bytes < bytes) return fail(ctx, LM_ERR_INVALID, "debug buffer too small (%lld needed)", (long long)bytes);
    cudaError_t e = cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(ctx, LM_ERR_RUNTIME, "cudaMemcpy: %s", cudaGetErrorString(e));
    return bytes;
}

}  // extern "C"
