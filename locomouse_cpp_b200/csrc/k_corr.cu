// k_corr.cu — template correlation (the dominant kernel; FP32-FMA bound).
//
// Replaces the six cv::filter2D calls of the reference hot loop (LocoMouse_class.cpp:845, 860,
// 2575-2576) plus the score consumers that directly follow them: threshold(>0) of the tail scores
// (2593-2594), `setTo(0, mask)` with mask = px <= 25 (782, 817, 849, 864) and the row-major scan
// for positive detections (1638-1648, 1776-1786).
//
// Numerics contract (SURVEY Q1, oracle/lm_oracle.cpp correlate_rows): every output pixel owns ONE
// fp32 accumulator initialised to float(-rho) and visits the taps in row-major order; FMA mode
// rounds once per tap (FFMA), the other mode twice (FMUL + FADD).  One thread owns a TY x TX patch
// of outputs, so the per-output operation order is exactly the oracle's -> bit-exact scores.
//
// Mapping: a "task" is one TY x TX output patch; the tasks of one (view, template) box are numbered
// row-major and dealt to CTAs 256 at a time, so every warp but the last of a box has 32 busy lanes.
// The CTA stages the window rows it needs (u8 -> fp32, full box width + halo) in shared memory
// once, next to the zero-padded template; the inner loop then issues only LDS.128 + FFMA:
// TY*KW*TX FFMA per (TX+KW-1)/4 pixel LDS.128 and TY*KW/4 weight LDS.128 (broadcast).
#include "lm_internal.h"
#include "corr_common.cuh"

namespace {

constexpr int CORR_THREADS = 256;

struct CorrJob {
    int view, feat, is_tail;
    int x_begin;             // first output column of this strip (wide boxes are cut into column strips)
    int out_w, out_h;        // outputs computed by this job: strip width x box_h
    int ngx, ntasks;         // column groups, total tasks
    int cta_begin, ncta;     // CTA range inside a frame's block of CTAs
    int off_x, off_y;        // window column/row of tap (0,0) for output (0,0): halo - anchor
    int kh, kwp4;            // template rows, smem row stride (floats)
    int pitch;               // smem tile pitch (floats)
    int ax, ay;
    float init;
    const float *w;          // device template, row stride kwp4? no: kwp (see LmTemplateDev)
    int w_stride;
};

constexpr int MAX_JOBS = 24;

struct CorrParams {
    CorrJob job[MAX_JOBS];
    int njobs;
    int ctas_per_frame;
    int B;
    int det_cap;
    int box_w[2];            // bb_w per view (index space of LmDet.idx)
    int win_w[2], win_h[2], win_pitch[2];
    int64_t win_stride[2];
    const uint8_t *win[2];
    uint8_t *tailbin[2];
    int tail_pitch;
    int64_t tailbin_stride[2];
    LmDet *det;
    int32_t *det_count;
};


template <int KW, int TX, int TY, bool FMA>
__global__ void __launch_bounds__(CORR_THREADS, (KW <= 32) ? 2 : 1) k_corr(const __grid_constant__ CorrParams P) {
    constexpr int NP = ((TX + KW - 1 + 3) / 4) * 4;  // pixel registers per tile row (multiple of 4)
    constexpr int KW4 = ((KW + 3) / 4) * 4;
    extern __shared__ __align__(16) float smem[];

    const int f = blockIdx.x / P.ctas_per_frame;
    const int c = blockIdx.x - f * P.ctas_per_frame;
    int ji = 0;
    for (int q = 1; q < P.njobs; ++q)
        if (c >= P.job[q].cta_begin) ji = q;
    const CorrJob &J = P.job[ji];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int first_task = (c - J.cta_begin) * CORR_THREADS;
    const int ntask_cta = min(CORR_THREADS, J.ntasks - first_task);
    const int rg_first = first_task / J.ngx;
    const int rg_last = (first_task + ntask_cta - 1) / J.ngx;
    const int tile_rows = (rg_last - rg_first + 1) * TY + J.kh - 1;
    const int pitch = J.pitch;

    float *wsm = smem;                       // [kh][KW4]
    float *tile = smem + J.kh * KW4;         // [tile_rows][pitch]

    // ---- stage template (zero padded to KW4) and window rows (u8 -> f32) -------------------------
    for (int idx = tid; idx < J.kh * KW4; idx += CORR_THREADS) {
        int j = idx / KW4, i = idx - j * KW4;
        wsm[idx] = (i < J.w_stride) ? J.w[j * J.w_stride + i] : 0.f;
    }
    {
        // Window rows -> fp32 tile.  All of a thread's global loads of a batch are issued before any is
        // consumed (8 independent 32-bit loads in flight per thread), so the staging costs about one L2
        // round trip per batch instead of one per word; bytes become floats with the 2^23 magic-number
        // trick (PRMT + FADD, exact for 0..255) instead of the quarter-rate I2F pipe.
        const int v = J.view;
        const uint8_t *wbase = P.win[v] + (int64_t)f * P.win_stride[v];
        const int win_w = P.win_w[v], win_h = P.win_h[v], wp = P.win_pitch[v];
        const int row0 = rg_first * TY + J.off_y;
        const int p4 = pitch >> 2;
        const int nq = tile_rows * p4;
        constexpr int SB = 8;
        for (int base = 0; base < nq; base += CORR_THREADS * SB) {
            uint32_t u[SB];
#pragma unroll
            for (int q = 0; q < SB; ++q) {
                const int idx = base + q * CORR_THREADS + tid;
                uint32_t w = 0u;
                if (idx < nq) {
                    const int r = idx / p4, c4 = idx - r * p4;
                    const int wr = row0 + r, wc = J.off_x + c4 * 4;
                    if (wr >= 0 && wr < win_h) {
                        const uint8_t *src = wbase + (int64_t)wr * wp;
                        if (((wc & 3) == 0) && wc >= 0 && wc + 4 <= wp) {
                            // window rows are zero padded up to the pitch, so a full word is always valid
                            w = __ldg(reinterpret_cast<const uint32_t *>(src + wc));
                        } else {
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const int cc = wc + e;
                                if (cc >= 0 && cc < win_w) w |= (uint32_t)__ldg(src + cc) << (8 * e);
                            }
                        }
                    }
                }
                u[q] = w;
            }
#pragma unroll
            for (int q = 0; q < SB; ++q) {
                const int idx = base + q * CORR_THREADS + tid;
                if (idx < nq) {
                    float4 o;
                    o.x = __uint_as_float(__byte_perm(u[q], 0x4B000000u, 0x7540)) - 8388608.f;
                    o.y = __uint_as_float(__byte_perm(u[q], 0x4B000000u, 0x7541)) - 8388608.f;
                    o.z = __uint_as_float(__byte_perm(u[q], 0x4B000000u, 0x7542)) - 8388608.f;
                    o.w = __uint_as_float(__byte_perm(u[q], 0x4B000000u, 0x7543)) - 8388608.f;
                    reinterpret_cast<float4 *>(tile)[idx] = o;
                }
            }
        }
    }
    __syncthreads();
    if (warp * 32 >= ntask_cta) return;  // idle warps of the last CTA of a box

    const bool active = tid < ntask_cta;
    const int task = first_task + (active ? tid : 0);
    const int rg = task / J.ngx;
    const int cg = task - rg * J.ngx;
    const int rbase = (rg - rg_first) * TY;

    float acc[TY][TX];
#pragma unroll
    for (int t = 0; t < TY; ++t)
#pragma unroll
        for (int k = 0; k < TX; ++k) acc[t][k] = J.init;

    const float *prow = tile + rbase * pitch + cg * TX;
    const int kh = J.kh;
    const int nr = kh + TY - 1;
    // Tile row r feeds output row t with kernel row j = r - t.  A kernel row is applied in two halves
    // (taps [0,H0) then [H0,KW)): per accumulator the tap order is unchanged, but each half needs only
    // ~TX+KW/2 pixel registers, which leaves room to double-buffer them: while one half is being
    // multiplied the pixels of the next half (or of the next tile row) are already in flight, so the
    // steady state never waits at a shared-memory load.  Rows 0..TY-2 and kh..kh+TY-2 touch only some of
    // the TY output rows and run through the generic, branchy path.
    constexpr int H0 = (KW >= 8) ? (((KW / 2) + 3) / 4) * 4 : KW;
    constexpr int H1 = KW - H0;
    constexpr int NP0 = ((TX + H0 - 1 + 3) / 4) * 4;
    constexpr int NP1 = (H1 > 0) ? ((TX + H1 - 1 + 3) / 4) * 4 : 4;
    static_assert(H0 + NP1 <= NP + 4 && NP0 <= NP, "half windows stay inside the staged row");
    float pa[NP0], pb[NP1];
    auto generic_row = [&](int r) {
        load_pixels<NP0>(pa, prow + r * pitch);
        if (H1 > 0) load_pixels<NP1>(pb, prow + r * pitch + H0);
#pragma unroll
        for (int t = 0; t < TY; ++t) {
            const int j = r - t;
            if (j >= 0 && j < kh) {
                corr_taps<H0, TX, FMA, NP0>(acc[t], pa, wsm + j * KW4);
                if (H1 > 0) corr_taps<(H1 > 0 ? H1 : 1), TX, FMA, NP1>(acc[t], pb, wsm + j * KW4 + H0);
            }
        }
    };
    if (kh >= TY) {
        for (int r = 0; r < TY - 1; ++r) generic_row(r);
        load_pixels<NP0>(pa, prow + (TY - 1) * pitch);
        for (int r = TY - 1; r < kh; ++r) {
            if (H1 > 0) load_pixels<NP1>(pb, prow + r * pitch + H0);
#pragma unroll
            for (int t = 0; t < TY; ++t) corr_taps<H0, TX, FMA, NP0>(acc[t], pa, wsm + (r - t) * KW4);
            load_pixels<NP0>(pa, prow + (r + 1) * pitch);
            if (H1 > 0) {
#pragma unroll
                for (int t = 0; t < TY; ++t)
                    corr_taps<(H1 > 0 ? H1 : 1), TX, FMA, NP1>(acc[t], pb, wsm + (r - t) * KW4 + H0);
            }
        }
        for (int r = kh; r < nr; ++r) generic_row(r);
    } else {
        for (int r = 0; r < nr; ++r) generic_row(r);
    }

    // ---- epilogue ------------------------------------------------------------------------------------
    const int x0 = cg * TX, y0 = rg * TY;
    if (J.is_tail) {
        if (!active) return;
        uint8_t *tb = P.tailbin[J.view] + (int64_t)f * P.tailbin_stride[J.view];
#pragma unroll
        for (int t = 0; t < TY; ++t) {
            const int y = y0 + t;
            if (y >= J.out_h) continue;
#pragma unroll
            for (int k = 0; k < TX; ++k) {
                const int x = x0 + k;
                if (x < J.out_w) tb[(int64_t)y * P.tail_pitch + J.x_begin + x] = acc[t][k] > 0.f ? 1 : 0;
            }
        }
        return;
    }
    // paw / snout: positives that are not masked by (px <= 25); TAIL_MASK is applied by the NMS kernel
    unsigned hit = 0;  // bit t*TX+k
    int cnt = 0;
    if (active) {
#pragma unroll
        for (int t = 0; t < TY; ++t) {
            const int y = y0 + t;
#pragma unroll
            for (int k = 0; k < TX; ++k) {
                const int x = x0 + k;
                if (y < J.out_h && x < J.out_w && acc[t][k] > 0.f) {
                    const float centre = tile[(rbase + t + J.ay) * pitch + x + J.ax];
                    if (centre > 25.f) {
                        hit |= 1u << (t * TX + k);
                        ++cnt;
                    }
                }
            }
        }
    }
    static_assert(TX * TY <= 32, "hit mask is 32 bits");
    const unsigned any = __ballot_sync(0xffffffffu, cnt > 0);
    if (!any) return;
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    const int list = (f * 2 + J.feat) * 2 + J.view;
    int base = 0;
    if (lane == 31) base = atomicAdd(&P.det_count[list], total);
    base = __shfl_sync(0xffffffffu, base, 31);
    int o = base + incl - cnt;
    LmDet *out = P.det + (int64_t)list * P.det_cap;
    const int bw = P.box_w[J.view];
#pragma unroll
    for (int t = 0; t < TY; ++t)
#pragma unroll
        for (int k = 0; k < TX; ++k)
            if (hit & (1u << (t * TX + k))) {
                if (o < P.det_cap) {
                    LmDet d;
                    d.idx = (uint32_t)((y0 + t) * bw + J.x_begin + x0 + k);
                    d.score = acc[t][k];
                    out[o] = d;
                }
                ++o;
            }
}

constexpr int kTX = 8, kTY = 4;
const int kKwp[] = {8, 16, 24, 30, 32, 48, 60, 64};

template <int KW>
cudaError_t launch_kw(const CorrParams &P, size_t smem, bool fma, cudaStream_t s) {
    auto kf = k_corr<KW, kTX, kTY, true>;
    auto km = k_corr<KW, kTX, kTY, false>;
    static LmDevOnce once;
    if (auto setup = once.first()) {
        cudaError_t e = lm_allow_max_dynamic_smem(kf);
        if (e == cudaSuccess) e = lm_allow_max_dynamic_smem(km);
        if (e != cudaSuccess) return e;
    }
    if (fma)
        kf<<<P.B * P.ctas_per_frame, CORR_THREADS, smem, s>>>(P);
    else
        km<<<P.B * P.ctas_per_frame, CORR_THREADS, smem, s>>>(P);
    return cudaGetLastError();
}

size_t job_smem(const CorrJob &J) {
    // worst case rows: a CTA's 256 tasks span at most ceil(255 / ngx) + 1 row groups
    int rgs = (CORR_THREADS - 1) / J.ngx + 2;
    int total_rg = (J.out_h + kTY - 1) / kTY;
    if (rgs > total_rg) rgs = total_rg;
    size_t rows = (size_t)rgs * kTY + J.kh - 1;
    return ((size_t)J.kh * J.kwp4 + rows * J.pitch) * sizeof(float);
}

int full_out_w(const LmBatch &b, int view, int feat) { return feat == LM_TAIL ? b.tail_w : b.view[view].box_w; }

CorrJob make_job(const LmBatch &b, int view, int feat, int kwp, int x_begin, int strip_w) {
    const LmTemplateDev &T = b.tmpl[view][feat];
    const LmView &V = b.view[view];
    CorrJob J{};
    J.view = view;
    J.feat = feat;
    J.is_tail = (feat == LM_TAIL);
    J.x_begin = x_begin;
    J.out_w = strip_w;
    J.out_h = V.box_h;
    J.ngx = (J.out_w + kTX - 1) / kTX;
    int ngy = (J.out_h + kTY - 1) / kTY;
    J.ntasks = J.ngx * ngy;
    J.ncta = (J.ntasks + CORR_THREADS - 1) / CORR_THREADS;
    J.off_x = V.halo_x - T.ax + x_begin;
    J.off_y = V.halo_y - T.ay;
    J.kh = T.kh;
    J.kwp4 = ((kwp + 3) / 4) * 4;
    int np = ((kTX + kwp - 1 + 3) / 4) * 4;
    J.pitch = (J.ngx - 1) * kTX + np;
    J.ax = T.ax;
    J.ay = T.ay;
    J.init = T.init;
    J.w = T.w;
    J.w_stride = T.kwp;
    return J;
}

}  // namespace

int lm_corr_kwp(int kw) {
    for (int v : kKwp)
        if (v >= kw) return v;
    return -1;
}

// Column strips: the narrowest split of the box whose tile fits the shared-memory budget
// (two CTAs per SM for kernel rows up to 32 taps, one CTA per SM beyond).
static int strip_width(const LmBatch &b, int view, int feat, int kwp, size_t *smem_out) {
    const size_t budget = (kwp <= 32) ? 110 * 1024 : 224 * 1024;
    const int W = full_out_w(b, view, feat);
    for (int ns = 1; ns <= W; ++ns) {
        int sw = (((W + ns - 1) / ns + kTX - 1) / kTX) * kTX;
        CorrJob J = make_job(b, view, feat, kwp, 0, sw);
        size_t sm = job_smem(J);
        if (sm <= budget || sw <= kTX) {
            if (smem_out) *smem_out = sm;
            return sw;
        }
    }
    return kTX;
}

size_t lm_corr_smem_bytes(const LmBatch &b, int view, int feat) {
    int kwp = lm_corr_kwp(b.tmpl[view][feat].kw);
    if (kwp < 0) return (size_t)-1;
    size_t sm = 0;
    strip_width(b, view, feat, kwp, &sm);
    return sm;
}

// One launch per distinct padded kernel width; all (view, template) boxes that share it ride in the
// same grid so the tail of one box overlaps the head of the next.
int lm_launch_corr(const LmBatch &b, cudaStream_t s) {
    int launches = 0;
    bool done[2][3] = {};
    for (int v0 = 0; v0 < 2; ++v0)
        for (int k0 = 0; k0 < 3; ++k0) {
            if (done[v0][k0]) continue;
            const int kwp = lm_corr_kwp(b.tmpl[v0][k0].kw);
            CorrParams P{};
            size_t smem = 0;
            int cta = 0;
            for (int v = 0; v < 2; ++v)
                for (int k = 0; k < 3; ++k) {
                    if (done[v][k] || lm_corr_kwp(b.tmpl[v][k].kw) != kwp) continue;
                    if (k == LM_TAIL && b.tail_w <= 0) {
                        done[v][k] = true;
                        continue;
                    }
                    const int W = full_out_w(b, v, k);
                    const int sw = strip_width(b, v, k, kwp, nullptr);
                    for (int xb = 0; xb < W; xb += sw) {
                        if (P.njobs >= MAX_JOBS) return -1;
                        CorrJob J = make_job(b, v, k, kwp, xb, (W - xb < sw) ? (W - xb) : sw);
                        J.cta_begin = cta;
                        cta += J.ncta;
                        size_t sm = job_smem(J);
                        if (sm > smem) smem = sm;
                        P.job[P.njobs++] = J;
                    }
                    done[v][k] = true;
                }
            if (!P.njobs) continue;
            P.ctas_per_frame = cta;
            P.B = b.B;
            P.det_cap = b.det_cap;
            for (int v = 0; v < 2; ++v) {
                P.box_w[v] = b.view[v].box_w;
                P.win_w[v] = b.view[v].win_w;
                P.win_h[v] = b.view[v].win_h;
                P.win_pitch[v] = b.view[v].win_pitch;
                P.win_stride[v] = b.view[v].win_stride;
                P.win[v] = b.win[v];
                P.tailbin[v] = b.tailbin[v];
                P.tailbin_stride[v] = (int64_t)b.bb_h[v] * b.tail_pitch;
            }
            P.tail_pitch = b.tail_pitch;
            P.det = b.det;
            P.det_count = b.det_count;
            cudaError_t e = cudaSuccess;
            const bool fma = b.fma_mode != 0;
            switch (kwp) {
                case 8: e = launch_kw<8>(P, smem, fma, s); break;
                case 16: e = launch_kw<16>(P, smem, fma, s); break;
                case 24: e = launch_kw<24>(P, smem, fma, s); break;
                case 30: e = launch_kw<30>(P, smem, fma, s); break;
                case 32: e = launch_kw<32>(P, smem, fma, s); break;
                case 48: e = launch_kw<48>(P, smem, fma, s); break;
                case 60: e = launch_kw<60>(P, smem, fma, s); break;
                case 64: e = launch_kw<64>(P, smem, fma, s); break;
                default: e = cudaErrorInvalidValue;
            }
            if (e != cudaSuccess) return -1;
            ++launches;
        }
    return launches;
}
