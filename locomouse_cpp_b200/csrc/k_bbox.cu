// k_bbox.cu — pass 1 of LocoMouse_TM_DE on the device (SURVEY §8f-1): the per-frame part of
// LocoMouse_TM_DE::computeBoundingBox / computeMouseBox_DE (LocoMouse_TM_DE.cpp:8-113).
//
// The reference reads every frame with the base-class readFrame (subtract, normalise, calibration gather, flip;
// class.cpp:1273-1333), stretches the side view with imadjust_default (3244-3311), zeroes four border bands
// (TM_DE.cpp:68-71), thresholds (75), sums columns (91) and takes the first / last column whose sum reaches
// MIN_PIXEL_COUNT (firstLastOverT, class.hpp:411-442).  Every pixel operation after the gather is a 256-entry
// look-up, so no image is materialised:
//   k_minmax + k_lut (k_pre.cu)  per-frame min/max of sat(F - BKG) -> normalisation LUT  (imadjust(0, 0.6) off)
//   k_bb_hist16 histogram of the normalised side view, gathered ONCE through the calibration map (16-pixel runs as aligned
//               words where the folded map allows, as in k_prep); the raw differences are kept, one byte per pixel
//               (k_bb_hist: the per-pixel gather without the folded arrays, used by LocoMouse_TM's front end)
//   k_bb_pred   one thread replays imadjust_default's float cumulative scan (order matters), all threads then build
//               pred[d] = ( imadjust_default( normalise(d) ) > threshold )
//   k_bb_cols   column sums of pred over the rows / columns that survive the zeroed bands (streamed from the kept
//               differences), stored per frame (lm_debug_fetch item 6), first / last, bb_x
// The whole-video moving average that follows is sequential and stays on the host (lm_moving_average).
#include <cstdlib>

#include "lm_internal.h"

namespace {

struct BBoxDev {
    const uint8_t *frames;
    int64_t frame_bytes;
    const uint8_t *bkg;
    const int32_t *calib;
    int n_cols, flip, B;
    lm_bb_de_params p;
    const uint8_t *lut;   // [B + 1][256] normalisation LUT, slot f + 1
    uint32_t *hist;       // [B][256]
    uint8_t *pred;        // [B][256]
    const int32_t *calib_flip;   // folded per-video arrays of k_fold_calib (k_pre.cu); all three set: k_bb_hist16 runs
    const uint8_t *bkg_warp, *run_mode;
    uint8_t *diff;        // [B][side_h * side_w] raw difference sat(F - BKG) of every side-view pixel, written by k_bb_hist (may be null)
    double *bb_x;         // [B]
    int32_t *lims;        // [B][2]
    int32_t *sums;        // [B][side_w] column sums (null: not kept)
};

__global__ void __launch_bounds__(256) k_bb_hist(const __grid_constant__ BBoxDev P) {
    // per-warp private histograms; a dark side view puts most pixels into a handful of bins (32 lanes hitting one
    // shared-memory word would serialise), so the most common values are counted in registers (below)
    __shared__ uint32_t sh[8][256];
    __shared__ uint8_t lut[256];
    const int f = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < 8 * 256; i += 256) (&sh[0][0])[i] = 0;
    lut[tid] = P.lut[(f + 1) * 256 + tid];
    __syncthreads();
    const uint8_t *F = P.frames + (int64_t)f * P.frame_bytes;
    const int npx = P.p.side_w * P.p.side_h;
    // each lane takes UNR pixels per step, 32 * UNR consecutive pixels per warp; all calibration loads of a step are
    // issued first, then all frame / background loads: the gather chain is latency-bound otherwise
    constexpr int UNR = 8;
    const int stride = gridDim.x * 256 * UNR;
    uint32_t low[4] = {0u, 0u, 0u, 0u};
    for (int i0 = (blockIdx.x * 256 + warp * 32) * UNR; i0 < npx; i0 += stride) {
        int idx[UNR], bin[UNR];
#pragma unroll
        for (int q = 0; q < UNR; ++q) {
            const int i = i0 + q * 32 + lane;
            idx[q] = -1;
            if (i < npx) {
                const int r = i / P.p.side_w, x = P.p.side_x + (i - r * P.p.side_w);
                const int xs = P.flip ? (P.n_cols - 1 - x) : x;
                idx[q] = __ldg(P.calib + (int64_t)(P.p.side_y + r) * P.n_cols + xs);
            }
        }
#pragma unroll
        for (int q = 0; q < UNR; ++q) {
            bin[q] = -1;
            if (idx[q] >= 0) {
                const int d = (int)__ldg(F + idx[q]) - (int)__ldg(P.bkg + idx[q]);
                bin[q] = d < 0 ? 0 : d;
                // the gathered difference is kept (one coalesced byte per pixel): k_bb_cols streams it instead of gathering
                // every pixel through the calibration map a second time
                if (P.diff) P.diff[(int64_t)f * npx + (i0 + q * 32 + lane)] = (uint8_t)bin[q];
            }
        }
        // Differences 0 .. 3 (the static background plus sensor noise: most of a side view) are counted in registers and
        // added once per thread at the end; only the rarer, more varied values go to the warp's shared-memory histogram.
#pragma unroll
        for (int q = 0; q < UNR; ++q) {
            const int d = bin[q];
            low[0] += d == 0;
            low[1] += d == 1;
            low[2] += d == 2;
            low[3] += d == 3;
            if (d >= 4) atomicAdd(&sh[warp][lut[d]], 1u);   // rarer and spread over many bins: few same-word collisions
        }
    }
#pragma unroll
    for (int d = 0; d < 4; ++d) {   // the four register counters, reduced over the warp, into this warp's histogram
        const uint32_t t = __reduce_add_sync(0xffffffffu, low[d]);
        if (lane == 0 && t) atomicAdd(&sh[warp][lut[d]], t);
        __syncwarp();
    }
    __syncthreads();
    uint32_t tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += sh[w][tid];
    if (tot) atomicAdd(&P.hist[f * 256 + tid], tot);
}

// The same histogram (and the stored differences) with k_prep's run tier: a thread takes 16 consecutive side-view pixels; where
// the calibration map says they come from 16 consecutive raw bytes (run_mode, folded once per video by k_fold_calib) they cost
// one map load, five aligned frame words and five background words instead of 16 dependent gather chains.  Differences 0 .. 3
// are counted with SIMD-in-a-word compares; the others go to the warp's shared-memory histogram one by one.
__global__ void __launch_bounds__(256) k_bb_hist16(const __grid_constant__ BBoxDev P) {
    __shared__ uint32_t sh[8][256];
    __shared__ uint8_t lut[256];
    const int f = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < 8 * 256; i += 256) (&sh[0][0])[i] = 0;
    lut[tid] = P.lut[(f + 1) * 256 + tid];
    __syncthreads();
    const uint8_t *F = P.frames + (int64_t)f * P.frame_bytes;
    const int fbytes = (int)P.frame_bytes;
    const int sw = P.p.side_w, nseg = (sw + 15) >> 4, items = nseg * P.p.side_h;
    uint8_t *D = P.diff + (int64_t)f * sw * P.p.side_h;
    uint32_t low[4] = {0u, 0u, 0u, 0u};
    for (int it = blockIdx.x * 256 + tid; it < items; it += gridDim.x * 256) {
        const int r = it / nseg, c16 = (it - r * nseg) << 4;
        const int valid = min(16, sw - c16);
        const int base = (P.p.side_y + r) * P.n_cols + P.p.side_x + c16;
        uint32_t d4[4] = {0u, 0u, 0u, 0u};
        bool done = false;
        if (valid == 16) {
            const int mode = __ldg(P.run_mode + base);
            if (mode & 12) {
                const int i0 = __ldg(P.calib_flip + base);
                const int lo_i = (mode & 4) ? i0 : i0 - 15;
                if (lo_i >= 4 && lo_i + 24 <= fbytes) {   // the aligned words read lie inside this frame's bytes
                    const uintptr_t a = reinterpret_cast<uintptr_t>(F) + (uintptr_t)(unsigned)lo_i;
                    const uint32_t *fp = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
                    const unsigned shf = ((unsigned)a & 3u) * 8u;
                    const uint32_t f0 = __ldg(fp), f1 = __ldg(fp + 1), f2 = __ldg(fp + 2), f3 = __ldg(fp + 3), f4 = __ldg(fp + 4);
                    uint32_t fw[4] = {__funnelshift_r(f0, f1, shf), __funnelshift_r(f1, f2, shf), __funnelshift_r(f2, f3, shf), __funnelshift_r(f3, f4, shf)};
                    if (!(mode & 4)) {   // descending run: pixel q is raw byte lo_i + 15 - q
                        const uint32_t t0 = __byte_perm(fw[3], 0u, 0x0123), t1 = __byte_perm(fw[2], 0u, 0x0123);
                        const uint32_t t2 = __byte_perm(fw[1], 0u, 0x0123), t3 = __byte_perm(fw[0], 0u, 0x0123);
                        fw[0] = t0; fw[1] = t1; fw[2] = t2; fw[3] = t3;
                    }
                    const uint32_t *kp = reinterpret_cast<const uint32_t *>(P.bkg_warp + (base & ~3));   // padded behind the last pixel
                    const unsigned ks = (unsigned)(base & 3) * 8u;
                    const uint32_t k0 = __ldg(kp), k1 = __ldg(kp + 1), k2 = __ldg(kp + 2), k3 = __ldg(kp + 3), k4 = __ldg(kp + 4);
                    d4[0] = __vsubus4(fw[0], __funnelshift_r(k0, k1, ks));   // per-byte max(F - BKG, 0)
                    d4[1] = __vsubus4(fw[1], __funnelshift_r(k1, k2, ks));
                    d4[2] = __vsubus4(fw[2], __funnelshift_r(k2, k3, ks));
                    d4[3] = __vsubus4(fw[3], __funnelshift_r(k3, k4, ks));
                    done = true;
                }
            }
        }
        if (!done) {
            for (int q = 0; q < valid; ++q) {
                const int d = max((int)__ldg(F + __ldg(P.calib_flip + base + q)) - (int)__ldg(P.bkg_warp + base + q), 0);
                d4[q >> 2] |= (uint32_t)d << (8 * (q & 3));
            }
        }
        // keep the differences for k_bb_cols (word stores where the row offset allows, bytes otherwise)
        const int o = r * sw + c16;
        if (valid == 16 && !(reinterpret_cast<uintptr_t>(D + o) & 3)) {
#pragma unroll
            for (int w = 0; w < 4; ++w) reinterpret_cast<uint32_t *>(D + o)[w] = d4[w];
        } else {
            for (int q = 0; q < valid; ++q) D[o + q] = (uint8_t)(d4[q >> 2] >> (8 * (q & 3)));
        }
        // histogram: bytes 0 .. 3 by SIMD compares (pixels beyond `valid` are zero bytes: taken off the zero count below)
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const uint32_t x = d4[w];
            low[0] += __popc(__vcmpeq4(x, 0x00000000u)) >> 3;
            low[1] += __popc(__vcmpeq4(x, 0x01010101u)) >> 3;
            low[2] += __popc(__vcmpeq4(x, 0x02020202u)) >> 3;
            low[3] += __popc(__vcmpeq4(x, 0x03030303u)) >> 3;
            uint32_t big = __vcmpgeu4(x, 0x04040404u) & 0x01010101u;   // one flag bit per byte >= 4
            while (big) {
                const int q = (__ffs(big) - 1) >> 3;
                big &= big - 1;
                atomicAdd(&sh[warp][lut[(x >> (8 * q)) & 0xffu]], 1u);
            }
        }
        low[0] -= (uint32_t)(16 - valid);
    }
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const uint32_t t = __reduce_add_sync(0xffffffffu, low[d]);
        if (lane == 0 && t) atomicAdd(&sh[warp][lut[d]], t);
        __syncwarp();
    }
    __syncthreads();
    uint32_t tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += sh[w][tid];
    if (tot) atomicAdd(&P.hist[f * 256 + tid], tot);
}


__global__ void __launch_bounds__(256) k_bb_pred(const __grid_constant__ BBoxDev P) {
    __shared__ float s_ab[2];
    __shared__ int s_identity;
    __shared__ uint32_t h[256];
    const int f = blockIdx.x, tid = threadIdx.x;
    h[tid] = P.hist[f * 256 + tid];
    __syncthreads();
    if (tid == 0) {
        // imadjust_default, LocoMouse_class.cpp:3258-3296, operation for operation (float scan, double cv::sum)
        double acc = 0.0;
        for (int i = 0; i < 256; ++i) acc = __dadd_rn(acc, (double)(float)h[i]);
        const float sum_histf = (float)acc;
        float cumsum = 0.f;
        int i0 = 0, i1 = 0, imin = 0, imax = 0;
        bool check_min = true, check_max = true;
        for (int i = 0; i < 256; ++i) {
            cumsum = __fadd_rn(cumsum, (float)h[i]);
            const float cn = __fdiv_rn(cumsum, sum_histf);
            if ((cn > 0.01f) & check_min) {
                i0 = i;
                check_min = false;
                imin = i;
            }
            if ((cn >= 0.99f) & check_max) {
                i1 = i;
                check_max = false;
                imax = i;
            }
            if (!(check_min || check_max)) break;
        }
        if (imin == imax) i1 = 256;
        const float r0 = __fdiv_rn((float)i0, 255.f), r1 = __fdiv_rn((float)i1, 255.f);
        const double s = (double)__fsub_rn(r1, r0);
        const double alpha = __ddiv_rn(1.0, s), beta = __dmul_rn(-(double)r0, alpha);
        s_identity = (fabs(alpha) == 1.0);
        s_ab[0] = (float)alpha;
        s_ab[1] = (float)beta;
    }
    __syncthreads();
    // pred[d]: raw difference d -> normalised pixel -> stretched pixel -> threshold
    const int pn = P.lut[(f + 1) * 256 + tid];
    int q = pn;
    if (!s_identity) {
        q = __float2int_rn(__fmaf_rn((float)pn, s_ab[0], s_ab[1]));
        q = min(255, max(0, q));
    }
    P.pred[f * 256 + tid] = ((double)q > P.p.threshold) ? 1 : 0;
}

__global__ void __launch_bounds__(256) k_bb_cols(const __grid_constant__ BBoxDev P) {
    __shared__ uint8_t pred[256];
    __shared__ int s_first, s_last, s_cnt;
    const int f = blockIdx.x, tid = threadIdx.x;
    pred[tid] = P.pred[f * 256 + tid];
    if (tid == 0) {
        s_first = 0x7fffffff;
        s_last = -1;
        s_cnt = 0;
    }
    __syncthreads();
    const uint8_t *F = P.frames + (int64_t)f * P.frame_bytes;
    const int c0 = max(0, P.p.zero_col_pre), c1 = min(P.p.side_w, P.p.zero_col_post);
    const int r0 = max(0, P.p.zero_row_pre), r1 = min(P.p.side_h, P.p.zero_row_post);
    const uint8_t *D = P.diff ? P.diff + (int64_t)f * P.p.side_w * P.p.side_h : nullptr;
    for (int x = tid; x < P.p.side_w; x += 256) {
        int sum = 0;
        if (D && x >= c0 && x < c1) {
            // consecutive threads read consecutive bytes of a row; eight rows in flight per thread
            for (int r = r0; r < r1; r += 8) {
                int d[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) d[q] = (r + q < r1) ? (int)__ldg(D + (int64_t)(r + q) * P.p.side_w + x) : -1;
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if (d[q] >= 0) sum += pred[d[q]];
            }
        } else if (x >= c0 && x < c1) {
            // rows in groups of 8 with the two dependent gathers (calibration index -> frame / background bytes) issued
            // back to back: the column sum is latency-bound otherwise
            const int xs = P.flip ? (P.n_cols - 1 - (P.p.side_x + x)) : (P.p.side_x + x);
            for (int r = r0; r < r1; r += 8) {
                int idx[8], d[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) idx[q] = (r + q < r1) ? __ldg(P.calib + (int64_t)(P.p.side_y + r + q) * P.n_cols + xs) : -1;
#pragma unroll
                for (int q = 0; q < 8; ++q) d[q] = idx[q] >= 0 ? (int)__ldg(F + idx[q]) - (int)__ldg(P.bkg + idx[q]) : -1000;
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if (d[q] > -1000) sum += pred[d[q] < 0 ? 0 : d[q]];
            }
        }
        if (P.sums) P.sums[(int64_t)f * P.p.side_w + x] = sum;
        if (sum >= P.p.min_count) {  // firstLastOverT: p[i] >= th
            atomicMin(&s_first, x);
            atomicMax(&s_last, x);
            atomicAdd(&s_cnt, 1);
        }
    }
    __syncthreads();
    if (tid == 0) {
        int first = -1, last = -1;
        if (s_cnt > 0) {
            first = s_first;
            last = s_cnt >= 2 ? s_last : 0;  // with one qualifying column the reference leaves slot 1 at its initial 0
        }
        P.lims[f * 2 + 0] = first;
        P.lims[f * 2 + 1] = last;
        P.bb_x[f] = fmin((double)(P.p.side_w - 1), __dmul_rn((double)last, P.p.width_margin));
    }
}

}  // namespace

static BBoxDev bbox_dev(const LmBatch &b, const lm_bb_de_params &p, uint32_t *hist, uint8_t *pred, double *bb_x, int32_t *lims, int32_t *sums,
                        uint8_t *diff) {
    BBoxDev P{};
    P.frames = b.frames;
    P.frame_bytes = b.frame_bytes;
    P.bkg = b.bkg;
    P.calib = b.calib;
    P.n_cols = b.n_cols;
    P.flip = b.flip;
    P.B = b.B;
    P.p = p;
    P.lut = b.lut;
    P.hist = hist;
    P.pred = pred;
    P.calib_flip = b.calib_flip;
    P.bkg_warp = b.bkg_warp;
    P.run_mode = b.run_mode;
    P.diff = diff;
    P.bb_x = bb_x;
    P.lims = lims;
    P.sums = sums;
    return P;
}

// The front end LocoMouse_TM_DE and LocoMouse_TM share: per-frame normalisation LUT, side-view histogram, imadjust_default
// and the threshold, folded into pred[f][d] (d = raw difference).  p: the side view rectangle and the threshold are used.
int lm_launch_bbox_pred(const LmBatch &b, const lm_bb_de_params &p, uint32_t *hist, uint8_t *pred, cudaStream_t s, uint8_t *diff) {
    int launches = 0;
    if (cudaMemsetAsync(b.minmax, 0, (size_t)(b.B + 1) * 2 * sizeof(int32_t), s) != cudaSuccess) return -1;
    if (cudaMemsetAsync(hist, 0, (size_t)b.B * 256 * sizeof(uint32_t), s) != cudaSuccess) return -1;
    int nl = lm_launch_minmax(b, s);
    if (nl < 0) return -1;
    launches += nl;
    const BBoxDev P = bbox_dev(b, p, hist, pred, nullptr, nullptr, nullptr, diff);
    const int npx = p.side_w * p.side_h;
    int gx = (npx + 256 * 16 - 1) / (256 * 16);
    gx = gx < 1 ? 1 : (gx > 64 ? 64 : gx);
    if (P.diff && P.calib_flip && P.bkg_warp && P.run_mode) {
        // 16 pixels per item: a few items per thread amortise the CTA's histogram set-up and final 256 global atomics
        int g16 = (((p.side_w + 15) / 16) * p.side_h + 256 * 8 - 1) / (256 * 8);
        g16 = g16 < 1 ? 1 : (g16 > 32 ? 32 : g16);
        if (const char *e = getenv("LM_BB_GX")) g16 = atoi(e) > 0 ? atoi(e) : g16;
        k_bb_hist16<<<dim3(g16, b.B), 256, 0, s>>>(P);
    }
    else
        k_bb_hist<<<dim3(gx, b.B), 256, 0, s>>>(P);
    k_bb_pred<<<b.B, 256, 0, s>>>(P);
    launches += 2;
    return cudaGetLastError() == cudaSuccess ? launches : -1;
}

// b: frames / bkg / calib / minmax / lut / n_cols / flip / B filled in by the caller (imadjust must be 0)
int lm_launch_bbox_tm_de(const LmBatch &b, const lm_bb_de_params &p, uint32_t *hist, uint8_t *pred, double *bb_x, int32_t *lims,
                         int32_t *sums, cudaStream_t s, uint8_t *diff) {
    int launches = lm_launch_bbox_pred(b, p, hist, pred, s, diff);
    if (launches < 0) return -1;
    const BBoxDev P = bbox_dev(b, p, hist, pred, bb_x, lims, sums, diff);
    k_bb_cols<<<b.B, 256, 0, s>>>(P);
    launches += 1;
    return cudaGetLastError() == cudaSuccess ? launches : -1;
}
