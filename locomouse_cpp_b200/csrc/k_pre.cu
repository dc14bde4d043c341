// k_pre.cu — frame pre-processing: background subtraction, per-frame min/max, normalisation,
// calibration gather, flip, imadjust, and the bounding-box crop of both views.
//
// Replaces LocoMouse::readFrame (LocoMouse_class.cpp:1273-1333: subtract 1304, normalize 1310,
// correctImage 1337-1406, flip 1323), LocoMouse_TM::readFrame's imadjust (LocoMouse_TM.cpp:243-249,
// LUT at LocoMouse_class.cpp:3223-3241), cropBoundingBox (1408-1478) and storePreviousImage (1508):
// nothing but the crop windows the detectors read is ever materialised, and the "previous image"
// is simply the previous raw frame, re-derived on the fly by the pairing kernel.
//
//  k_minmax : the only pass over whole raw frames (HBM bound): 16-byte loads of F and BKG,
//             per-byte saturating subtract with SIMD-in-word intrinsics, warp + atomic reduction.
//  k_lut    : per frame 256-entry LUT = imadjust ∘ saturate_u8(rint(fma(d, a, b))) with
//             a = float(255 * (1/(max-min))), b = float(-min * scale) (cv::normalize semantics).
//  k_prep   : per frame and view, window = crop + template halo; window pixel (r,c) in calibrated
//             image coordinates -> raw index through the calibration map (with the flip folded in) ->
//             lut[sat(F - BKG)]; zero outside the image (the reference's zero padded I_PAD).
#include "lm_internal.h"

namespace {

__device__ __forceinline__ const uint8_t *frame_ptr(const LmBatch &b, int i) {  // i in [-1, B)
    return i < 0 ? b.prev : b.frames + (int64_t)i * b.frame_bytes;
}

// ---- k_minmax ------------------------------------------------------------------------------------
// minmax[slot] = (255 - min, max) of d = max(F - BKG, 0), so that both reduce with atomicMax from a zero-initialised
// buffer.  The only pass over whole raw frames, hence HBM-bound.  Because max(., 0) is monotone, min d = max(min(F - BKG), 0)
// and max d = max(max(F - BKG), 0): the kernel tracks the SIGNED difference and clamps once per frame.
// A CTA owns a 16 kB pixel range (MM_VEC 16-byte vectors per thread, lanes on consecutive vectors) and walks MM_GROUP
// consecutive frames with the negated background of that range held in registers as s16x2 lanes (even / odd bytes), so the
// L2-resident background costs 1/MM_GROUP of the frame traffic; all MM_VEC loads of a frame are in flight together
// (streaming loads: a frame is read once).  Per four pixels: two widening ops (LOP3 + PRMT) and four fused add-min / add-max
// (VIADDMNMX.S16x2; the byte-SIMD intrinsics __vsubus4 / __vminu4 are emulated with dozens of instructions on this
// architecture and had made the pass ALU-bound).  Per-frame partials go warp (REDUX) -> shared memory, one barrier per CTA.
constexpr int MM_GROUP = 8;
constexpr int MM_VEC = 4;
constexpr int MM_THREADS = 256;

struct NegBkg {
    uint32_t e[4], o[4];
};
__device__ __forceinline__ NegBkg mm_neg(const uint4 &k) {
    NegBkg r;
    const uint32_t w[4] = {k.x, k.y, k.z, k.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        r.e[q] = __vneg2(w[q] & 0x00ff00ffu);
        r.o[q] = __vneg2(__byte_perm(w[q], 0u, 0x4341));
    }
    return r;
}
// one 32-bit word = four pixels: mn = min(mn, f - k), mx = max(mx, f - k) per s16 lane
__device__ __forceinline__ void mm_word(uint32_t &mn, uint32_t &mx, uint32_t f, uint32_t nke, uint32_t nko) {
    const uint32_t fe = f & 0x00ff00ffu, fo = __byte_perm(f, 0u, 0x4341);  // bytes 0,2 / bytes 1,3 as 16-bit lanes
    mn = __viaddmin_s16x2(fe, nke, mn);
    mx = __viaddmax_s16x2(fe, nke, mx);
    mn = __viaddmin_s16x2(fo, nko, mn);
    mx = __viaddmax_s16x2(fo, nko, mx);
}
__device__ __forceinline__ void mm_acc(uint32_t &mn, uint32_t &mx, const uint4 &f, const NegBkg &k) {
    mm_word(mn, mx, f.x, k.e[0], k.o[0]);
    mm_word(mn, mx, f.y, k.e[1], k.o[1]);
    mm_word(mn, mx, f.z, k.e[2], k.o[2]);
    mm_word(mn, mx, f.w, k.e[3], k.o[3]);
}
// clamp the signed lane extrema at 0 and reduce over the warp
__device__ __forceinline__ void mm_warp_reduce(uint32_t mn, uint32_t mx, int &lo, int &hi) {
    lo = min((int)(short)(mn & 0xffffu), (int)(short)(mn >> 16));
    hi = max((int)(short)(mx & 0xffffu), (int)(short)(mx >> 16));
    lo = __reduce_min_sync(0xffffffffu, max(lo, 0));  // REDUX: one instruction per warp reduction
    hi = __reduce_max_sync(0xffffffffu, max(hi, 0));
}

// ALIGNED: background, first frame and frame_bytes are all multiples of 16 (every frame of the batch is then 16-byte
// aligned and has no tail): vector path without per-frame checks.  Otherwise: the same ranges byte by byte.
template <bool ALIGNED>
__global__ void __launch_bounds__(MM_THREADS, 3) k_minmax(const __grid_constant__ LmBatch b, int slot0, int nslots) {
    __shared__ int slo[MM_GROUP][MM_THREADS / 32], shi[MM_GROUP][MM_THREADS / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t n = b.frame_bytes;
    const uint8_t *K = b.bkg;
    const int g0 = blockIdx.y * MM_GROUP;
    const int ng = min(MM_GROUP, nslots - g0);
    const int64_t vbase = (int64_t)blockIdx.x * (MM_THREADS * MM_VEC) + threadIdx.x;  // this thread's vectors: vbase + q * MM_THREADS
    if (ALIGNED) {
        const int64_t nvec = n >> 4;
        const uint4 *K4 = reinterpret_cast<const uint4 *>(K);
        NegBkg k[MM_VEC];
        bool ok[MM_VEC];
#pragma unroll
        for (int q = 0; q < MM_VEC; ++q) {
            ok[q] = vbase + q * MM_THREADS < nvec;
            // a vector past the end reads as F = K = 0: difference 0 would disturb the minimum, so it is skipped below
            k[q] = mm_neg(ok[q] ? __ldg(K4 + vbase + q * MM_THREADS) : make_uint4(0, 0, 0, 0));
        }
        for (int g = 0; g < ng; ++g) {
            const int slot = slot0 + g0 + g;  // slot 0 = halo frame (-1)
            const uint8_t *F = frame_ptr(b, slot - 1);
            uint32_t mn = 0x7fff7fffu, mx = 0x80008000u;  // s16x2 lanes
            if (F) {
                const uint4 *F4 = reinterpret_cast<const uint4 *>(F) + vbase;
                uint4 f[MM_VEC];
#pragma unroll
                for (int q = 0; q < MM_VEC; ++q)
                    if (ok[q]) f[q] = __ldcs(F4 + q * MM_THREADS);  // streamed once
#pragma unroll
                for (int q = 0; q < MM_VEC; ++q)
                    if (ok[q]) mm_acc(mn, mx, f[q], k[q]);
            }
            int lo, hi;
            mm_warp_reduce(mn, mx, lo, hi);
            if (lane == 0) {
                slo[g][w] = lo;
                shi[g][w] = hi;
            }
        }
    } else {
        const int64_t t0 = (int64_t)blockIdx.x * (MM_THREADS * MM_VEC * 16);
        for (int g = 0; g < ng; ++g) {
            const uint8_t *F = frame_ptr(b, slot0 + g0 + g - 1);
            int lo = 0x7fff, hi = -0x8000;
            if (F)
                for (int64_t t = t0 + threadIdx.x; t < min(n, t0 + MM_THREADS * MM_VEC * 16); t += MM_THREADS) {
                    const int d = (int)F[t] - (int)K[t];
                    lo = min(lo, d);
                    hi = max(hi, d);
                }
            lo = __reduce_min_sync(0xffffffffu, max(lo, 0));
            hi = __reduce_max_sync(0xffffffffu, max(hi, 0));
            if (lane == 0) {
                slo[g][w] = lo;
                shi[g][w] = hi;
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < ng) {
        const int g = threadIdx.x, slot = slot0 + g0 + g;
        if (frame_ptr(b, slot - 1)) {
            int lo = slo[g][0], hi = shi[g][0];
#pragma unroll
            for (int q = 1; q < MM_THREADS / 32; ++q) {
                lo = min(lo, slo[g][q]);
                hi = max(hi, shi[g][q]);
            }
            // a CTA whose range holds no pixel of the frame contributes (0x7fff -> clamped, -0x8000 -> 0): lo > 255 is skipped
            if (lo <= 255) atomicMax(&b.minmax[slot * 2 + 0], 255 - lo);
            atomicMax(&b.minmax[slot * 2 + 1], hi);
        }
    }
}

// ---- k_lut ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lut(const __grid_constant__ LmBatch b, int slot0) {
    const int slot = slot0 + blockIdx.x;
    const int v = threadIdx.x;
    const int smin = 255 - b.minmax[slot * 2 + 0], smax = b.minmax[slot * 2 + 1];
    // cv::normalize(NORM_MINMAX, 0..255) then Mat::convertTo(CV_8U, scale, shift):
    const double range = (double)smax - (double)smin;
    const double scale = __dmul_rn(255.0, range > 2.2204460492503131e-16 ? __ddiv_rn(1.0, range) : 0.0);
    const double shift = __dsub_rn(0.0, __dmul_rn((double)smin, scale));
    const float a = __double2float_rn(scale), sh = __double2float_rn(shift);
    int q = __float2int_rn(__fmaf_rn((float)v, a, sh));  // cvRound: half to even
    q = min(255, max(0, q));
    if (b.imadjust) {
        // imadjust(I, I, 0, 0.6, 0, 1): round() is half away from zero (values are non-negative)
        const double high_in = __dmul_rn(0.6, 255.0);
        const double range_div = __ddiv_rn(255.0, high_in);
        double t;
        if ((double)q <= 0.0)
            t = 0.0;
        else if ((double)q >= high_in)
            t = 255.0;
        else
            t = __dmul_rn((double)q, range_div);
        q = (int)round(t);
        q = min(255, max(0, q));
    }
    b.lut[slot * 256 + v] = (uint8_t)q;
}

// ---- k_prep --------------------------------------------------------------------------------------
// Per video, once (k_fold_calib): the calibration map with the optional mirror folded in, calib_flip[r][c] =
// calib[r][flip ? n_cols - 1 - c : c]; the background seen through it, bkg_warp[r][c] = bkg[calib_flip[r][c]]; and run flags:
// real calibration maps are piecewise runs of consecutive raw bytes, run_mode[r][c] says whether the 4 / 16 pixels that start
// at column c come from 4 / 16 consecutive raw bytes (ascending, or descending for a mirrored map).
// k_prep: one CTA = PREP_ROWS window rows of one (frame, view); a thread produces 16 window pixels (one 16-byte store).
//   tier 1  the 16 pixels are one run: one map load, five aligned frame words + funnel shifts, per-byte saturating
//           subtract of the background words, 16 table look-ups;
//   tier 2  per 4-pixel word: a run of 4 (two aligned frame words) or four separate gathers;
//   tier 3  words that cross the image border: per-pixel predicates.
constexpr int PREP_ROWS = 32;
constexpr int PREP_THREADS = 256;

__global__ void __launch_bounds__(256) k_fold_calib(const int32_t *__restrict__ calib, const uint8_t *__restrict__ bkg, int n_rows, int n_cols,
                                                    int flip, int32_t *__restrict__ calib_flip, uint8_t *__restrict__ bkg_warp,
                                                    uint8_t *__restrict__ run_mode) {
    const int64_t n = (int64_t)n_rows * n_cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / n_cols), c = (int)(i - (int64_t)r * n_cols);
        const int32_t *row = calib + (int64_t)r * n_cols;
        auto at = [&](int cc) { return row[flip ? n_cols - 1 - cc : cc]; };
        const int32_t src = at(c);
        calib_flip[i] = src;
        bkg_warp[i] = bkg[src];
        // bit 0 / 1: pixels c .. c+3 come from raw bytes src, src+1, .. / src, src-1, ..; bit 2 / 3: the same for c .. c+15
        int up = 0, down = 0;
        for (int q = 1; q < 16 && c + q < n_cols; ++q) {
            const int32_t a = at(c + q);
            if (a == src + q && up == q - 1) up = q;
            if (a == src - q && down == q - 1) down = q;
            if (up < q && down < q) break;
        }
        run_mode[i] = (uint8_t)((up >= 3 ? 1 : 0) | (down >= 3 ? 2 : 0) | (up >= 15 ? 4 : 0) | (down >= 15 ? 8 : 0));
    }
}

// four bytes at an arbitrary address through two aligned words (the caller guarantees both words lie inside the buffer)
__device__ __forceinline__ uint32_t ldg_u32_unaligned(const uint8_t *p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
    return __funnelshift_r(__ldg(w), __ldg(w + 1), ((unsigned)a & 3u) * 8u);
}
__device__ __forceinline__ uint32_t prep_lut4(const uint8_t *lut, uint32_t d4) {
    return (uint32_t)lut[d4 & 0xffu] | ((uint32_t)lut[(d4 >> 8) & 0xffu] << 8) | ((uint32_t)lut[(d4 >> 16) & 0xffu] << 16) | ((uint32_t)lut[d4 >> 24] << 24);
}

__global__ void __launch_bounds__(PREP_THREADS) k_prep(const __grid_constant__ LmBatch b) {
    const int f = blockIdx.y, v = blockIdx.z;
    const LmView &V = b.view[v];
    const int r0 = blockIdx.x * PREP_ROWS;
    if (r0 >= V.win_h) return;
    __shared__ uint8_t lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = b.lut[(f + 1) * 256 + i];
    __syncthreads();
    const int r1 = min(V.win_h, r0 + PREP_ROWS);
    const uint8_t *__restrict__ F = b.frames + (int64_t)f * b.frame_bytes;
    const uint8_t *__restrict__ Kw = b.bkg_warp;   // 4-byte aligned, padded by >= 24 bytes
    const int32_t *__restrict__ C2 = b.calib_flip;
    const uint8_t *__restrict__ RM = b.run_mode;
    const int fbytes = (int)b.frame_bytes;
    const int x0 = (int)b.bb_x[f] - b.bb_w + 1 - V.halo_x;
    const int ypos = (int)(v == LM_BOTTOM ? b.bb_y_bottom[f] : b.bb_y_side[f]);
    const int y0 = ypos - V.box_h + 1 - V.halo_y;
    uint8_t *W = b.win[v] + (int64_t)f * V.win_stride;
    const int nseg = V.win_pitch >> 4, n_cols = b.n_cols, n_rows = b.n_rows;
    const int items = (r1 - r0) * nseg;
    for (int it = threadIdx.x; it < items; it += PREP_THREADS) {
        const int rr = it / nseg, sg = it - rr * nseg;
        const int r = r0 + rr, c16 = sg << 4, xx0 = x0 + c16, yy = y0 + r;
        uint32_t o[4] = {0u, 0u, 0u, 0u};
        if (yy >= 0 && yy < n_rows && c16 < V.win_w && xx0 + 16 > 0 && xx0 < n_cols) {
            const int base = yy * n_cols + xx0;
            bool done = false;
            if (xx0 >= 0 && xx0 + 16 <= n_cols) {
                const int mode = __ldg(RM + base);
                if (mode & 12) {   // tier 1: one run of 16 raw bytes
                    const int i0 = __ldg(C2 + base);
                    const int lo_i = (mode & 4) ? i0 : i0 - 15;
                    if (lo_i >= 4 && lo_i + 24 <= fbytes) {   // the aligned words read lie inside this frame's bytes
                        const uintptr_t a = reinterpret_cast<uintptr_t>(F) + (uintptr_t)(unsigned)lo_i;
                        const uint32_t *fp = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
                        const unsigned sh = ((unsigned)a & 3u) * 8u;
                        const uint32_t f0 = __ldg(fp), f1 = __ldg(fp + 1), f2 = __ldg(fp + 2), f3 = __ldg(fp + 3), f4 = __ldg(fp + 4);
                        uint32_t fw[4] = {__funnelshift_r(f0, f1, sh), __funnelshift_r(f1, f2, sh), __funnelshift_r(f2, f3, sh), __funnelshift_r(f3, f4, sh)};
                        if (!(mode & 4)) {   // descending run: pixel q is raw byte lo_i + 15 - q
                            const uint32_t t0 = __byte_perm(fw[3], 0u, 0x0123), t1 = __byte_perm(fw[2], 0u, 0x0123);
                            const uint32_t t2 = __byte_perm(fw[1], 0u, 0x0123), t3 = __byte_perm(fw[0], 0u, 0x0123);
                            fw[0] = t0; fw[1] = t1; fw[2] = t2; fw[3] = t3;
                        }
                        const uint32_t *kp = reinterpret_cast<const uint32_t *>(Kw + (base & ~3));
                        const unsigned ks = (unsigned)(base & 3) * 8u;
                        const uint32_t k0 = __ldg(kp), k1 = __ldg(kp + 1), k2 = __ldg(kp + 2), k3 = __ldg(kp + 3), k4 = __ldg(kp + 4);
                        o[0] = prep_lut4(lut, __vsubus4(fw[0], __funnelshift_r(k0, k1, ks)));   // per-byte max(F - BKG, 0)
                        o[1] = prep_lut4(lut, __vsubus4(fw[1], __funnelshift_r(k1, k2, ks)));
                        o[2] = prep_lut4(lut, __vsubus4(fw[2], __funnelshift_r(k2, k3, ks)));
                        o[3] = prep_lut4(lut, __vsubus4(fw[3], __funnelshift_r(k3, k4, ks)));
                        done = true;
                    }
                }
            }
            if (!done) {
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const int c4 = c16 + 4 * w, xw = xx0 + 4 * w, bw = base + 4 * w;
                    if (c4 >= V.win_w) break;
                    if (xw >= 0 && xw + 4 <= n_cols) {   // tier 2: the word lies inside the image
                        const int32_t *cp = C2 + bw;
                        const int i0 = __ldg(cp);
                        const int mode = __ldg(RM + bw) & 3;
                        const int lo_i = mode == 2 ? i0 - 3 : i0;
                        uint32_t f4;
                        if (mode != 0 && lo_i >= 4 && lo_i + 8 <= fbytes) {
                            f4 = ldg_u32_unaligned(F + lo_i);
                            if (mode == 2) f4 = __byte_perm(f4, 0u, 0x0123);
                        } else {
                            const int i1 = __ldg(cp + 1), i2 = __ldg(cp + 2), i3 = __ldg(cp + 3);
                            f4 = (uint32_t)__ldg(F + i0) | ((uint32_t)__ldg(F + i1) << 8) | ((uint32_t)__ldg(F + i2) << 16) | ((uint32_t)__ldg(F + i3) << 24);
                        }
                        o[w] = prep_lut4(lut, __vsubus4(f4, ldg_u32_unaligned(Kw + bw)));
                    } else {   // tier 3: image border
                        uint32_t out = 0;
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            if (xw + q >= 0 && xw + q < n_cols) {
                                const int d = max((int)__ldg(F + __ldg(C2 + bw + q)) - (int)__ldg(Kw + bw + q), 0);
                                out |= (uint32_t)lut[d] << (8 * q);
                            }
                        o[w] = out;
                    }
                }
            }
            // pixels right of the window (the pitch rounds the row up to 16 bytes) stay zero
            const int valid = V.win_w - c16;
            if (valid < 16) {
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const int vb = valid - 4 * w;
                    if (vb <= 0) o[w] = 0u;
                    else if (vb < 4) o[w] &= (1u << (8 * vb)) - 1u;
                }
            }
        }
        *reinterpret_cast<uint4 *>(W + (int64_t)r * V.win_pitch + c16) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

}  // namespace

int lm_launch_minmax(const LmBatch &b, cudaStream_t s) {
    // slots 0..B (slot 0 = halo frame).  Enough CTAs per frame to keep HBM busy at any batch size.
    const int slot0 = b.prev ? 0 : 1;
    const int nslots = b.B + 1 - slot0;
    if (nslots <= 0) return 0;
    const int64_t per_cta = (int64_t)MM_THREADS * MM_VEC * 16;
    const int bx = (int)((b.frame_bytes + per_cta - 1) / per_cta);
    const dim3 grid(bx, (nslots + MM_GROUP - 1) / MM_GROUP);
    // every frame (and the halo frame) 16-byte aligned, no tail bytes: the vector path
    const bool aligned = (b.frame_bytes & 15) == 0 && (reinterpret_cast<uintptr_t>(b.frames) & 15) == 0 && (reinterpret_cast<uintptr_t>(b.bkg) & 15) == 0 &&
                         (b.prev == nullptr || (reinterpret_cast<uintptr_t>(b.prev) & 15) == 0);
    static LmDevOnce once;
    if (auto setup = once.first()) {
        lm_prefer_max_shared(k_minmax<true>);
        lm_prefer_max_shared(k_minmax<false>);
        lm_prefer_max_shared(k_lut);
    }
    if (aligned)
        k_minmax<true><<<grid, MM_THREADS, 0, s>>>(b, slot0, nslots);
    else
        k_minmax<false><<<grid, MM_THREADS, 0, s>>>(b, slot0, nslots);
    k_lut<<<nslots, 256, 0, s>>>(b, slot0);
    return 2;
}

int lm_launch_prep(const LmBatch &b, cudaStream_t s) {
    int maxh = 0;
    for (int v = 0; v < 2; ++v) maxh = b.view[v].win_h > maxh ? b.view[v].win_h : maxh;
    const int bx = (maxh + PREP_ROWS - 1) / PREP_ROWS;
    static LmDevOnce once;
    if (auto setup = once.first()) lm_prefer_max_shared(k_prep);
    k_prep<<<dim3(bx < 1 ? 1 : bx, b.B, 2), PREP_THREADS, 0, s>>>(b);
    return 1;
}

int lm_launch_fold_calib(const int32_t *calib, const uint8_t *bkg, int n_rows, int n_cols, int flip, int32_t *calib_flip, uint8_t *bkg_warp,
                         uint8_t *run_mode, cudaStream_t s) {
    k_fold_calib<<<lm_sm_count() * 4, 256, 0, s>>>(calib, bkg, n_rows, n_cols, flip, calib_flip, bkg_warp, run_mode);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}
