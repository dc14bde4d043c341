// k_bbox_base.cu — pass 1 of the base class on the device (SURVEY §8f-1): the per-frame part of
// LocoMouse::computeBoundingBox / computeMouseBox / largestBWAreaObject (LocoMouse_class.cpp:579-653, 921-997).
//
// Per frame the reference reads the image with the base-class readFrame (class.cpp:1273-1333), median-filters it with a
// k x k window (medianBlur on a copy padded by k/2 zeros that stays zero, see oracle/lm_oracle.cpp mouse_box_base),
// thresholds at 2.55 (-> 1 where the median is >= 3), keeps the largest connected component of the side view and of the
// bottom view, sums each along both axes (CV_32S, 255 per pixel) and takes the first / last entry that passes
// min_pixel_visible (firstLastOverT, class.hpp:411-442, which reads those integer sums through a float pointer).
// No 8-bit image is materialised:
//   k_minmax + k_lut (k_pre.cu)  per-frame normalisation LUT (imadjust(0, 0.6) off)
//   k_bbb_bin    bit image  b = [ normalise(sat(F - BKG)) >= 3 ]  of the whole calibrated image, gathered through the
//                calibration map (a warp = 32 consecutive pixels = one word, __ballot_sync)
//   k_bbb_major  median >= 3  <=>  at least (k*k+1)/2 of the zero-extended k x k window are set: window popcounts on the
//                bit image
//   k_bbb_cc     per (frame, view): the view's bits -> shared memory -> run-based largest component (cc_runs.cuh) ->
//                per-column / per-row counts -> the four sum vectors (stored per frame, lm_debug_fetch item 6) -> the four
//                (first, last) pairs
//   k_bbb_cc_slow  the same through the pixel union-find in global memory, for views with more runs than fit
// The six per-frame numbers and the whole-video post-processing (computeMouseBoxSize, vecmovingaverage) are host work.
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "cc_runs.cuh"
#include "lm_internal.h"

namespace {

struct BBaseDev {
    const uint8_t *frames;
    int64_t frame_bytes;
    const uint8_t *bkg;
    const int32_t *calib;
    const uint8_t *lut;      // [B + 1][256] normalisation LUT, slot f + 1
    int n_rows, n_cols, flip, B, conn;
    int wpr;                 // words per bit-image row
    uint32_t *bits, *major;  // [B][n_rows][wpr]
    lm_bb_base_params p;
    int32_t *lims;           // [B][4][2]: Row_side, Row_bottom, Col_side, Col_bottom
    int32_t *sums;           // [B][lm_bbox_base_sums(p)]: the same four vectors (255 per pixel; null: not kept)
    int *need_slow;          // [B][2]
    int runcap;
    // slow path scratch: SLOW_SLOTS x (3 ints per pixel of the larger view + its u8 map and mask)
    int32_t *cc;
    uint8_t *vmap, *vmask;
    int64_t cc_stride;
};

constexpr int BB_SLOW_SLOTS = 8;

__global__ void __launch_bounds__(256) k_bbb_bin(const __grid_constant__ BBaseDev P) {
    __shared__ uint8_t lut[256];
    const int f = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    lut[tid] = P.lut[(f + 1) * 256 + tid];
    __syncthreads();
    const uint8_t *F = P.frames + (int64_t)f * P.frame_bytes;
    uint32_t *out = P.bits + (int64_t)f * P.n_rows * P.wpr;
    const int nwords = P.n_rows * P.wpr;
    for (int w0 = (blockIdx.x * 8 + warp) * 4; w0 < nwords; w0 += gridDim.x * 32) {
        int idx[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {   // the calibration loads of four words first: the gather chain is latency-bound
            const int wi = w0 + q;
            idx[q] = -1;
            if (wi < nwords) {
                const int r = wi / P.wpr, x = (wi - r * P.wpr) * 32 + lane;
                if (x < P.n_cols) idx[q] = __ldg(P.calib + (int64_t)r * P.n_cols + (P.flip ? P.n_cols - 1 - x : x));
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            bool on = false;
            if (idx[q] >= 0) {
                const int d = (int)__ldg(F + idx[q]) - (int)__ldg(P.bkg + idx[q]);
                on = lut[d < 0 ? 0 : d] >= 3;  // threshold(I, I, 2.55, 1, THRESH_BINARY) on 8-bit data
            }
            const uint32_t word = __ballot_sync(0xffffffffu, on);
            if (lane == 0 && w0 + q < nwords) out[w0 + q] = word;
        }
    }
}

// One thread = one output word (32 pixels).  For each of the k window rows the three neighbouring input words give every
// pixel's k-bit horizontal window by a funnel shift; the counts add up over the rows.
__global__ void __launch_bounds__(128) k_bbb_major(const __grid_constant__ BBaseDev P) {
    const int f = blockIdx.y;
    const int k = P.p.median_filter_size, h = k >> 1, need = (k * k + 1) >> 1;
    const uint32_t kmask = k >= 32 ? 0xffffffffu : ((1u << k) - 1u);
    const uint32_t *in = P.bits + (int64_t)f * P.n_rows * P.wpr;
    uint32_t *out = P.major + (int64_t)f * P.n_rows * P.wpr;
    const int nwords = P.n_rows * P.wpr;
    for (int wi = blockIdx.x * blockDim.x + threadIdx.x; wi < nwords; wi += gridDim.x * blockDim.x) {
        const int r = wi / P.wpr, c = wi - r * P.wpr;
        int cnt[32];
#pragma unroll
        for (int q = 0; q < 32; ++q) cnt[q] = 0;
        for (int dy = -h; dy <= h; ++dy) {
            const int rr = r + dy;
            if (rr < 0 || rr >= P.n_rows) continue;  // zero padding
            const uint32_t *row = in + rr * P.wpr;
            const uint32_t lo = c > 0 ? __ldg(row + c - 1) : 0u, mid = __ldg(row + c), hi = c + 1 < P.wpr ? __ldg(row + c + 1) : 0u;
            if ((lo | mid | hi) == 0u) continue;
            // 96-bit strip: pixel q's window starts at strip bit 32 + q - h (h <= 15: two funnel shifts cover every case)
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                const int s = 32 + q - h;  // 17 .. 63
                const uint32_t wbits = s < 32 ? __funnelshift_r(lo, mid, s) : __funnelshift_r(mid, hi, s - 32);
                cnt[q] += __popc(wbits & kmask);
            }
        }
        uint32_t word = 0;
#pragma unroll
        for (int q = 0; q < 32; ++q) word |= (uint32_t)(cnt[q] >= need) << q;
        const int valid = P.n_cols - c * 32;
        if (valid < 32) word &= (valid <= 0) ? 0u : ((1u << valid) - 1u);
        out[wi] = word;
    }
}

// bits [x0, x0 + 32) of a bit row (zero beyond the row's words)
__device__ __forceinline__ uint32_t bits_at(const uint32_t *row, int wpr, int x0) {
    const int w = x0 >> 5, s = x0 & 31;
    const uint32_t lo = (w >= 0 && w < wpr) ? __ldg(row + w) : 0u, hi = (w + 1 >= 0 && w + 1 < wpr) ? __ldg(row + w + 1) : 0u;
    return __funnelshift_r(lo, hi, s);
}

// firstLastOverT on integer sums: the first index with sums[i] >= th goes to slot 0, every later one to slot 1 (so with a
// single qualifying index slot 1 stays 0); none -> (-1, -1).  as_float: compared as the float with the sum's bit pattern.
__device__ void first_last(const int *sums, int L, int scale, int th, int as_float, int32_t *out, int *s_acc) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        s_acc[0] = 0x7fffffff;
        s_acc[1] = -1;
        s_acc[2] = 0;
    }
    __syncthreads();
    const float thf = (float)th;
    for (int i = tid; i < L; i += TAIL_THREADS) {
        const int s = sums[i] * scale;
        const float v = as_float ? __int_as_float(s) : (float)s;
        if (v >= thf) {
            atomicMin(&s_acc[0], i);
            atomicMax(&s_acc[1], i);
            atomicAdd(&s_acc[2], 1);
        }
    }
    __syncthreads();
    if (tid == 0) {
        out[0] = s_acc[2] > 0 ? s_acc[0] : -1;
        out[1] = s_acc[2] > 0 ? (s_acc[2] >= 2 ? s_acc[1] : 0) : -1;
    }
    __syncthreads();
}

// the frame's Row_* (view v, L entries) or Col_* (rows entries) vector in P.sums
__device__ __forceinline__ int32_t *base_sums(const BBaseDev &P, int f, int v, bool col) {
    const lm_bb_base_params &p = P.p;
    int32_t *o = P.sums + (int64_t)f * (p.side_w + p.bottom_w + p.side_h + p.bottom_h);
    return col ? o + p.side_w + p.bottom_w + (v ? p.side_h : 0) : o + (v ? p.side_w : 0);
}

__global__ void __launch_bounds__(TAIL_THREADS) k_bbb_cc(const __grid_constant__ BBaseDev P) {
    extern __shared__ __align__(16) unsigned char raw[];
    const int f = blockIdx.x, v = blockIdx.y, tid = threadIdx.x;
    const int vx = v ? P.p.bottom_x : P.p.side_x, vy = v ? P.p.bottom_y : P.p.side_y;
    const int cols = v ? P.p.bottom_w : P.p.side_w, rows = v ? P.p.bottom_h : P.p.side_h;
    const int wpr = (cols + 31) >> 5;
    TailSmem S;
    unsigned char *p = raw;
    S.bits = reinterpret_cast<uint32_t *>(p); p += (size_t)rows * wpr * 4;
    S.obits = reinterpret_cast<uint32_t *>(p); p += (size_t)rows * wpr * 4;
    S.rowfirst = reinterpret_cast<int *>(p); p += (size_t)(rows + 1) * 4;
    const size_t rcap = (size_t)((P.runcap > 1 ? P.runcap : 1) + 63) & ~(size_t)63;
    S.parent = reinterpret_cast<int *>(p); p += rcap * 4;
    S.area = reinterpret_cast<int *>(p); p += rcap * 4;
    S.key = reinterpret_cast<int *>(p); p += rcap * 4;
    S.colany = nullptr;
    S.cnt = reinterpret_cast<int *>(p); p += (size_t)cols * 4;
    S.sum = reinterpret_cast<int *>(p); p += (size_t)cols * 4;
    S.rowcnt = reinterpret_cast<int *>(p); p += (size_t)rows * 4;
    S.rrow = reinterpret_cast<unsigned short *>(p); p += rcap * 2;
    S.rx0 = reinterpret_cast<unsigned short *>(p); p += rcap * 2;
    S.rx1 = reinterpret_cast<unsigned short *>(p); p += rcap * 2;
    __shared__ int scratch[40];
    __shared__ unsigned long long s_best;
    __shared__ int s_acc[3];
    const uint32_t *img = P.major + (int64_t)f * P.n_rows * P.wpr;
    for (int wi = tid; wi < rows * wpr; wi += TAIL_THREADS) {
        const int r = wi / wpr, c = wi - r * wpr;
        uint32_t w = bits_at(img + (int64_t)(vy + r) * P.wpr, P.wpr, vx + c * 32);
        const int valid = cols - c * 32;
        if (valid < 32) w &= (valid <= 0) ? 0u : ((1u << valid) - 1u);
        S.bits[wi] = w;
    }
    if (tid == 0) P.need_slow[f * 2 + v] = 0;
    __syncthreads();
    if (!largest_region_runs(S, rows, cols, wpr, P.conn, false, scratch, &s_best, P.runcap)) {
        if (tid == 0) P.need_slow[f * 2 + v] = 1;
        return;
    }
    int32_t *lim = P.lims + (int64_t)f * 8;
    // Row_* = per-column sums (scanned over min(N_COLS, view width) entries), Col_* = per-row sums; 255 per pixel
    if (P.sums) {
        int32_t *rs = base_sums(P, f, v, false), *cs = base_sums(P, f, v, true);
        for (int i = tid; i < min(P.n_cols, cols); i += TAIL_THREADS) rs[i] = S.cnt[i] * 255;
        for (int i = tid; i < rows; i += TAIL_THREADS) cs[i] = S.rowcnt[i] * 255;
    }
    first_last(S.cnt, min(P.n_cols, cols), 255, P.p.min_pixel_visible, P.p.sums_as_float, lim + (v ? 2 : 0), s_acc);
    first_last(S.rowcnt, rows, 255, P.p.min_pixel_visible, P.p.sums_as_float, lim + (v ? 6 : 4), s_acc);
}

// Views whose maps have more runs than the shared-memory path holds: expand the view to a u8 map, label its pixels with
// the global-memory union-find, count the winner's pixels per column / row.  BB_SLOW_SLOTS CTAs share the flagged views.
__global__ void __launch_bounds__(SLOW_THREADS) k_bbb_cc_slow(const __grid_constant__ BBaseDev P) {
    extern __shared__ int sm[];
    __shared__ unsigned long long s_best;
    __shared__ int s_acc[3];
    const int slot = blockIdx.x, tid = threadIdx.x;
    int *L = P.cc + (int64_t)slot * 3 * P.cc_stride, *area = L + P.cc_stride, *key = area + P.cc_stride;
    uint8_t *vmap = P.vmap + (int64_t)slot * P.cc_stride, *vmask = P.vmask + (int64_t)slot * P.cc_stride;
    int seen = 0;
    for (int u = 0; u < P.B * 2; ++u) {
        if (!P.need_slow[u]) continue;
        if ((seen++ % BB_SLOW_SLOTS) != slot) continue;
        const int f = u >> 1, v = u & 1;
        const int vx = v ? P.p.bottom_x : P.p.side_x, vy = v ? P.p.bottom_y : P.p.side_y;
        const int cols = v ? P.p.bottom_w : P.p.side_w, rows = v ? P.p.bottom_h : P.p.side_h;
        const uint32_t *img = P.major + (int64_t)f * P.n_rows * P.wpr;
        for (int i = tid; i < rows * cols; i += SLOW_THREADS) {
            const int r = i / cols, x = vx + (i - r * cols);
            vmap[i] = (img[(int64_t)(vy + r) * P.wpr + (x >> 5)] >> (x & 31)) & 1u;
        }
        int *colcnt = sm, *colsum = sm + cols, *rowcnt = sm + 2 * cols;
        for (int r = tid; r < rows; r += SLOW_THREADS) rowcnt[r] = 0;
        __syncthreads();
        cc_largest(vmap, nullptr, rows, cols, cols, P.conn, L, area, key, vmask, colcnt, colsum, nullptr, &s_best);
        for (int i = tid; i < rows * cols; i += SLOW_THREADS)
            if (vmask[i]) atomicAdd(&rowcnt[i / cols], 1);
        __syncthreads();
        int32_t *lim = P.lims + (int64_t)f * 8;
        for (int pass = 0; pass < 2; ++pass) {
            const int *sums = pass ? rowcnt : colcnt;
            const int Lc = pass ? rows : min(P.n_cols, cols);
            if (P.sums) {
                int32_t *out = base_sums(P, f, v, pass != 0);
                for (int i = tid; i < Lc; i += SLOW_THREADS) out[i] = sums[i] * 255;
            }
            __syncthreads();
            if (tid == 0) {
                s_acc[0] = 0x7fffffff;
                s_acc[1] = -1;
                s_acc[2] = 0;
            }
            __syncthreads();
            const float thf = (float)P.p.min_pixel_visible;
            for (int i = tid; i < Lc; i += SLOW_THREADS) {
                const int s = sums[i] * 255;
                const float val = P.p.sums_as_float ? __int_as_float(s) : (float)s;
                if (val >= thf) {
                    atomicMin(&s_acc[0], i);
                    atomicMax(&s_acc[1], i);
                    atomicAdd(&s_acc[2], 1);
                }
            }
            __syncthreads();
            if (tid == 0) {
                int32_t *o = lim + (pass ? (v ? 6 : 4) : (v ? 2 : 0));
                o[0] = s_acc[2] > 0 ? s_acc[0] : -1;
                o[1] = s_acc[2] > 0 ? (s_acc[2] >= 2 ? s_acc[1] : 0) : -1;
            }
        }
        __syncthreads();
    }
}

size_t bbb_cc_smem(int rows, int cols, int runcap) {
    const size_t rcap = (size_t)((runcap > 1 ? runcap : 1) + 63) & ~(size_t)63;
    const int wpr = (cols + 31) >> 5;
    const size_t s = (size_t)rows * wpr * 4 * 2 + (size_t)(rows + 1) * 4 + rcap * 4 * 3 + (size_t)cols * 4 * 2 + (size_t)rows * 4 + rcap * 2 * 3;
    return (s + 15) & ~(size_t)15;
}

}  // namespace

size_t lm_bbox_base_bits_bytes(int n_rows, int n_cols, int B) { return (size_t)B * n_rows * ((n_cols + 31) / 32) * sizeof(uint32_t); }
size_t lm_bbox_base_slow_ints(const lm_bb_base_params &p) {
    return (size_t)std::max((int64_t)p.side_w * p.side_h, (int64_t)p.bottom_w * p.bottom_h);
}

// b: frames / bkg / calib / minmax / lut / n_rows / n_cols / flip / conn / B filled in by the caller (imadjust must be 0).
// bits / major: lm_bbox_base_bits_bytes each; cc: BB_SLOW_SLOTS * 3 * lm_bbox_base_slow_ints ints; vmap / vmask: BB_SLOW_SLOTS *
// lm_bbox_base_slow_ints bytes each; need_slow: [B][2]; lims: [B][4][2].
int lm_launch_bbox_base(const LmBatch &b, const lm_bb_base_params &p, uint32_t *bits, uint32_t *major, int32_t *cc, uint8_t *vmap, uint8_t *vmask,
                        int *need_slow, int32_t *lims, int32_t *sums, cudaStream_t s) {
    int launches = 0;
    if (cudaMemsetAsync(b.minmax, 0, (size_t)(b.B + 1) * 2 * sizeof(int32_t), s) != cudaSuccess) return -1;
    int nl = lm_launch_minmax(b, s);
    if (nl < 0) return -1;
    launches += nl;
    BBaseDev P{};
    P.frames = b.frames;
    P.frame_bytes = b.frame_bytes;
    P.bkg = b.bkg;
    P.calib = b.calib;
    P.lut = b.lut;
    P.n_rows = b.n_rows;
    P.n_cols = b.n_cols;
    P.flip = b.flip;
    P.B = b.B;
    P.conn = b.conn;
    P.wpr = (b.n_cols + 31) / 32;
    P.bits = bits;
    P.major = major;
    P.p = p;
    P.lims = lims;
    P.sums = sums;
    P.need_slow = need_slow;
    P.cc = cc;
    P.vmap = vmap;
    P.vmask = vmask;
    P.cc_stride = (int64_t)lm_bbox_base_slow_ints(p);
    const int nwords = b.n_rows * P.wpr;
    int dev_smem = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    // dynamic shared memory each kernel may ask for = the opt-in limit minus its own static shared memory
    cudaFuncAttributes fa_cc{}, fa_slow{};
    if (cudaFuncGetAttributes(&fa_cc, k_bbb_cc) != cudaSuccess || cudaFuncGetAttributes(&fa_slow, k_bbb_cc_slow) != cudaSuccess) return -1;
    const int dyn_cc = dev_smem - (int)fa_cc.sharedSizeBytes, dyn_slow = dev_smem - (int)fa_slow.sharedSizeBytes;
    // the largest run capacity (<= RUNCAP, 16-bit run ids) that fits beside the larger view's bit images
    const int rmax = std::max(p.side_h, p.bottom_h), cmax = std::max(p.side_w, p.bottom_w);
    int runcap = RUNCAP;
    while (runcap > 0 && bbb_cc_smem(rmax, cmax, runcap) > (size_t)std::max(dyn_cc, 0)) runcap -= 256;
    if (const char *e = getenv("LM_BBOX_RUNCAP")) runcap = std::max(0, std::min(runcap, atoi(e)));
    P.runcap = std::max(runcap, 0);
    static LmDevOnce once;
    if (auto setup = once.first()) {
        if (cudaFuncSetAttribute(k_bbb_cc, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_cc) != cudaSuccess) return -1;
        if (cudaFuncSetAttribute(k_bbb_cc_slow, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_slow) != cudaSuccess) return -1;
    }
    int gx = (nwords + 32 * 8 - 1) / (32 * 8);
    gx = gx < 1 ? 1 : (gx > 48 ? 48 : gx);
    k_bbb_bin<<<dim3(gx, b.B), 256, 0, s>>>(P);
    int gm = (nwords + 127) / 128;
    gm = gm < 1 ? 1 : (gm > 1024 ? 1024 : gm);
    k_bbb_major<<<dim3(gm, b.B), 128, 0, s>>>(P);
    const size_t smem = bbb_cc_smem(rmax, cmax, P.runcap);
    if (smem <= (size_t)std::max(dyn_cc, 0) && P.runcap > 0) {
        k_bbb_cc<<<dim3(b.B, 2), TAIL_THREADS, smem, s>>>(P);
    } else {  // views too large for the shared-memory labelling: everything takes the global-memory path
        int *ns = need_slow;
        std::vector<int> ones((size_t)b.B * 2, 1);
        if (cudaMemcpyAsync(ns, ones.data(), ones.size() * sizeof(int), cudaMemcpyHostToDevice, s) != cudaSuccess) return -1;
        if (cudaStreamSynchronize(s) != cudaSuccess) return -1;  // `ones` goes out of scope
    }
    const size_t slow_smem = (size_t)(2 * cmax + rmax) * sizeof(int);
    if (slow_smem > (size_t)std::max(dyn_slow, 0)) return -1;
    k_bbb_cc_slow<<<BB_SLOW_SLOTS, SLOW_THREADS, slow_smem, s>>>(P);
    launches += 4;
    return cudaGetLastError() == cudaSuccess ? launches : -1;
}
