// k_bbox_tm.cu — pass 1 of LocoMouse_TM on the device (SURVEY §8f-1): the per-frame part of
// LocoMouse_TM::computeBoundingBox / computeMouseBox_DD / bwAreaOpen / imfill (LocoMouse_TM.cpp:115-269).
//
// Per frame the reference reads the image with the base-class readFrame, stretches the side view with imadjust_default,
// zeroes four bands, thresholds, removes connected components of fewer than MIN_PIXEL_COUNT pixels (bwAreaOpen), filters
// the 0 / 1 image with the DISK_FILTER matrix into an 8-bit image (rounded float sums, replicated border), fills every
// region that a flood fill from pixel (0, 0) cannot reach (imfill), sums the columns and takes the first / last column
// that passes min_pixel_visible (firstLastOverT, which reads the CV_32S sums through a float pointer).  Nothing but bit
// images is materialised:
//   k_minmax + k_lut (k_pre.cu), k_bb_hist + k_bb_pred (k_bbox.cu)   pred[d] = imadjust_default(normalise(d)) > threshold
//   k_bbtm_bin    bit image of the side view through the calibration map, bands zeroed (a warp = one 32-pixel word)
//   k_bbtm_open   per frame: run-based component labelling in shared memory, runs of components below the area limit cleared
//   k_bbtm_disk   a thread = one output word; words whose whole neighbourhood is empty are skipped; otherwise taps over set
//                 pixels are counted per distinct kernel weight (popcounts) and only sums within the rounding margin of 0.5
//                 replay OpenCV's float adds in row-major tap order
//   k_bbtm_fill   per frame: 4-connected labelling of the seed-valued pixels, the component of pixel (0, 0) = the flood
//                 fill; column sums via a difference array; first / last; bb_x
// Frames whose run count exceeds the shared-memory capacity set a flag and are redone by the same code with its run arrays
// in global memory (k_bbtm_open / k_bbtm_fill instantiated with GLOBAL = true, one CTA per flagged frame).
#include <algorithm>
#include <cstdlib>

#include "cc_runs.cuh"
#include "lm_internal.h"

namespace {

constexpr int TM_DISK_LEVELS = 8;   // distinct kernel weights the counting path of k_bbtm_disk handles

struct BBTmDev {
    const uint8_t *frames;
    int64_t frame_bytes;
    const uint8_t *bkg;
    const int32_t *calib;
    const uint8_t *pred;   // [B][256]
    int n_cols, flip, B, conn;
    int side_x, side_y, W, H, wpr;
    int zc0, zc1, zr0, zr1;  // surviving columns [zc0, zc1), rows [zr0, zr1)
    int min_pixel_count, min_pixel_visible, as_float;
    int K;
    const float *disk;       // device, [K][K]
    uint32_t *bits_a, *bits_b;  // [B][H][wpr]
    int *need_slow;          // [B][2]: open, fill
    int runcap;              // run capacity of the shared-memory path
    // global run arrays for the slow path: one slot of worst-case size per frame of the chunk
    int *g_parent, *g_area;
    unsigned short *g_rrow, *g_rx0, *g_rx1;
    int64_t g_stride;        // runs per slot
    double *bb_x;            // [B]
    int32_t *lims;           // [B][2]
};

__global__ void __launch_bounds__(256) k_bbtm_bin(const __grid_constant__ BBTmDev P) {
    __shared__ uint8_t pred[256];
    const int f = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pred[tid] = P.pred[f * 256 + tid];
    __syncthreads();
    const uint8_t *F = P.frames + (int64_t)f * P.frame_bytes;
    uint32_t *out = P.bits_a + (int64_t)f * P.H * P.wpr;
    const int nwords = P.H * P.wpr;
    for (int w0 = (blockIdx.x * 8 + warp) * 4; w0 < nwords; w0 += gridDim.x * 32) {
        int idx[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {   // the calibration loads of four words first: the gather chain is latency-bound
            const int wi = w0 + q;
            idx[q] = -1;
            if (wi < nwords) {
                const int r = wi / P.wpr, x = (wi - r * P.wpr) * 32 + lane;
                if (x >= P.zc0 && x < P.zc1 && r >= P.zr0 && r < P.zr1) {
                    const int xi = P.side_x + x;
                    idx[q] = __ldg(P.calib + (int64_t)(P.side_y + r) * P.n_cols + (P.flip ? P.n_cols - 1 - xi : xi));
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            bool on = false;
            if (idx[q] >= 0) {
                const int d = (int)__ldg(F + idx[q]) - (int)__ldg(P.bkg + idx[q]);
                on = pred[d < 0 ? 0 : d] != 0;
            }
            const uint32_t word = __ballot_sync(0xffffffffu, on);
            if (lane == 0 && w0 + q < nwords) out[w0 + q] = word;
        }
    }
}

// ---- run-based labelling ---------------------------------------------------------------------------------------------
struct RunArrays {
    unsigned short *rrow, *rx0, *rx1;
    int *parent, *area;
};

// Labels the runs of the bit image `bits` (rows x wpr words in shared memory, bits beyond `cols` zero): on return run i has
// row / x0 / x1, parent[i] = its root and area[root] = the component's pixel count.  rowfirst: [rows + 1] in shared memory.
// Returns the number of runs, or -1 when it exceeds cap (nothing written then).
__device__ int label_runs(const uint32_t *bits, int rows, int cols, int wpr, int conn, int *rowfirst, const RunArrays &R, int cap, int *scratch) {
    const int tid = threadIdx.x;
    const int nwords = rows * wpr;
    const int chunk = (nwords + TAIL_THREADS - 1) / TAIL_THREADS;
    const int w0 = tid * chunk, w1 = min(nwords, w0 + chunk);
    int mine = 0;
    for (int wi = w0; wi < w1; ++wi) {
        const int c = wi % wpr;
        const uint32_t b = bits[wi];
        const uint32_t carry = (c > 0) ? (bits[wi - 1] >> 31) : 0u;
        mine += __popc(b & ~((b << 1) | carry));
    }
    int total;
    int base = block_exscan(mine, scratch, &total);
    if (total > cap) return -1;
    for (int i = tid; i <= rows; i += TAIL_THREADS) rowfirst[i] = total;
    __syncthreads();
    for (int wi = w0; wi < w1; ++wi) {
        const int r = wi / wpr, c = wi - r * wpr;
        const uint32_t b = bits[wi];
        const uint32_t carry = (c > 0) ? (bits[wi - 1] >> 31) : 0u;
        uint32_t starts = b & ~((b << 1) | carry);
        while (starts) {
            const int bit = __ffs(starts) - 1;
            starts &= starts - 1;
            const int x0 = c * 32 + bit;
            int x1;
            {
                int cw = c;
                uint32_t inv = ~bits[wi] & (0xffffffffu << bit);
                while (inv == 0u && cw + 1 < wpr) {
                    ++cw;
                    inv = ~bits[r * wpr + cw];
                }
                x1 = (inv ? cw * 32 + __ffs(inv) - 1 : wpr * 32) - 1;
                if (x1 >= cols) x1 = cols - 1;
            }
            const int id = base++;
            R.rrow[id] = (unsigned short)r;
            R.rx0[id] = (unsigned short)x0;
            R.rx1[id] = (unsigned short)x1;
            R.parent[id] = id;
            R.area[id] = 0;
            atomicMin(&rowfirst[r], id);
        }
    }
    __syncthreads();
    if (tid == 0) {
        int nxt = total;
        for (int r = rows; r >= 0; --r) {
            if (rowfirst[r] > nxt) rowfirst[r] = nxt;
            nxt = rowfirst[r];
        }
    }
    __syncthreads();
    const int ext = (conn == 8) ? 1 : 0;
    for (int id = tid; id < total; id += TAIL_THREADS) {
        const int r = R.rrow[id];
        if (r == 0) continue;
        const int lo = (int)R.rx0[id] - ext, hi = (int)R.rx1[id] + ext;
        // the previous row's runs are x-sorted: binary search for the first one that ends at or after lo
        int a = rowfirst[r - 1], e = rowfirst[r];
        while (a < e) {
            const int mid = (a + e) >> 1;
            if ((int)R.rx1[mid] < lo) a = mid + 1;
            else e = mid;
        }
        for (int q = a; q < rowfirst[r]; ++q) {
            if ((int)R.rx0[q] > hi) break;
            uf_union_s(R.parent, id, q);
        }
    }
    __syncthreads();
    for (int id = tid; id < total; id += TAIL_THREADS) {
        const int root = uf_find_s(R.parent, id);
        R.parent[id] = root;
        atomicAdd(&R.area[root], (int)R.rx1[id] - (int)R.rx0[id] + 1);
    }
    __syncthreads();
    return total;
}

__device__ __forceinline__ RunArrays carve_runs(unsigned char *p, int cap) {
    RunArrays R;
    R.parent = reinterpret_cast<int *>(p); p += (size_t)cap * 4;
    R.area = reinterpret_cast<int *>(p); p += (size_t)cap * 4;
    R.rrow = reinterpret_cast<unsigned short *>(p); p += (size_t)cap * 2;
    R.rx0 = reinterpret_cast<unsigned short *>(p); p += (size_t)cap * 2;
    R.rx1 = reinterpret_cast<unsigned short *>(p);
    return R;
}
__device__ __forceinline__ RunArrays global_runs(const BBTmDev &P, int slot) {
    RunArrays R;
    const int64_t o = (int64_t)slot * P.g_stride;
    R.parent = P.g_parent + o;
    R.area = P.g_area + o;
    R.rrow = P.g_rrow + o;
    R.rx0 = P.g_rx0 + o;
    R.rx1 = P.g_rx1 + o;
    return R;
}

// clears / sets bits [x0, x1] of a bit row in shared memory
__device__ __forceinline__ void row_clear(uint32_t *row, int x0, int x1) {
    for (int cw = x0 >> 5; cw <= (x1 >> 5); ++cw) {
        const int a = max(x0, cw * 32) - cw * 32, e = min(x1, cw * 32 + 31) - cw * 32;
        const uint32_t m = (e == 31 ? 0xffffffffu : ((1u << (e + 1)) - 1u)) & (0xffffffffu << a);
        atomicAnd(&row[cw], ~m);
    }
}

// shared memory of k_bbtm_open / k_bbtm_fill: bits [H][wpr] | rowfirst [H + 1] | diff [W + 2] | run arrays (fast path)
__host__ __device__ inline size_t tm_smem_fixed(int H, int W, int wpr) { return (size_t)H * wpr * 4 + (size_t)(H + 1) * 4 + (size_t)(W + 2) * 4; }
size_t tm_smem(int H, int W, int wpr, int cap) { return ((tm_smem_fixed(H, W, wpr) + 15) & ~(size_t)15) + (size_t)cap * 14 + 16; }

// bwAreaOpen (LocoMouse_TM.cpp:158-187): bits_a -> bits_b with the components of fewer than min_pixel_count pixels removed
template <bool GLOBAL>
__global__ void __launch_bounds__(TAIL_THREADS) k_bbtm_open(const __grid_constant__ BBTmDev P) {
    extern __shared__ __align__(16) unsigned char raw[];
    __shared__ int scratch[40];
    uint32_t *bits = reinterpret_cast<uint32_t *>(raw);
    int *rowfirst = reinterpret_cast<int *>(bits + (size_t)P.H * P.wpr);
    const size_t fixed = (tm_smem_fixed(P.H, P.W, P.wpr) + 15) & ~(size_t)15;
    const RunArrays R = GLOBAL ? global_runs(P, blockIdx.x) : carve_runs(raw + fixed, P.runcap);
    const int cap = GLOBAL ? (int)P.g_stride : P.runcap;
    const int nwords = P.H * P.wpr, tid = threadIdx.x;
    for (int f = blockIdx.x; f < P.B; f += gridDim.x) {   // grid = B: one frame per CTA
        if (GLOBAL && !P.need_slow[f * 2 + 0]) continue;
        const uint32_t *in = P.bits_a + (int64_t)f * nwords;
        uint32_t *out = P.bits_b + (int64_t)f * nwords;
        for (int i = tid; i < nwords; i += TAIL_THREADS) bits[i] = in[i];
        __syncthreads();
        const int total = label_runs(bits, P.H, P.W, P.wpr, P.conn, rowfirst, R, cap, scratch);
        if (total < 0) {  // more runs than the shared-memory arrays hold: redone by the global-memory instance
            if (tid == 0) P.need_slow[f * 2 + 0] = 1;
            __syncthreads();
            continue;
        }
        for (int id = tid; id < total; id += TAIL_THREADS)
            if ((unsigned)R.area[R.parent[id]] < (unsigned)P.min_pixel_count) row_clear(bits + (int)R.rrow[id] * P.wpr, R.rx0[id], R.rx1[id]);
        __syncthreads();
        for (int i = tid; i < nwords; i += TAIL_THREADS) out[i] = bits[i];
        __syncthreads();
    }
}

// bit x of a bit row with the column clamped to [0, W - 1] (BORDER_REPLICATE)
__device__ __forceinline__ uint32_t bit_clamped(const uint32_t *row, int x, int W) {
    x = x < 0 ? 0 : (x >= W ? W - 1 : x);
    return (__ldg(row + (x >> 5)) >> (x & 31)) & 1u;
}

// filter2D(., CV_8UC1, DISK_FILTER, (-1,-1), 0, BORDER_REPLICATE) on the 0 / 1 image bits_b -> bits_a = [ result >= 1 ]
// (the host guarantees that no sum of taps rounds above 1).  A thread = one output word.  Words whose neighbourhood is empty
// are 0.  Otherwise each of the K window rows is fetched once as a 64-bit strip (columns 32c - an .. 32c - an + 63, edge
// pixels replicated) into shared memory; per pixel the taps over set pixels are COUNTED per distinct kernel weight
// (popcounts against per-row masks) and the sum formed in double: when it is farther from 0.5 than the worst-case rounding
// error of OpenCV's float accumulation, the result is certain; the few pixels inside that margin -- and kernels with more
// than TM_DISK_LEVELS distinct weights or more than 32 columns -- replay OpenCV's float adds in row-major tap order.
struct DiskLevels {
    int L;                      // 0: always the exact replay
    double val[TM_DISK_LEVELS];
    double margin;
};
constexpr int DISK_THREADS = 128;

__global__ void __launch_bounds__(DISK_THREADS) k_bbtm_disk(const __grid_constant__ BBTmDev P, const __grid_constant__ DiskLevels D,
                                                             const uint32_t *__restrict__ level_mask /* [L][K] */) {
    extern __shared__ __align__(16) unsigned char dsm[];
    const int K = P.K, an = K >> 1;
    float *kern = reinterpret_cast<float *>(dsm);                                         // [K][K]
    uint32_t *lmask = reinterpret_cast<uint32_t *>(kern + K * K);                         // [L][K]
    unsigned long long *wins = reinterpret_cast<unsigned long long *>(dsm + (((size_t)(K * K + TM_DISK_LEVELS * K) * 4 + 15) & ~(size_t)15));  // [K][DISK_THREADS]
    for (int i = threadIdx.x; i < K * K; i += DISK_THREADS) kern[i] = P.disk[i];
    for (int i = threadIdx.x; i < D.L * K; i += DISK_THREADS) lmask[i] = level_mask[i];
    __syncthreads();
    const bool counting = D.L > 0 && K <= 32;
    const int f = blockIdx.y, nwords = P.H * P.wpr;
    const uint32_t *in = P.bits_b + (int64_t)f * nwords;
    uint32_t *out = P.bits_a + (int64_t)f * nwords;
    for (int wi = blockIdx.x * DISK_THREADS + threadIdx.x; wi < nwords; wi += gridDim.x * DISK_THREADS) {
        const int r = wi / P.wpr, c = wi - r * P.wpr;
        const int ra = max(0, r - an), rb = min(P.H - 1, r + K - 1 - an);
        const int ca = max(0, (c * 32 - an) >> 5), cb = min(P.wpr - 1, (c * 32 + 31 + K - 1 - an) >> 5);
        uint32_t any = 0;
        for (int rr = ra; rr <= rb; ++rr)
            for (int cc = ca; cc <= cb; ++cc) any |= __ldg(in + rr * P.wpr + cc);
        uint32_t word = 0;
        if (any) {
            const int valid = min(32, P.W - c * 32);
            const int x_lo = c * 32 - an;   // column of strip bit 0
            if (counting) {
                const bool interior = x_lo >= 0 && x_lo + 63 < P.W;
                for (int j = 0; j < K; ++j) {
                    int rr = r + j - an;
                    rr = rr < 0 ? 0 : (rr >= P.H ? P.H - 1 : rr);
                    const uint32_t *row = in + rr * P.wpr;
                    unsigned long long w;
                    if (interior) {
                        const int w0 = x_lo >> 5, sh = x_lo & 31;
                        const uint32_t a0 = __ldg(row + w0), a1 = __ldg(row + w0 + 1), a2 = (w0 + 2 < P.wpr) ? __ldg(row + w0 + 2) : 0u;
                        w = (unsigned long long)__funnelshift_r(a0, a1, sh) | ((unsigned long long)__funnelshift_r(a1, a2, sh) << 32);
                    } else {
                        w = 0ull;
                        for (int t = 0; t < 32 + K - 1; ++t) w |= (unsigned long long)bit_clamped(row, x_lo + t, P.W) << t;
                    }
                    wins[j * DISK_THREADS + threadIdx.x] = w;
                }
            }
            for (int q = 0; q < valid; ++q) {
                bool decided = false;
                int v = 0;
                if (counting) {
                    double sd = 0.0;
                    for (int l = 0; l < D.L; ++l) {
                        int cnt = 0;
                        for (int j = 0; j < K; ++j) cnt += __popc((uint32_t)(wins[j * DISK_THREADS + threadIdx.x] >> q) & lmask[l * K + j]);
                        sd += D.val[l] * (double)cnt;
                    }
                    if (fabs(sd - 0.5) > D.margin) {
                        v = sd > 0.5 ? 1 : 0;
                        decided = true;
                    }
                }
                if (!decided) {   // OpenCV's float accumulation, tap by tap in row-major order
                    const int x = c * 32 + q;
                    float s = 0.f;
                    for (int j = 0; j < K; ++j) {
                        int rr = r + j - an;
                        rr = rr < 0 ? 0 : (rr >= P.H ? P.H - 1 : rr);
                        const uint32_t *row = in + rr * P.wpr;
                        for (int i = 0; i < K; ++i)
                            if (bit_clamped(row, x + i - an, P.W)) s = __fadd_rn(s, kern[j * K + i]);  // + k * 1; a 0 pixel adds k * 0 = 0
                    }
                    v = __float2int_rn(s) >= 1 ? 1 : 0;   // saturate_cast<uchar>(float): round half to even
                }
                word |= (uint32_t)v << q;
            }
        }
        out[wi] = word;
    }
}

// imfill (LocoMouse_TM.cpp:252-269) + reduce + firstLastOverT: bits_a = the filtered 0 / 1 image
template <bool GLOBAL>
__global__ void __launch_bounds__(TAIL_THREADS) k_bbtm_fill(const __grid_constant__ BBTmDev P) {
    extern __shared__ __align__(16) unsigned char raw[];
    __shared__ int scratch[40];
    __shared__ int s_first, s_last, s_cnt;
    uint32_t *bits = reinterpret_cast<uint32_t *>(raw);
    int *rowfirst = reinterpret_cast<int *>(bits + (size_t)P.H * P.wpr);
    int *diff = rowfirst + P.H + 1;  // [W + 2]
    const size_t fixed = (tm_smem_fixed(P.H, P.W, P.wpr) + 15) & ~(size_t)15;
    const RunArrays R = GLOBAL ? global_runs(P, blockIdx.x) : carve_runs(raw + fixed, P.runcap);
    const int cap = GLOBAL ? (int)P.g_stride : P.runcap;
    const int nwords = P.H * P.wpr, tid = threadIdx.x;
    for (int f = blockIdx.x; f < P.B; f += gridDim.x) {
        if (GLOBAL && !P.need_slow[f * 2 + 1]) continue;
        const uint32_t *in = P.bits_a + (int64_t)f * nwords;
        const uint32_t seed = in[0] & 1u;  // value of pixel (0, 0)
        // the pixels with the seed's value (bits beyond the last column stay 0)
        for (int i = tid; i < nwords; i += TAIL_THREADS) {
            const int c = i % P.wpr;
            const int valid = P.W - c * 32;
            const uint32_t vm = valid >= 32 ? 0xffffffffu : (valid <= 0 ? 0u : ((1u << valid) - 1u));
            bits[i] = (seed ? in[i] : ~in[i]) & vm;
        }
        for (int i = tid; i < P.W + 2; i += TAIL_THREADS) diff[i] = 0;
        if (tid == 0) {
            s_first = 0x7fffffff;
            s_last = -1;
            s_cnt = 0;
        }
        __syncthreads();
        const int total = label_runs(bits, P.H, P.W, P.wpr, 4, rowfirst, R, cap, scratch);  // floodFill: 4-connected
        if (total < 0) {
            if (tid == 0) P.need_slow[f * 2 + 1] = 1;
            __syncthreads();
            continue;
        }
        // run 0 starts at pixel (0, 0): its component is what the flood fill reaches
        const int seed_root = R.parent[0];
        for (int id = tid; id < total; id += TAIL_THREADS)
            if (R.parent[id] == seed_root) {
                atomicAdd(&diff[R.rx0[id]], 1);
                atomicAdd(&diff[(int)R.rx1[id] + 1], -1);
            }
        __syncthreads();
        // reached[c] = prefix sum of diff; column sum = seed * reached + 255 * (H - reached)  (out = in | ~filled)
        {
            const int chunk = (P.W + TAIL_THREADS - 1) / TAIL_THREADS;
            const int c0 = tid * chunk, c1 = min(P.W, c0 + chunk);
            int mine = 0;
            for (int c = c0; c < c1; ++c) mine += diff[c];
            int tot;
            int run = block_exscan(mine, scratch, &tot);
            for (int c = c0; c < c1; ++c) {
                run += diff[c];
                const int sum = (int)seed * run + 255 * (P.H - run);
                const float v = P.as_float ? __int_as_float(sum) : (float)sum;
                if (v >= (float)P.min_pixel_visible) {   // firstLastOverT: p[i] >= th
                    atomicMin(&s_first, c);
                    atomicMax(&s_last, c);
                    atomicAdd(&s_cnt, 1);
                }
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
            P.bb_x[f] = (double)last;
        }
        __syncthreads();
    }
}

}  // namespace

size_t lm_bbox_tm_bits_bytes(const lm_bb_tm_params &p, int B) { return (size_t)B * p.side_h * ((p.side_w + 31) / 32) * sizeof(uint32_t); }
// worst-case number of runs of one side view (every other pixel set)
size_t lm_bbox_tm_slow_runs(const lm_bb_tm_params &p) { return (size_t)p.side_h * ((size_t)p.side_w / 2 + 1); }

// b: frames / bkg / calib / minmax / lut / n_cols / flip / conn / B filled in by the caller (imadjust must be 0).
// hist / pred: [B][256]; bits_a / bits_b: lm_bbox_tm_bits_bytes each; need_slow: [B][2]; g_runs: chunk capacity x
// lm_bbox_tm_slow_runs x 14 bytes (slots: the frames of a chunk); disk: the kernel on the device.
int lm_launch_bbox_tm(const LmBatch &b, const lm_bb_tm_params &p, const float *d_disk, uint32_t *hist, uint8_t *pred, uint32_t *bits_a,
                      uint32_t *bits_b, int *need_slow, unsigned char *g_runs, int g_slots, uint32_t *level_mask, double *bb_x, int32_t *lims, cudaStream_t s) {
    // 1. pred[d]: the front end shared with LocoMouse_TM_DE (normalisation LUT, histogram, imadjust_default, threshold)
    lm_bb_de_params q{};
    q.side_x = p.side_x;
    q.side_y = p.side_y;
    q.side_w = p.side_w;
    q.side_h = p.side_h;
    q.threshold = (double)p.side_threshold;
    int launches = lm_launch_bbox_pred(b, q, hist, pred, s);
    if (launches < 0) return -1;
    BBTmDev P{};
    P.frames = b.frames;
    P.frame_bytes = b.frame_bytes;
    P.bkg = b.bkg;
    P.calib = b.calib;
    P.pred = pred;
    P.n_cols = b.n_cols;
    P.flip = b.flip;
    P.B = b.B;
    P.conn = b.conn;
    P.side_x = p.side_x;
    P.side_y = p.side_y;
    P.W = p.side_w;
    P.H = p.side_h;
    P.wpr = (p.side_w + 31) / 32;
    P.zc0 = std::max(0, p.zero_col_pre);
    P.zc1 = std::min(p.side_w, p.zero_col_post);
    P.zr0 = std::max(0, p.zero_row_pre);
    P.zr1 = std::min(p.side_h, p.zero_row_post);
    P.min_pixel_count = p.min_pixel_count;
    P.min_pixel_visible = p.min_pixel_visible;
    P.as_float = p.sums_as_float != 0;
    P.K = p.disk_size;
    P.disk = d_disk;
    P.bits_a = bits_a;
    P.bits_b = bits_b;
    P.need_slow = need_slow;
    P.bb_x = bb_x;
    P.lims = lims;
    const size_t runs = lm_bbox_tm_slow_runs(p);
    P.g_stride = (int64_t)runs;
    {
        unsigned char *g = g_runs;
        if (g_slots < b.B) return -1;
        const size_t n = (size_t)g_slots * runs;
        P.g_parent = reinterpret_cast<int *>(g); g += n * 4;
        P.g_area = reinterpret_cast<int *>(g); g += n * 4;
        P.g_rrow = reinterpret_cast<unsigned short *>(g); g += n * 2;
        P.g_rx0 = reinterpret_cast<unsigned short *>(g); g += n * 2;
        P.g_rx1 = reinterpret_cast<unsigned short *>(g);
    }
    int dev_smem = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaFuncAttributes fa{};
    int budget = dev_smem;
    for (const void *fn : {(const void *)k_bbtm_open<false>, (const void *)k_bbtm_open<true>, (const void *)k_bbtm_fill<false>, (const void *)k_bbtm_fill<true>}) {
        if (cudaFuncGetAttributes(&fa, fn) != cudaSuccess) return -1;
        budget = std::min(budget, dev_smem - (int)fa.sharedSizeBytes);
    }
    const size_t fixed = tm_smem(P.H, P.W, P.wpr, 0);
    if (fixed > (size_t)std::max(budget, 0)) return -2;  // the side view's bit image does not fit into shared memory
    // run capacity of the fast path: at most 4096 (two CTAs per SM for the reference geometry), less when the image is large
    int runcap = 4096;
    while (runcap > 0 && tm_smem(P.H, P.W, P.wpr, runcap) > (size_t)std::min(budget, 110 * 1024)) runcap -= 256;
    if (const char *e = getenv("LM_BBOX_RUNCAP")) runcap = std::max(0, std::min(runcap, atoi(e)));
    P.runcap = std::max(runcap, 0);
    static LmDevOnce once;
    if (auto setup = once.first()) {
        if (cudaFuncSetAttribute(k_bbtm_open<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, budget) != cudaSuccess ||
            cudaFuncSetAttribute(k_bbtm_open<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, budget) != cudaSuccess ||
            cudaFuncSetAttribute(k_bbtm_fill<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, budget) != cudaSuccess ||
            cudaFuncSetAttribute(k_bbtm_fill<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, budget) != cudaSuccess ||
            cudaFuncSetAttribute(k_bbtm_disk, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024) != cudaSuccess)
            return -1;
    }
    if (cudaMemsetAsync(need_slow, 0, (size_t)b.B * 2 * sizeof(int), s) != cudaSuccess) return -1;
    const int nwords = P.H * P.wpr;
    int gx = (nwords + 32 * 8 - 1) / (32 * 8);
    gx = gx < 1 ? 1 : (gx > 48 ? 48 : gx);
    k_bbtm_bin<<<dim3(gx, b.B), 256, 0, s>>>(P);
    const size_t smem_fast = tm_smem(P.H, P.W, P.wpr, P.runcap), smem_slow = tm_smem(P.H, P.W, P.wpr, 0);
    if (P.runcap > 0)
        k_bbtm_open<false><<<b.B, TAIL_THREADS, smem_fast, s>>>(P);
    else if (cudaMemsetAsync(need_slow, 1, (size_t)b.B * 2 * sizeof(int), s) != cudaSuccess)  // any non-zero value flags the frame
        return -1;
    k_bbtm_open<true><<<b.B, TAIL_THREADS, smem_slow, s>>>(P);
    // distinct non-zero kernel weights -> per-row tap masks for the counting path of k_bbtm_disk
    DiskLevels D{};
    uint32_t h_mask[TM_DISK_LEVELS * 64] = {0};
    {
        const int K = P.K;
        float vals[TM_DISK_LEVELS];
        int L = 0;
        double sum_abs = 0.0;
        bool ok = K <= 32;
        for (int i = 0; i < K * K && ok; ++i) {
            const float w = p.disk[i];
            sum_abs += fabs((double)w);
            if (w == 0.f) continue;
            int l = 0;
            while (l < L && vals[l] != w) ++l;
            if (l == L) {
                if (L == TM_DISK_LEVELS) {
                    ok = false;
                    break;
                }
                vals[L++] = w;
            }
            h_mask[l * K + i / K] |= 1u << (i % K);
        }
        D.L = ok ? L : 0;
        for (int l = 0; l < D.L; ++l) D.val[l] = (double)vals[l];
        // each of OpenCV's float adds rounds by at most 2^-24 of a partial sum bounded by sum|w|
        D.margin = 4.0 * (double)K * K * 5.9604644775390625e-8 * (sum_abs > 1.0 ? sum_abs : 1.0) + 1e-9;
    }
    if (cudaMemcpyAsync(level_mask, h_mask, (size_t)TM_DISK_LEVELS * 64 * sizeof(uint32_t), cudaMemcpyHostToDevice, s) != cudaSuccess) return -1;
    int gd = (nwords + DISK_THREADS - 1) / DISK_THREADS;
    gd = gd < 1 ? 1 : (gd > 256 ? 256 : gd);
    const size_t disk_smem = (((size_t)(P.K * P.K + TM_DISK_LEVELS * P.K) * 4 + 15) & ~(size_t)15) + (size_t)P.K * DISK_THREADS * 8;
    k_bbtm_disk<<<dim3(gd, b.B), DISK_THREADS, disk_smem, s>>>(P, D, level_mask);
    if (P.runcap > 0) k_bbtm_fill<false><<<b.B, TAIL_THREADS, smem_fast, s>>>(P);
    k_bbtm_fill<true><<<b.B, TAIL_THREADS, smem_slow, s>>>(P);
    launches += 6;
    return cudaGetLastError() == cudaSuccess ? launches : -1;
}
