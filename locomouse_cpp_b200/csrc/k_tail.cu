// k_tail.cu — tail detection after the two tail correlations: one CTA per frame.
//
// Replaces LocoMouse::detectLineCandidates from the binarisation on (LocoMouse_class.cpp:2593-2742)
// and selectLargestRegion (2744-2767):
//   bottom (score > 0) map -> largest connected region (= TAIL_MASK, also consumed by the bottom
//   NMS kernel) -> column-max masks the side map -> largest side region -> the bottom extent
//   [first,last) is split into n_tail_points segments -> per-segment centroids (cv::moments of a
//   binary image = pixel counts and coordinate sums, (int) truncation) -> TRACKS_TAIL (x, y, z).
//
// Connected components are labelled on RUNS, entirely in shared memory:
//   1. the u8 map is read once with 16-byte loads and packed to a row-major bit image;
//   2. run starts are  bits & ~(bits << 1 | carry) ; a block scan numbers the runs row-major, so the
//      runs of a row are contiguous and x-sorted;
//   3. every run is united with the runs of the previous row it touches (8-connectivity: [x0-1,x1+1],
//      4-connectivity: [x0,x1]) by lock-free union-find (atomicMin hooks, smaller id = root);
//   4. per root: area = sum of run lengths, OpenCV label order key = min over runs of the first 2x2 block
//      ((r>>1)*ceil(W/2) + (x0>>1)) for 8-connectivity / first pixel (r*W + x0) for 4-connectivity;
//      "largest" = max area, ties -> smallest key (oracle/lm_oracle.cpp largest_region, pinned vs cv2).
// Frames whose maps have more than RUNCAP runs take the pixel-based global-memory path (k_tail_slow).
#include <cstdlib>

#include "lm_internal.h"
#include "cc_runs.cuh"

namespace {

// u8 map [rows][pitch] (global) -> bit image in shared memory, optionally gated by colany
__device__ void load_bits(const uint8_t *bin, int rows, int cols, int pitch, int wpr, const int *colgate,
                          uint32_t *bits) {
    const int tid = threadIdx.x;
    const int nwords = rows * wpr;
    for (int wi = tid; wi < nwords; wi += TAIL_THREADS) {
        const int r = wi / wpr, c = wi - r * wpr;
        const int x0 = c * 32;
        const uint8_t *src = bin + (int64_t)r * pitch + x0;
        uint32_t w = 0;
        if (x0 + 32 <= pitch && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(src));
            const uint4 b = __ldg(reinterpret_cast<const uint4 *>(src) + 1);
            const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                // 4 bytes (each 0/1) -> 4 bits
                uint32_t t = v[q] & 0x01010101u;
                t = (t | (t >> 7) | (t >> 14) | (t >> 21)) & 0xfu;
                w |= t << (4 * q);
            }
        } else {
            for (int q = 0; q < 32 && x0 + q < cols; ++q) w |= (uint32_t)(src[q] != 0) << q;
        }
        // clear bits beyond the box and apply the column gate
        const int valid = min(32, cols - x0);
        if (valid < 32) w &= (valid <= 0) ? 0u : ((1u << valid) - 1u);
        if (colgate) {
            uint32_t g = 0;
            for (int q = 0; q < valid; ++q) g |= (uint32_t)(colgate[x0 + q] != 0) << q;
            w &= g;
        }
        bits[wi] = w;
    }
}

// winner mask bits (shared) -> u8 0/1 map (global)
__device__ void store_mask(const uint32_t *obits, int rows, int cols, int pitch, int wpr, uint8_t *mask) {
    const int nq = rows * (pitch >> 2);  // 4-pixel groups
    const int qpr = pitch >> 2;
    for (int i = threadIdx.x; i < nq; i += TAIL_THREADS) {
        const int r = i / qpr, x = (i - r * qpr) << 2;
        uint32_t out = 0;
        if (x < cols) {
            const uint32_t w = obits[r * wpr + (x >> 5)] >> (x & 31);
            out = (w & 1u) | ((w & 2u) << 7) | ((w & 4u) << 14) | ((w & 8u) << 21);
        }
        reinterpret_cast<uint32_t *>(mask + (int64_t)r * pitch)[x >> 2] = out;
    }
}

__device__ void write_tracks(const LmBatch &b, int f, int first, int last, const int *cnt_b, const int *sum_b,
                             const int *cnt_s, const int *sum_s) {
    const int np = b.n_tail_points, tid = threadIdx.x;
    int32_t *tr = b.tail + (int64_t)f * 3 * np;
    for (int i = tid; i < 3 * np; i += blockDim.x) tr[i] = -1;
    __syncthreads();
    if (last < 0) return;  // no tail region: all -1 (class.cpp:2654-2661)
    const int width = last - first, rem = width % np, reg = (width - rem) / np;
    if (tid < np) {
        const int i = tid;
        const int segw = reg + (i < rem ? 1 : 0);
        const int segx = first + i * reg + (i < rem ? i : rem);
        long long m00 = 0, m10 = 0, m01 = 0;
        for (int c = 0; c < segw; ++c) {
            m00 += cnt_b[segx + c];
            m10 += (long long)c * cnt_b[segx + c];
            m01 += sum_b[segx + c];
        }
        int x = -1;
        if (m00 > 0) {
            x = (int)(m10 / m00) + segx;
            tr[i] = x;
            tr[np + i] = (int)(m01 / m00);
        }
        if (x > 0 && cnt_s[x] > 0) tr[2 * np + i] = sum_s[x] / cnt_s[x];
    }
}

__global__ void __launch_bounds__(TAIL_THREADS) k_tail(const __grid_constant__ LmBatch b, int *need_slow, int runcap) {
    extern __shared__ __align__(16) unsigned char raw[];
    const int f = blockIdx.x, tid = threadIdx.x;
    const int cols = b.tail_w, pitch = b.tail_pitch;
    const int hb = b.bb_h[LM_BOTTOM], hs = b.bb_h[LM_SIDE], hmax = max(hb, hs);
    const int wpr = (cols + 31) >> 5;
    TailSmem S;
    unsigned char *p = raw;
    S.bits = reinterpret_cast<uint32_t *>(p); p += (size_t)hmax * wpr * 4;
    S.obits = S.bits;   // the winner mask replaces the input bits once the runs are extracted (cc_runs.cuh)
    S.rowfirst = reinterpret_cast<int *>(p); p += (size_t)(hmax + 1) * 4;
    const size_t rcap = (size_t)((runcap > 1 ? runcap : 1) + 63) & ~(size_t)63;  // run arrays are sized for the launch's threshold
    S.parent = reinterpret_cast<int *>(p); p += rcap * 4;
    S.area = reinterpret_cast<int *>(p); p += rcap * 4;
    S.key = reinterpret_cast<int *>(p); p += rcap * 4;
    S.colany = reinterpret_cast<int *>(p); p += (size_t)cols * 4;
    int *cnt_b = reinterpret_cast<int *>(p); p += (size_t)cols * 4;
    int *sum_b = reinterpret_cast<int *>(p); p += (size_t)cols * 4;
    int *cnt_s = reinterpret_cast<int *>(p); p += (size_t)cols * 4;
    int *sum_s = reinterpret_cast<int *>(p); p += (size_t)cols * 4;
    S.rrow = reinterpret_cast<unsigned short *>(p); p += rcap * 2;
    S.rx0 = reinterpret_cast<unsigned short *>(p); p += rcap * 2;
    S.rx1 = reinterpret_cast<unsigned short *>(p); p += rcap * 2;
    __shared__ int scratch[40];
    __shared__ unsigned long long s_best;
    __shared__ int s_first, s_last;

    const uint8_t *bin_b = b.tailbin[LM_BOTTOM] + (int64_t)f * hb * pitch;
    const uint8_t *bin_s = b.tailbin[LM_SIDE] + (int64_t)f * hs * pitch;
    uint8_t *mask_b = b.tailmask + (int64_t)f * hb * pitch;

    if (tid == 0) {
        s_first = 0x7fffffff;
        s_last = -1;
        need_slow[f] = 0;
    }
    load_bits(bin_b, hb, cols, pitch, wpr, nullptr, S.bits);
    __syncthreads();
    S.cnt = cnt_b;
    S.sum = sum_b;
    if (!largest_region_runs(S, hb, cols, wpr, b.conn, true, scratch, &s_best, runcap)) {
        if (tid == 0) need_slow[f] = 1;
        return;
    }
    store_mask(S.obits, hb, cols, pitch, wpr, mask_b);
    for (int c = tid; c < cols; c += TAIL_THREADS)
        if (S.colany[c]) {
            atomicMin(&s_first, c);
            atomicMax(&s_last, c);
        }
    __syncthreads();   // the winner mask (same memory as the bit image) has been written out by every thread
    load_bits(bin_s, hs, cols, pitch, wpr, S.colany, S.bits);
    __syncthreads();
    S.cnt = cnt_s;
    S.sum = sum_s;
    if (!largest_region_runs(S, hs, cols, wpr, b.conn, false, scratch, &s_best, runcap)) {
        if (tid == 0) need_slow[f] = 1;
        return;
    }
    write_tracks(b, f, s_first, s_last, cnt_b, sum_b, cnt_s, sum_s);
}

__global__ void __launch_bounds__(SLOW_THREADS) k_tail_slow(const __grid_constant__ LmBatch b, const int *need_slow) {
    extern __shared__ int sm[];
    const int f = blockIdx.x, tid = threadIdx.x;
    if (!need_slow[f]) return;
    const int cols = b.tail_w, pitch = b.tail_pitch;
    int *colany = sm, *cnt_b = sm + cols, *sum_b = sm + 2 * cols, *cnt_s = sm + 3 * cols, *sum_s = sm + 4 * cols;
    __shared__ unsigned long long s_best;
    __shared__ int s_first, s_last;
    int *L = b.cc + (int64_t)f * 3 * b.cc_stride, *area = L + b.cc_stride, *key = area + b.cc_stride;
    const int hb = b.bb_h[LM_BOTTOM], hs = b.bb_h[LM_SIDE];
    const uint8_t *bin_b = b.tailbin[LM_BOTTOM] + (int64_t)f * hb * pitch;
    const uint8_t *bin_s = b.tailbin[LM_SIDE] + (int64_t)f * hs * pitch;
    uint8_t *mask_b = b.tailmask + (int64_t)f * hb * pitch;
    uint8_t *mask_s = b.sidemask + (int64_t)f * hs * pitch;
    if (tid == 0) {
        s_first = 0x7fffffff;
        s_last = -1;
    }
    cc_largest(bin_b, nullptr, hb, cols, pitch, b.conn, L, area, key, mask_b, cnt_b, sum_b, colany, &s_best);
    for (int c = tid; c < cols; c += SLOW_THREADS)
        if (colany[c]) {
            atomicMin(&s_first, c);
            atomicMax(&s_last, c);
        }
    cc_largest(bin_s, colany, hs, cols, pitch, b.conn, L, area, key, mask_s, cnt_s, sum_s, nullptr, &s_best);
    write_tracks(b, f, s_first, s_last, cnt_b, sum_b, cnt_s, sum_s);
}

size_t tail_smem(const LmBatch &b, int runcap) {
    const size_t rcap = (size_t)((runcap > 1 ? runcap : 1) + 63) & ~(size_t)63;
    const int hmax = b.bb_h[0] > b.bb_h[1] ? b.bb_h[0] : b.bb_h[1];
    const int wpr = (b.tail_w + 31) >> 5;
    size_t s = (size_t)hmax * wpr * 4 + (size_t)(hmax + 1) * 4 + rcap * 4 * 3 + (size_t)b.tail_w * 4 * 5 +
               rcap * 2 * 3;
    return (s + 15) & ~(size_t)15;
}

}  // namespace

int lm_launch_tail(const LmBatch &b, cudaStream_t s) {
    if (b.tail_w <= 0) return 0;
    static LmDevOnce once;
    if (auto setup = once.first()) {
        cudaFuncSetAttribute(k_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        lm_prefer_max_shared(k_tail);
        lm_prefer_max_shared(k_tail_slow);
    }
    int *need_slow = b.cc_flag;
    // Run capacity of the shared-memory path; frames with more runs take k_tail_slow.  The default keeps the footprint
    // below a quarter of an SM (4 CTAs per SM: one wave for a 512-frame sub-batch).  LM_TAIL_RUNCAP overrides it (tests
    // lower it to exercise the slow path).
    int runcap = TAIL_RUNCAP_DEFAULT;
    if (const char *e = getenv("LM_TAIL_RUNCAP")) {
        int v = atoi(e);
        if (v >= 0 && v <= RUNCAP) runcap = v;
    }
    const size_t smem = tail_smem(b, runcap);
    k_tail<<<b.B, TAIL_THREADS, smem, s>>>(b, need_slow, runcap);
    k_tail_slow<<<b.B, SLOW_THREADS, (size_t)(5 * b.tail_w) * sizeof(int), s>>>(b, need_slow);
    return 2;
}
