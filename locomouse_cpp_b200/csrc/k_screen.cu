// k_screen.cu — tensor-core screen for the template correlation + sparse exact re-evaluation.
//
// Only two facts about a detector score are ever consumed downstream (LocoMouse_class.cpp): for the
// paw / snout templates its exact value IF it is > 0 and the centre pixel is not masked (1644, 1781,
// 849, 864); for the tail templates its sign (2593-2594).  Far more than 95 % of the outputs of a real
// frame are negative or masked, so the six cv::filter2D calls (845, 860, 2575-2576) are evaluated in
// two steps that together give bit-identical results to the dense exact kernel (k_corr.cu):
//
//  k_screen       (tcgen05, kind::i8, accumulators in TMEM)  every output's score in 16-bit fixed-point
//                 weights, EXACT integer arithmetic, as a banded-Toeplitz implicit GEMM:
//                     V[y, x] = sum_j sum_k  I[y + j + dy, x0 + k] * T_j[k, x - x0]
//                 M = 128 output rows, N = 32 output columns x {hi, lo} weight digit, K = 32*ks window
//                 bytes; the A operand of kernel row j is the SAME shared-memory tile as for row 0 with the
//                 descriptor start address moved j rows (16 B) down; B (the Toeplitz images of all kernel
//                 rows) stays resident in shared memory for the CTA's lifetime.  A rigorous error bound
//                 (quantisation + fp32 rounding of the exact path, lm_screen_build) turns into two integer
//                 thresholds: V <= t_lo proves score <= 0, V > t_hi proves score > 0.
//  k_corr_sparse  (FP32 FFMA, oracle tap order)  re-evaluates only the 2x4 output patches that contain an
//                 output the screen could not decide (paw / snout: possibly positive and unmasked; tail:
//                 sign not proven) and emits exactly what the dense kernel emits for those patches.
//
// Warp roles of k_screen (persistent, one CTA per SM): warps 0-3 epilogue (TMEM lanes 32w..32w+31),
// warps 4-5 window-tile loaders (global -> shared, 16-byte column panels), warp 6 MMA issuer + TMEM owner.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "lm_internal.h"
#include "corr_common.cuh"
#include "umma_common.cuh"

namespace {

constexpr int SCR_THREADS = 224;
constexpr int SCR_TILE_M = 128;   // output rows per tile  (UMMA M)
constexpr int SCR_TILE_X = 32;    // output columns per tile
constexpr int SCR_N = 64;         // UMMA N = 32 columns x 2 digits
constexpr int SCR_STAGES = 4;     // window-tile ring
constexpr int SCR_TMEM_COLS = 128;  // two accumulators of 64 columns
constexpr int SCR_BJ = 1024;      // bytes of one 16-byte K chunk of B: 64 rows x 16 B

struct ScreenJobDev {
    LmScreenJob j;
    int view, feat, is_tail;
    int out_w, out_h;
    int nxt, nyt;
    int cta_begin, ncta;
    int halo_x, halo_y;
    int *ntasks;
};

struct ScreenParams {
    ScreenJobDev job[6];
    int njobs;
    int B;
    const uint8_t *win[2];
    int win_h[2], win_pitch[2];
    int64_t win_stride[2];
    uint8_t *tailbin[2];
    int tail_pitch;
    int64_t tailbin_stride[2];
};

__global__ void __launch_bounds__(SCR_THREADS, 1) k_screen(const __grid_constant__ ScreenParams P) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t bars[2 * SCR_STAGES + 4];
    __shared__ uint32_t tmem_base_s;

    int ji = 0;
    for (int q = 1; q < P.njobs; ++q)
        if ((int)blockIdx.x >= P.job[q].cta_begin) ji = q;
    const ScreenJobDev &J = P.job[ji];
    const int rank = blockIdx.x - J.cta_begin;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kh = J.j.kh, ks = J.j.ks, rows = J.j.rows;
    const int npanel = 2 * ks;
    const uint32_t panel_a = (uint32_t)rows * 16u;
    const uint32_t stage_bytes = panel_a * npanel;
    const uint32_t b_bytes = (uint32_t)kh * npanel * SCR_BJ;
    uint8_t *sB = smem;
    uint8_t *sA = smem + b_bytes;
    const int tiles_per_frame = J.nxt * J.nyt;
    const int ntiles = P.B * tiles_per_frame;

    const uint32_t bar0 = smem_u32(bars);
    auto a_full = [&](int s) { return bar0 + 8u * s; };
    auto a_empty = [&](int s) { return bar0 + 8u * (SCR_STAGES + s); };
    auto d_full = [&](int a) { return bar0 + 8u * (2 * SCR_STAGES + a); };
    auto d_empty = [&](int a) { return bar0 + 8u * (2 * SCR_STAGES + 2 + a); };

    // ---- one-time setup: B operand -> shared memory, barriers, TMEM ------------------------------------------
    {
        const int4 *src = reinterpret_cast<const int4 *>(J.j.Bimg);
        int4 *dst = reinterpret_cast<int4 *>(sB);
        for (uint32_t i = tid; i < b_bytes / 16; i += SCR_THREADS) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        for (int s = 0; s < SCR_STAGES; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a_full(s)), "r"(64));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a_empty(s)), "r"(1));
        }
        for (int a = 0; a < 2; ++a) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(d_full(a)), "r"(1));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(d_empty(a)), "r"(128));
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 6) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "r"(SCR_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    if (warp >= 4 && warp < 6) {
        // ================= loaders: window rows [y0, y0 + rows) x columns [x0, x0 + 32 ks) -> 16-byte panels =====
        const int ll = tid - 128;  // 0..63
        const int v = J.view;
        const int win_h = P.win_h[v], pitch = P.win_pitch[v];
        const int nchunks = rows * npanel;
        int stage = 0;
        uint32_t phase = 0;
        for (int t = rank; t < ntiles; t += J.ncta) {
            const int f = t / tiles_per_frame, rem = t - f * tiles_per_frame;
            const int yt = rem / J.nxt, xt = rem - yt * J.nxt;
            const int y0 = yt * SCR_TILE_M, x0 = xt * SCR_TILE_X;
            const uint8_t *wbase = P.win[v] + (int64_t)f * P.win_stride[v];
            mbar_wait(a_empty(stage), phase ^ 1u);
            uint8_t *dstA = sA + (uint32_t)stage * stage_bytes;
            constexpr int UNR = 5;
            for (int base = 0; base < nchunks; base += 64 * UNR) {
                int4 val[UNR];
#pragma unroll
                for (int q = 0; q < UNR; ++q) {
                    const int idx = base + q * 64 + ll;
                    int4 x = make_int4(0, 0, 0, 0);
                    if (idx < nchunks) {
                        const int r = idx / npanel, p = idx - r * npanel;
                        const int wr = y0 + r, wc = x0 + 16 * p;
                        if (wr < win_h && wc + 16 <= pitch) x = __ldg(reinterpret_cast<const int4 *>(wbase + (int64_t)wr * pitch + wc));
                    }
                    val[q] = x;
                }
#pragma unroll
                for (int q = 0; q < UNR; ++q) {
                    const int idx = base + q * 64 + ll;
                    if (idx < nchunks) {
                        const int r = idx / npanel, p = idx - r * npanel;
                        *reinterpret_cast<int4 *>(dstA + (uint32_t)p * panel_a + (uint32_t)r * 16u) = val[q];
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic stores -> visible to the tensor core
            mbar_arrive(a_full(stage));
            if (++stage == SCR_STAGES) {
                stage = 0;
                phase ^= 1u;
            }
        }
    } else if (warp == 6) {
        // ================= MMA issuer: kh * ks instructions per tile, one thread ================================
        // u8 x s8 -> s32, both operands K-major, N = 64, M = 128
        const uint32_t idesc = (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(SCR_N >> 3) << 17) | ((uint32_t)(SCR_TILE_M >> 4) << 24);
        const uint64_t bdesc0 = umma_desc(smem_u32(sB), SCR_BJ);
        const uint32_t a_step = (2u * panel_a) >> 4, b_step = (2u * SCR_BJ) >> 4;  // one K step, in descriptor units
        const uint32_t b_row = ((uint32_t)npanel * SCR_BJ) >> 4;                  // one kernel row of B
        int stage = 0, acc = 0;
        uint32_t phase = 0, accphase = 0;
        for (int t = rank; t < ntiles; t += J.ncta) {
            mbar_wait(d_empty(acc), accphase ^ 1u);
            mbar_wait(a_full(stage), phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (elect_one()) {
                const uint32_t d = tmem + (uint32_t)acc * SCR_N;
                uint64_t adesc = umma_desc(smem_u32(sA) + (uint32_t)stage * stage_bytes + (uint32_t)J.j.dy * 16u, panel_a);
                uint64_t bdesc = bdesc0;
                uint32_t accum = 0;
                for (int j = 0; j < kh; ++j) {
                    uint64_t ad = adesc, bd = bdesc;
                    for (int k = 0; k < ks; ++k) {
                        umma_i8(d, ad, bd, idesc, accum);
                        accum = 1;
                        ad += a_step;
                        bd += b_step;
                    }
                    adesc += 1;  // next kernel row: the same tile, 16 bytes (one row) further down
                    bdesc += b_row;
                }
                umma_commit(a_empty(stage));  // frees the window tile when these MMAs have read it
                umma_commit(d_full(acc));     // accumulator complete
            }
            __syncwarp();
            if (++stage == SCR_STAGES) {
                stage = 0;
                phase ^= 1u;
            }
            if (++acc == 2) {
                acc = 0;
                accphase ^= 1u;
            }
        }
    } else {
        // ================= epilogue: thresholds -> survivor patches (+ provisional tail signs) ==================
        const int v = J.view;
        const int pitch = P.win_pitch[v];
        const long long t_lo = J.j.t_lo, t_hi = J.j.t_hi;
        int acc = 0;
        uint32_t accphase = 0;
        for (int t = rank; t < ntiles; t += J.ncta) {
            const int f = t / tiles_per_frame, rem = t - f * tiles_per_frame;
            const int yt = rem / J.nxt, xt = rem - yt * J.nxt;
            const int y = yt * SCR_TILE_M + tid, x0 = xt * SCR_TILE_X;
            mbar_wait(d_full(acc), accphase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t hi[32], lo[32];
            const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)acc * SCR_N;
            tmem_ld32(ta, hi);
            tmem_ld32(ta + 32, lo);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            mbar_arrive(d_empty(acc));
            if (++acc == 2) {
                acc = 0;
                accphase ^= 1u;
            }
            const bool rowok = y < J.out_h;
            uint32_t need = 0, sign = 0;  // bit c: output (y, x0 + c) needs the exact kernel / is provisionally > 0
#pragma unroll
            for (int c = 0; c < 32; ++c) {
                const long long V = (long long)(int)hi[c] * 256 + (long long)(int)lo[c];
                if (V > t_lo) need |= 1u << c;
                if (V > t_hi) sign |= 1u << c;
            }
            const int wvalid = J.out_w - x0;  // columns of this tile inside the box
            const uint32_t colmask = wvalid >= 32 ? 0xffffffffu : (wvalid <= 0 ? 0u : ((1u << wvalid) - 1u));
            need = rowok ? (need & colmask) : 0u;
            if (J.is_tail) {
                if (rowok) {
                    // provisional sign map (undecided outputs are rewritten by k_corr_sparse)
                    uint8_t *tb = P.tailbin[v] + (int64_t)f * P.tailbin_stride[v] + (int64_t)y * P.tail_pitch + x0;
                    uint32_t w[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const uint32_t nib = (sign >> (4 * q)) & 0xfu;
                        w[q] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
                    }
                    reinterpret_cast<uint4 *>(tb)[0] = make_uint4(w[0], w[1], w[2], w[3]);
                    reinterpret_cast<uint4 *>(tb)[1] = make_uint4(w[4], w[5], w[6], w[7]);
                }
                need &= ~sign;  // undecided = above t_lo but not above t_hi
            } else if (need) {
                // setTo(0, mask): outputs whose centre pixel is <= 25 are never detections (class.cpp:782, 817)
                const uint8_t *crow = P.win[v] + (int64_t)f * P.win_stride[v] + (int64_t)(y + J.halo_y) * pitch + x0 + J.halo_x;
                uint32_t m = need;
                while (m) {
                    const int c = __ffs(m) - 1;
                    m &= m - 1;
                    if (__ldg(crow + c) <= 25) need &= ~(1u << c);
                }
            }
            // 2x4 patches: lanes 2k, 2k+1 hold the two rows of patch row (y >> 1); bit q of pf = columns 4q .. 4q+3
            uint32_t pf = lm_nibble_any(need);
            pf |= __shfl_xor_sync(0xffffffffu, pf, 1);
            const int cnt = ((lane & 1) == 0) ? __popc(pf) : 0;
            const uint32_t any = __ballot_sync(0xffffffffu, cnt > 0);
            if (any) {
                int incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int u = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += u;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                int base = 0;
                if (lane == 31) base = atomicAdd(J.ntasks, total);
                base = __shfl_sync(0xffffffffu, base, 31);
                int o = base + incl - cnt;
                if (cnt) {
                    const uint32_t head = ((uint32_t)f << 16) | ((uint32_t)(y >> 1) << 8);
                    uint32_t m = pf;
                    while (m) {
                        const int q = __ffs(m) - 1;
                        m &= m - 1;
                        if (o < J.j.task_cap) J.j.tasks[o] = head | (uint32_t)((x0 >> 2) + q);
                        ++o;
                    }
                }
            }
        }
    }
    // ---- teardown ---------------------------------------------------------------------------------------------
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 6) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(SCR_TMEM_COLS));
    }
}

// =================================================================================================================
// k_corr_sparse: one thread per undecided 2x4 patch, exact fp32 scores in the oracle's tap order.
// =================================================================================================================
constexpr int SP_THREADS = 128;
constexpr int SP_TX = 4, SP_TY = 2;   // patch = 2 rows x 4 columns (task word: frame << 16 | patch_row << 8 | patch_col)

struct SparseJob {
    int view, feat, is_tail;
    int out_w, out_h;
    int kh, kw, kwp;
    int dx, dy;        // window column / row of tap (0,0) for output (0,0)
    int halo_x, halo_y;
    float init;
    const float *w;    // device, row stride kw
    const uint32_t *tasks;
    const int *ntasks;
    int task_cap;
};

struct SparseParams {
    SparseJob job[6];
    int njobs;
    int det_cap, box_w;
    const uint8_t *win[2];
    int win_h[2], win_pitch[2];
    int64_t win_stride[2];
    uint8_t *tailbin[2];
    int tail_pitch;
    int64_t tailbin_stride[2];
    LmDet *det;
    int32_t *det_count;
};

template <int NP>
__device__ __forceinline__ void sp_load_words(uint32_t (&w)[NP / 4 + 1], const uint8_t *row_aligned) {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(row_aligned);
#pragma unroll
    for (int q = 0; q < NP / 4 + 1; ++q) w[q] = __ldg(src + q);
}

template <int NP>
__device__ __forceinline__ void sp_words_to_px(float (&p)[NP], const uint32_t (&w)[NP / 4 + 1], int shift) {
#pragma unroll
    for (int q = 0; q < NP / 4; ++q) {
        const uint32_t u = __funnelshift_r(w[q], w[q + 1], shift);
        p[4 * q + 0] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7540)) - 8388608.f;
        p[4 * q + 1] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7541)) - 8388608.f;
        p[4 * q + 2] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7542)) - 8388608.f;
        p[4 * q + 3] = __uint_as_float(__byte_perm(u, 0x4B000000u, 0x7543)) - 8388608.f;
    }
}

template <int KW, bool FMA>
__global__ void __launch_bounds__(SP_THREADS) k_corr_sparse(const __grid_constant__ SparseParams P, int kwp_filter) {
    constexpr int TX = SP_TX, TY = SP_TY;
    constexpr int NP = ((TX + KW - 1 + 3) / 4) * 4;
    constexpr int KW4 = ((KW + 3) / 4) * 4;
    extern __shared__ __align__(16) float wsm[];  // [kh][KW4]
    const SparseJob &J = P.job[blockIdx.y];
    if (J.kwp != kwp_filter) return;
    int ntasks = *J.ntasks;
    if (ntasks > J.task_cap) ntasks = J.task_cap;
    if ((int)(blockIdx.x * SP_THREADS) >= ntasks) return;
    const int tid = threadIdx.x;
    for (int idx = tid; idx < J.kh * KW4; idx += SP_THREADS) {
        const int j = idx / KW4, i = idx - j * KW4;
        wsm[idx] = (i < J.kw) ? J.w[j * J.kw + i] : 0.f;
    }
    __syncthreads();
    const int v = J.view;
    const int pitch = P.win_pitch[v], win_h = P.win_h[v];
    const int kh = J.kh;
    for (int ti = blockIdx.x * SP_THREADS + tid; ti < ntasks; ti += gridDim.x * SP_THREADS) {
        const uint32_t task = J.tasks[ti];
        const int f = (int)(task >> 16), y0 = (int)((task >> 8) & 255u) * TY, x0 = (int)(task & 255u) * TX;
        const uint8_t *wbase = P.win[v] + (int64_t)f * P.win_stride[v];
        const int col0 = x0 + J.dx;
        const int shift = (col0 & 3) * 8;
        const uint8_t *colbase = wbase + (col0 & ~3);
        const int row0 = y0 + J.dy;
        float acc[TY][TX];
#pragma unroll
        for (int t = 0; t < TY; ++t)
#pragma unroll
            for (int k = 0; k < TX; ++k) acc[t][k] = J.init;
        const int nr = kh + TY - 1;
        uint32_t wcur[NP / 4 + 1], wnext[NP / 4 + 1];
        auto rowptr = [&](int r) {
            int wr = row0 + r;
            wr = wr < win_h ? wr : win_h - 1;  // rows past the window only feed outputs outside the box
            return colbase + (int64_t)wr * pitch;
        };
        sp_load_words<NP>(wcur, rowptr(0));
        for (int r = 0; r < nr; ++r) {
            if (r + 1 < nr) sp_load_words<NP>(wnext, rowptr(r + 1));
            float px[NP];
            sp_words_to_px<NP>(px, wcur, shift);
            if (r >= TY - 1 && r < kh) {
#pragma unroll
                for (int t = 0; t < TY; ++t) corr_taps<KW, TX, FMA, NP>(acc[t], px, wsm + (r - t) * KW4);
            } else {
#pragma unroll
                for (int t = 0; t < TY; ++t) {
                    const int j = r - t;
                    if (j >= 0 && j < kh) corr_taps<KW, TX, FMA, NP>(acc[t], px, wsm + j * KW4);
                }
            }
#pragma unroll
            for (int q = 0; q < NP / 4 + 1; ++q) wcur[q] = wnext[q];
        }
        // ---- the dense kernel's epilogue for this patch ---------------------------------------------------------
        if (J.is_tail) {
            uint8_t *tb = P.tailbin[v] + (int64_t)f * P.tailbin_stride[v];
#pragma unroll
            for (int t = 0; t < TY; ++t) {
                const int y = y0 + t;
                if (y >= J.out_h) continue;
#pragma unroll
                for (int k = 0; k < TX; ++k) {
                    const int x = x0 + k;
                    if (x < J.out_w) tb[(int64_t)y * P.tail_pitch + x] = acc[t][k] > 0.f ? 1 : 0;
                }
            }
            continue;
        }
        unsigned hit = 0;
        int cnt = 0;
#pragma unroll
        for (int t = 0; t < TY; ++t) {
            const int y = y0 + t;
#pragma unroll
            for (int k = 0; k < TX; ++k) {
                const int x = x0 + k;
                if (y < J.out_h && x < J.out_w && acc[t][k] > 0.f) {
                    const uint8_t centre = __ldg(wbase + (int64_t)(y + J.halo_y) * pitch + x + J.halo_x);
                    if (centre > 25) {
                        hit |= 1u << (t * TX + k);
                        ++cnt;
                    }
                }
            }
        }
        if (cnt) {
            const int list = (f * 2 + J.feat) * 2 + v;
            int o = atomicAdd(&P.det_count[list], cnt);
            LmDet *out = P.det + (int64_t)list * P.det_cap;
#pragma unroll
            for (int t = 0; t < TY; ++t)
#pragma unroll
                for (int k = 0; k < TX; ++k)
                    if (hit & (1u << (t * TX + k))) {
                        if (o < P.det_cap) {
                            LmDet d;
                            d.idx = (uint32_t)((y0 + t) * P.box_w + x0 + k);
                            d.score = acc[t][k];
                            out[o] = d;
                        }
                        ++o;
                    }
        }
    }
}

template <int KW>
cudaError_t launch_sparse_kw(const SparseParams &P, dim3 grid, size_t smem, bool fma, cudaStream_t s) {
    static LmDevOnce once;
    if (auto setup = once.first()) {
        lm_prefer_max_shared(k_corr_sparse<KW, true>);
        lm_prefer_max_shared(k_corr_sparse<KW, false>);
    }
    if (fma)
        k_corr_sparse<KW, true><<<grid, SP_THREADS, smem, s>>>(P, KW);
    else
        k_corr_sparse<KW, false><<<grid, SP_THREADS, smem, s>>>(P, KW);
    return cudaGetLastError();
}

}  // namespace

// ---- host side: quantisation, Toeplitz image, thresholds ------------------------------------------------------
size_t lm_screen_smem_bytes(int kh, int ks, int rows, int stages) {
    return (size_t)kh * 2 * ks * SCR_BJ + (size_t)stages * 2 * ks * rows * 16;
}

// 16-bit fixed-point weights (balanced int8 digits v = 256 * hi + lo) and the rigorous decision thresholds.
static bool screen_quantize(const float *w, int ntaps, float init, std::vector<int> *vq, LmScreenHost *out) {
    double wmax = 0.0, wabs = 0.0;
    for (int i = 0; i < ntaps; ++i) {
        if (!std::isfinite(w[i])) return false;
        wmax = std::max(wmax, std::fabs((double)w[i]));
        wabs += std::fabs((double)w[i]);
    }
    if (!std::isfinite(init)) return false;
    const double scale = wmax > 0.0 ? wmax / 32000.0 : 1.0;
    vq->resize(ntaps);
    double eq = 0.0;
    for (int i = 0; i < ntaps; ++i) {
        long v = std::lround((double)w[i] / scale);
        v = std::max(-32000L, std::min(32000L, v));
        (*vq)[i] = (int)v;
        eq += std::fabs((double)w[i] - scale * (double)v);
    }
    // |exact fp32 score - real-valued score| <= (2 taps + 2) u (|rho| + 255 sum|w|)   (covers FMA and mul+add orders)
    // |real-valued score - scale * V + rho|  <= 255 sum|w - scale v|
    const double rho_f = -(double)init;
    const double u = std::ldexp(1.0, -24);
    const double efp = (2.0 * ntaps + 2.0) * u * (std::fabs(rho_f) + 255.0 * wabs) * 1.01;
    const double eps = (255.0 * eq + efp) * (1.0 + 1e-9) + 1e-300;
    const double lo = std::floor((rho_f - eps) / scale) - 1.0, hi = std::ceil((rho_f + eps) / scale) + 1.0;
    const double lim = 4.0e18;
    out->t_lo = (long long)std::max(-lim, std::min(lim, lo));
    out->t_hi = (long long)std::max(-lim, std::min(lim, hi));
    out->scale = scale;
    out->eps = eps;
    return true;
}
static inline void split_digits(int v, int *hi8, int *lo8) {
    *lo8 = ((v + 128) & 255) - 128;
    *hi8 = (v - *lo8) / 256;
}

bool lm_screen_quantize(const float *w, int kh, int kw, float init, LmScreenHost *out) {
    std::vector<int> vq;
    return screen_quantize(w, kh * kw, init, &vq, out);
}

bool lm_screen_build(const float *w, int kh, int kw, float init, int halo_x, int halo_y, int fma_mode, LmScreenHost *out,
                     std::vector<int8_t> *img) {
    (void)fma_mode;
    const int ax = kw / 2, ay = kh / 2;
    const int dx = halo_x - ax, dy = halo_y - ay;
    if (dx < 0 || dy < 0) return false;
    const int kbytes = SCR_TILE_X - 1 + dx + kw;  // window bytes a tile row needs
    const int ks = (kbytes + 31) / 32;
    const int rows = (SCR_TILE_M + kh - 1 + dy + 7) & ~7;
    if (lm_screen_smem_bytes(kh, ks, rows, SCR_STAGES) > 220 * 1024) return false;
    std::vector<int> vq;
    if (!screen_quantize(w, kh * kw, init, &vq, out)) return false;
    out->kh = kh;
    out->ks = ks;
    out->dx = dx;
    out->dy = dy;
    out->rows = rows;
    // B image: [kh][2 ks chunks][64 rows][16 bytes]; row n < 32: hi digit of output column n, n >= 32: lo digit of
    // column n - 32; element k of the row = digit(v[j][k - c - dx]) inside the band, 0 outside.
    const int npanel = 2 * ks;
    img->assign((size_t)kh * npanel * SCR_BJ, 0);
    for (int j = 0; j < kh; ++j)
        for (int c = 0; c < SCR_TILE_X; ++c)
            for (int i = 0; i < kw; ++i) {
                const int k = c + dx + i;
                int hi8, lo8;
                split_digits(vq[j * kw + i], &hi8, &lo8);
                const size_t base = (size_t)j * npanel * SCR_BJ + (size_t)(k >> 4) * SCR_BJ + (size_t)(k & 15);
                (*img)[base + (size_t)c * 16] = (int8_t)hi8;
                (*img)[base + (size_t)(c + 32) * 16] = (int8_t)lo8;
            }
    return true;
}

bool lm_screen_build_plane(const float *w, int kh, int kw, float init, int dx, int dy, int KH, int ks, int digit, int plane, int nplanes,
                           LmScreenHost *out, std::vector<int8_t> *img) {
    if (dx < 0 || dy < 0 || dy + kh > KH || SCR_TILE_X - 1 + dx + kw > 32 * ks || plane < 0 || plane >= nplanes) return false;
    std::vector<int> vq;
    if (!screen_quantize(w, kh * kw, init, &vq, out)) return false;
    out->kh = KH;
    out->ks = ks;
    out->dx = dx;
    out->dy = dy;
    out->rows = (SCR_TILE_M + KH - 1 + 7) & ~7;
    const int npanel = 2 * ks;
    const size_t chunk = (size_t)nplanes * 32 * 16;
    if (img->size() != (size_t)KH * npanel * chunk) return false;
    for (int jj = 0; jj < kh; ++jj)
        for (int c = 0; c < SCR_TILE_X; ++c)
            for (int i = 0; i < kw; ++i) {
                const int k = c + dx + i;
                int hi8, lo8;
                split_digits(vq[jj * kw + i], &hi8, &lo8);
                const size_t base = (size_t)(jj + dy) * npanel * chunk + (size_t)(k >> 4) * chunk + (size_t)(k & 15);
                (*img)[base + (size_t)(plane * 32 + c) * 16] = (int8_t)(digit == 0 ? hi8 : lo8);
            }
    return true;
}

int lm_launch_screen(const LmBatch &b, cudaStream_t s) {
    const int n_sm = lm_sm_count();
    ScreenParams P{};
    SparseParams Q{};
    size_t smem = 0;
    double work[6], total = 0.0;
    for (int v = 0; v < 2; ++v)
        for (int k = 0; k < 3; ++k) {
            if (k == LM_TAIL && b.tail_w <= 0) continue;
            const LmScreenJob &sj = b.scr.job[v][k];
            ScreenJobDev &J = P.job[P.njobs];
            J.j = sj;
            J.view = v;
            J.feat = k;
            J.is_tail = (k == LM_TAIL);
            J.out_w = J.is_tail ? b.tail_w : b.view[v].box_w;
            J.out_h = b.view[v].box_h;
            J.nxt = (J.out_w + SCR_TILE_X - 1) / SCR_TILE_X;
            J.nyt = (J.out_h + SCR_TILE_M - 1) / SCR_TILE_M;
            J.halo_x = b.view[v].halo_x;
            J.halo_y = b.view[v].halo_y;
            J.ntasks = b.scr.ntasks + (v * 3 + k);
            work[P.njobs] = (double)J.nxt * J.nyt * sj.kh * sj.ks;
            total += work[P.njobs];
            smem = std::max(smem, lm_screen_smem_bytes(sj.kh, sj.ks, sj.rows, SCR_STAGES));
            SparseJob &S = Q.job[Q.njobs++];
            S.view = v;
            S.feat = k;
            S.is_tail = J.is_tail;
            S.out_w = J.out_w;
            S.out_h = J.out_h;
            S.kh = b.tmpl[v][k].kh;
            S.kw = b.tmpl[v][k].kw;
            S.kwp = lm_corr_kwp(S.kw);
            S.dx = sj.dx;
            S.dy = sj.dy;
            S.halo_x = J.halo_x;
            S.halo_y = J.halo_y;
            S.init = b.tmpl[v][k].init;
            S.w = b.tmpl[v][k].w;
            S.tasks = sj.tasks;
            S.ntasks = J.ntasks;
            S.task_cap = sj.task_cap;
            ++P.njobs;
        }
    if (!P.njobs) return 0;
    // CTAs are dealt to the jobs in proportion to their MMA work (one persistent CTA per SM)
    if (b.scr.enabled == 1) {
        int left = n_sm, cta = 0;
        double wleft = total;
        for (int q = 0; q < P.njobs; ++q) {
            int n = (q == P.njobs - 1) ? left : (int)std::lround(left * work[q] / wleft);
            n = std::max(1, std::min(n, left - (P.njobs - 1 - q)));
            P.job[q].cta_begin = cta;
            P.job[q].ncta = n;
            cta += n;
            left -= n;
            wleft -= work[q];
        }
    }
    P.B = b.B;
    Q.det_cap = b.det_cap;
    Q.box_w = b.bb_w;
    for (int v = 0; v < 2; ++v) {
        P.win[v] = Q.win[v] = b.win[v];
        P.win_h[v] = Q.win_h[v] = b.view[v].win_h;
        P.win_pitch[v] = Q.win_pitch[v] = b.view[v].win_pitch;
        P.win_stride[v] = Q.win_stride[v] = b.view[v].win_stride;
        P.tailbin[v] = Q.tailbin[v] = b.tailbin[v];
        P.tailbin_stride[v] = Q.tailbin_stride[v] = (int64_t)b.bb_h[v] * b.tail_pitch;
    }
    P.tail_pitch = Q.tail_pitch = b.tail_pitch;
    Q.det = b.det;
    Q.det_count = b.det_count;

    if (cudaMemsetAsync(b.scr.ntasks, 0, 16 * sizeof(int), s) != cudaSuccess) return -1;
    static LmDevOnce once;
    if (auto setup = once.first()) {
        if (cudaFuncSetAttribute(k_screen, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024) != cudaSuccess) return -1;
    }
    if (b.scr.enabled == 2) {
        // The screen owns whole SMs (its B operand fills shared memory), everything else is latency bound: on its own
        // high-priority stream its CTAs take the SMs as soon as the previous sub-batch's screen leaves them.
        const bool hi = b.screen_stream && b.ev_screen_go && b.ev_screen_done;
        if (hi) {
            if (cudaEventRecord(b.ev_screen_go, s) != cudaSuccess || cudaStreamWaitEvent(b.screen_stream, b.ev_screen_go, 0) != cudaSuccess) return -1;
        }
        if (b.ev_screen_start) cudaEventRecord(b.ev_screen_start, hi ? b.screen_stream : s);
        if (!(lm_whatif_skip() & 4) && lm_launch_screen2_kernel(b, hi ? b.screen_stream : s) < 0) return -1;
        if (hi) {
            if (cudaEventRecord(b.ev_screen_done, b.screen_stream) != cudaSuccess || cudaStreamWaitEvent(s, b.ev_screen_done, 0) != cudaSuccess) return -1;
        }
    } else {
        int total_cta = P.job[P.njobs - 1].cta_begin + P.job[P.njobs - 1].ncta;
        k_screen<<<total_cta, SCR_THREADS, smem, s>>>(P);
        if (cudaGetLastError() != cudaSuccess) return -1;
    }
    if (b.ev_screen_done && !(b.scr.enabled == 2 && b.screen_stream && b.ev_screen_go)) cudaEventRecord(b.ev_screen_done, s);
    int launches = 1;
    // sparse exact pass: one launch per distinct padded kernel width (the jobs of other widths exit at once)
    bool done[6] = {};
    const bool fma = b.fma_mode != 0;
    for (int q0 = 0; q0 < Q.njobs; ++q0) {
        if (done[q0] || (lm_whatif_skip() & 8)) continue;
        const int kwp = lm_corr_kwp(Q.job[q0].kw);
        int kh_max = 0;
        for (int q = q0; q < Q.njobs; ++q)
            if (lm_corr_kwp(Q.job[q].kw) == kwp) {
                done[q] = true;
                kh_max = std::max(kh_max, Q.job[q].kh);
            }
        const size_t wsmem = (size_t)kh_max * (((kwp + 3) / 4) * 4) * sizeof(float);
        const dim3 grid(n_sm * 4, Q.njobs);
        cudaError_t e = cudaSuccess;
        switch (kwp) {
            case 8: e = launch_sparse_kw<8>(Q, grid, wsmem, fma, s); break;
            case 16: e = launch_sparse_kw<16>(Q, grid, wsmem, fma, s); break;
            case 24: e = launch_sparse_kw<24>(Q, grid, wsmem, fma, s); break;
            case 30: e = launch_sparse_kw<30>(Q, grid, wsmem, fma, s); break;
            case 32: e = launch_sparse_kw<32>(Q, grid, wsmem, fma, s); break;
            case 48: e = launch_sparse_kw<48>(Q, grid, wsmem, fma, s); break;
            case 60: e = launch_sparse_kw<60>(Q, grid, wsmem, fma, s); break;
            case 64: e = launch_sparse_kw<64>(Q, grid, wsmem, fma, s); break;
            default: e = cudaErrorInvalidValue;
        }
        if (e != cudaSuccess) return -1;
        ++launches;
    }
    return launches;
}
