// k_screen2.cu — the tensor-core screen of k_screen.cu on CTA PAIRS (tcgen05 cta_group::2).
//
// Why: a single CTA can only keep ONE template's Toeplitz operand resident (120 kB), i.e. N = 64 per instruction, which the
// tensor pipe executes in 32 cycles but which cannot be issued faster than every ~43-50 (tools/umma_pair_probe.cu).  A CTA pair
// executes one M = 256 instruction: each CTA streams its own 128 window rows (its own y tile of the same frame / x tile) and
// holds only HALF of B, so three templates fit and N = 192 runs at the tensor pipe's rate (96 cycles, 8187 MAC/clk/SM):
//   paw + snout + tail job : N = 192 = 32 columns x [paw hi | paw lo | tail hi || snout hi | snout lo | tail lo]; the first
//                            three planes live in CTA 0's shared memory, the others in CTA 1's.  x tiles right of the tail
//                            box issue the same operands with N = 128 (each CTA's first two planes, 64 cycles).
//   paw + snout job        : N = 128 (templates whose sizes differ too much to share kernel-row steps with the tail)
//   one-template job       : N = 64  = [hi || lo]; hi digits in CTA 0, lo digits in CTA 1.
// y tiles: either whole 256-row tile pairs per frame, or -- when that wastes more (side view: 150 of 256 rows) --
// "stacked": the sub-batch's windows, contiguous in memory at the window pitch, are treated as one tall image and cut
// into 256-row tile pairs (179-row windows: 84 % useful rows instead of 59 %); a tile may straddle two frames, each
// accumulator row maps back to (frame, y) and rows in the inter-frame halo are dropped.
// Everything else (exact int8 arithmetic, thresholds, 2x4 patch tasks for k_corr_sparse) is k_screen.cu's.
//
// Pair protocol: window-tile "full" and accumulator "empty" barriers live in the leader CTA (rank 0) and
// collect arrivals from both CTAs (remote arrive through mapa); tcgen05.commit multicasts "tile free" and
// "accumulator full" to the barrier at the same offset in both CTAs.  Only the leader issues MMAs.
// Window tiles are moved by the TMA unit (cp.async.bulk.tensor, cta_group::2: each CTA's boxes land in its own
// shared memory and their bytes are counted on the leader's "full" barrier), one elected producer thread per CTA.
#include <cuda.h>

#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>

#include "lm_internal.h"
#include "umma_common.cuh"

namespace {

// warps 0-7 epilogue (two groups of four: group g = warp >> 2 drains accumulator g, i.e. every other unit; warp & 3 = its TMEM
// lane quadrant), 8 TMA producer, 9 MMA issuer / TMEM owner.  In isolation the pair instruction runs at the tensor pipe's rate
// (tools/umma_pair_probe.cu: N = 192 -> 96 cycles); what it needs from the rest of the kernel is an epilogue that drains an
// accumulator within one unit's MMA time (60 x 64 .. 96 cycles), hence two groups and no dependent global-memory chains below.
constexpr int S2_THREADS = 320;
constexpr int S2_WARP_TMA = 8, S2_WARP_MMA = 9;
constexpr int S2_TILE_M = 128;
constexpr int S2_TILE_X = 32;
constexpr int S2_STAGES = 4;      // maximum ring depth; a job uses J.j.stages of them
constexpr int S2_TMEM_COLS = 512; // two accumulators of up to 256 columns
constexpr int S2_ACC_STRIDE = 256;
constexpr int S2_RING = 16;       // published unit indices in flight (the scheduler runs at most stages + 4 units ahead of the slowest reader)

struct Screen2JobDev {
    LmScreen2Job j;
    int out_h, out_w[3];
    int nxt;                  // x tiles
    int ntp;                  // 256-row tile pairs over the whole sub-batch
    int VH;                   // rows between consecutive frames in tile-row space (window height when stacked)
    int pair_begin, npair;
    int *next_unit;           // device counter (zeroed with the task counters): units beyond each pair's first are claimed here
    int halo_x, halo_y;
    // 32-bit form of the thresholds on H = hi + (lo >> 8) (V = 256 H + (lo & 255)):  V > t_lo  =>  H >= q_need;
    // H > q_sign  =>  V > t_hi.  Conservative by less than one hi-digit unit (256 of ~2e5 units between t_lo and t_hi).
    int q_need[3], q_sign[3];
};

struct Screen2Params {
    // Window tiles arrive by TMA: per job one tiled tensor map over the sub-batch's windows of its view, box = 16 bytes x
    // `rows` window rows = one K panel of a tile.  Stacked jobs see the windows as one tall 2-D image (a tile may run on
    // into the next frame), the others as [frame][row][byte] (rows past the window are zero-filled by the TMA unit).
    CUtensorMap tmap[6];
    Screen2JobDev job[6];
    int njobs;
    int B;
    const uint8_t *win[2];
    int win_h[2], win_pitch[2];
    int64_t win_stride[2];
    uint8_t *tailbin[2];
    int tail_pitch;
    int64_t tailbin_stride[2];
    int whatif;   // timing experiments only (LM_WHATIF_S2): 1 = no TMA loads after the ring's first fill, 2 = epilogue stops after draining TMEM,
                  // 4 = epilogue emits no tasks,
                  // 8 = accumulators released unread, 16 = the MMA warp does not wait for window tiles, 64 = print the jobs,
                  // 128 = print per-pair MMA-loop cycles; results of runs with bits 1-16 are meaningless
};

__device__ long long g_s2_dbg[3 * 80];   // LM_WHATIF_S2 & 128: per pair {cycles before the MMA loop, cycles in it, units}

__global__ void __cluster_dims__(2, 1, 1) __maxnreg__(96) k_screen2(const __grid_constant__ Screen2Params P) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t bars[2 * S2_STAGES + 4];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(8) uint64_t sbar[S2_RING];   // "unit of iteration it published", one per ring slot, in each CTA
    __shared__ int unit_ring[S2_RING];

    const long long dbg_t0 = clock64();
    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1;
    int ji = 0;
    for (int q = 1; q < P.njobs; ++q)
        if (pair >= P.job[q].pair_begin) ji = q;
    const Screen2JobDev &J = P.job[ji];
    const int prank = pair - J.pair_begin;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int KH = J.j.KH, ks = J.j.ks, rows = J.j.rows, nhalf = J.j.nhalf, nst = J.j.stages;
    const int npanel = 2 * ks;
    const uint32_t panel_a = (uint32_t)rows * 16u;
    const uint32_t stage_bytes = panel_a * npanel;
    const uint32_t chunk_b = (uint32_t)nhalf * 16u;
    const uint32_t b_bytes = (uint32_t)KH * npanel * chunk_b;
    uint8_t *sB = smem;
    uint8_t *sA = smem + b_bytes;
    const int nunits = J.ntp * J.nxt;
    const int VH = J.VH;

    const uint32_t bar0 = smem_u32(bars);
    auto a_full = [&](int s) { return bar0 + 8u * s; };                       // leader's copy is used
    auto a_empty = [&](int s) { return bar0 + 8u * (S2_STAGES + s); };        // local, multicast commit
    auto d_full = [&](int a) { return bar0 + 8u * (2 * S2_STAGES + a); };     // local, multicast commit
    auto d_empty = [&](int a) { return bar0 + 8u * (2 * S2_STAGES + 2 + a); };  // leader's copy is used

    // ---- one-time setup ---------------------------------------------------------------------------------------
    {
        const int4 *src = reinterpret_cast<const int4 *>(J.j.Bimg[rank]);
        int4 *dst = reinterpret_cast<int4 *>(sB);
        for (uint32_t i = tid; i < b_bytes / 16; i += S2_THREADS) dst[i] = __ldg(src + i);
    }
    if (tid == 0) {
        for (int s = 0; s < S2_STAGES; ++s) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a_full(s)), "r"(2));     // one arrive.expect_tx per CTA; the TMA units add the bytes
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a_empty(s)), "r"(1));
        }
        for (int a = 0; a < 2; ++a) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(d_full(a)), "r"(1));
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(d_empty(a)), "r"(8));    // one arrival per epilogue warp of the group that drains it, x 2 CTAs
        }
        for (int q = 0; q < S2_RING; ++q) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&sbar[q])), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == S2_WARP_MMA) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(S2_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();  // both CTAs' barriers are initialised and both B halves are in place
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    // Units (256-row tile pair x 32-column x tile) are dealt dynamically: a pair's first unit is its rank in the job, the others are
    // claimed from the job's counter by the leader CTA's producer warp, which publishes the index of iteration `it` in slot
    // it % S2_RING of both CTAs' rings (-1: no more work).  A pair whose SMs were still busy with another kernel when the launch
    // began simply claims fewer units; every role reads the ring after waiting for the slot's barrier.
    auto unit_of = [&](int it) -> int {
        mbar_wait_cluster(smem_u32(&sbar[it & (S2_RING - 1)]), (uint32_t)(it / S2_RING) & 1u);
        return *reinterpret_cast<volatile int *>(&unit_ring[it & (S2_RING - 1)]);
    };
    if (warp == S2_WARP_TMA) {
        // ================= TMA producer (both CTAs): this CTA's y tile of the unit ================================
        const CUtensorMap *tm = &P.tmap[ji];
        const bool stacked = J.j.stacked != 0;
        int stage = 0;
        uint32_t phase = 0;
        int u_claim = prank;   // leader: the unit of the coming iteration (lane 0 holds the claimed value)
        for (int it = 0;; ++it) {
            int u;
            if (rank == 0) {
                u = __shfl_sync(0xffffffffu, u_claim, 0);
                if (u >= nunits) u = -1;
                if (lane == 0) {
                    const uint32_t slot = (uint32_t)it & (S2_RING - 1);
                    unit_ring[slot] = u;
                    st_shared_cluster_u32(mapa_u32(smem_u32(&unit_ring[slot]), 1), (uint32_t)u);
                    mbar_arrive_cluster(smem_u32(&sbar[slot]), 0);
                    mbar_arrive_cluster(smem_u32(&sbar[slot]), 1);
                    if (u >= 0) u_claim = J.npair + atomicAdd(J.next_unit, 1);   // in flight while the ring stage is awaited below
                }
            } else {
                u = unit_of(it);
            }
            if (u < 0) break;
            const int tp = u / J.nxt, xt = u - tp * J.nxt;
            const int R0 = (2 * tp + (int)rank) * S2_TILE_M, x0 = xt * S2_TILE_X;  // first tile row in tile-row space
            mbar_wait(a_empty(stage), phase ^ 1u);
            if (elect_one()) {
                const uint32_t full = mapa_u32(a_full(stage), 0);  // the leader's barrier counts both CTAs' bytes
                const bool skip_load = (P.whatif & 1) && it >= nst;
                mbar_arrive_expect_tx_cluster(full, skip_load ? 0u : stage_bytes);
                const uint32_t dst = smem_u32(sA) + (uint32_t)stage * stage_bytes;
                if (skip_load) {
                } else if (stacked) {
                    for (int p = 0; p < npanel; ++p) tma_load_2d_pair(dst + (uint32_t)p * panel_a, tm, full, x0 + 16 * p, R0);
                } else {
                    const int f0 = R0 / VH, yf0 = R0 - f0 * VH;
                    for (int p = 0; p < npanel; ++p) tma_load_3d_pair(dst + (uint32_t)p * panel_a, tm, full, x0 + 16 * p, yf0, f0);
                }
            }
            __syncwarp();
            if (++stage == nst) {
                stage = 0;
                phase ^= 1u;
            }
        }
    } else if (warp == S2_WARP_MMA) {
        // ================= MMA issuer (leader CTA only) =============================================================
        if (rank == 0) {
            // u8 x s8 -> s32, K-major operands, M = 256 across the pair; N = 2 * nhalf, or 2 * nhalf_narrow right of the tail box
            const uint32_t idesc_base = (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(256 >> 4) << 24);
            const uint32_t idesc_wide = idesc_base | ((uint32_t)((2 * nhalf) >> 3) << 17);
            const uint32_t idesc_narrow = idesc_base | ((uint32_t)((2 * J.j.nhalf_narrow) >> 3) << 17);
            const uint64_t bdesc0 = umma_desc(smem_u32(sB), chunk_b);
            const uint32_t a_step = (2u * panel_a) >> 4, b_step = (2u * chunk_b) >> 4;
            const uint32_t b_row = ((uint32_t)npanel * chunk_b) >> 4;
            int stage = 0, acc = 0;
            uint32_t phase = 0, accphase = 0;
            const long long dbg_t1 = clock64();
            int dbg_units = 0;
            for (int it = 0;; ++it) {
                const int u = unit_of(it);
                if (u < 0) break;
                ++dbg_units;
                const int xt = u % J.nxt;
                const uint32_t idesc = (xt * S2_TILE_X >= J.j.narrow_x0) ? idesc_narrow : idesc_wide;
                mbar_wait(d_empty(acc), accphase ^ 1u);
                if (!(P.whatif & 16) || it < nst) mbar_wait(a_full(stage), phase);   // 16: window tiles not waited for
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (elect_one()) {
                    const uint32_t d = tmem + (uint32_t)acc * (uint32_t)S2_ACC_STRIDE;
                    const uint64_t adesc = umma_desc(smem_u32(sA) + (uint32_t)stage * stage_bytes, panel_a);
                    const uint32_t alo = (uint32_t)adesc, ahi = (uint32_t)(adesc >> 32), blo = (uint32_t)bdesc0, bhi = (uint32_t)(bdesc0 >> 32);
                    if (ks == 2 && KH % 6 == 0) {
                        umma_issue_tile<2, 6>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else if (ks == 2 && KH % 5 == 0) {
                        umma_issue_tile<2, 5>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else if (ks == 2 && KH % 4 == 0) {
                        umma_issue_tile<2, 4>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else if (ks == 3 && KH % 4 == 0) {
                        umma_issue_tile<3, 4>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else if (ks == 3 && KH % 3 == 0) {
                        umma_issue_tile<3, 3>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else if (ks == 1 && KH % 8 == 0) {
                        umma_issue_tile<1, 8>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else if (ks == 2) {
                        umma_issue_tile<2, 1>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else if (ks == 3) {
                        umma_issue_tile<3, 1>(d, alo, ahi, blo, bhi, a_step, b_step, b_row, idesc, KH);
                    } else {
                        uint32_t a_j = alo, b_j = blo, accum = 0;
                        for (int j = 0; j < KH; ++j) {
                            uint32_t a = a_j, b = b_j;
                            for (int k = 0; k < ks; ++k) {
                                umma_i8_2cta_lohi(d, a, ahi, b, bhi, idesc, accum);
                                accum = 1;
                                a += a_step;
                                b += b_step;
                            }
                            a_j += 1;  // next kernel row: 16 bytes further down the same tile (in both CTAs)
                            b_j += b_row;
                        }
                    }
                    umma_commit_2cta(a_empty(stage));
                    umma_commit_2cta(d_full(acc));
                }
                __syncwarp();
                if (++stage == nst) {
                    stage = 0;
                    phase ^= 1u;
                }
                if (++acc == 2) {
                    acc = 0;
                    accphase ^= 1u;
                }
            }
            if ((P.whatif & 128) && lane == 0) {
                g_s2_dbg[3 * pair] = dbg_t1 - dbg_t0;
                g_s2_dbg[3 * pair + 1] = clock64() - dbg_t1;
                g_s2_dbg[3 * pair + 2] = dbg_units;
            }
        }
    } else {
        // ================= epilogue (both CTAs): this CTA's 128 rows x N columns ===================================
        const int v = J.j.view;
        const int pitch = P.win_pitch[v];
        const int grp = warp >> 2, quad = warp & 3;
        const int row_in_tile = quad * 32 + lane;
        bool any_point = false;   // paw / snout slots consult the centre pixel
        for (int t = 0; t < J.j.ntmpl; ++t) any_point |= J.j.feat[t] != LM_TAIL;
        for (int it = 0;; ++it) {
            const int u = unit_of(it);
            if (u < 0) break;
            if ((it & 1) != grp) continue;
            const int acc = grp;
            const uint32_t accphase = (uint32_t)(it >> 1) & 1u;
            const int tp = u / J.nxt, xt = u - tp * J.nxt;
            const int R = (2 * tp + (int)rank) * S2_TILE_M + row_in_tile, x0 = xt * S2_TILE_X;
            const int f = R / VH, y = R - f * VH;   // VH % 4 == 0: the two rows of a patch share f and y >> 1
            const int nar = x0 >= J.j.narrow_x0 ? 1 : 0;
            const int nt = nar ? J.j.ntmpl_narrow : J.j.ntmpl;
            const bool rowok = f < P.B && y < J.out_h;
            // centre pixels of this row's 32 outputs (class.cpp:849, 864: candidates need a centre pixel > 25), fetched before
            // the wait so that their latency is hidden: nine aligned words, bit c of cmask = pixel c > 25
            uint32_t cw[9];
            uint32_t csh = 0;
            if (any_point) {
                const uint8_t *crow = P.win[v] + (int64_t)f * P.win_stride[v] + (int64_t)(y + J.halo_y) * pitch + x0 + J.halo_x;
                const uint32_t *cbase = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(crow) & ~(uintptr_t)3);
                csh = (uint32_t)(reinterpret_cast<uintptr_t>(crow) & 3u) * 8u;
#pragma unroll
                for (int q = 0; q < 9; ++q) cw[q] = rowok ? __ldg(cbase + q) : 0u;
            }
            mbar_wait(d_full(acc), accphase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (P.whatif & 8) {   // accumulator released unread
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(d_empty(acc), 0);
                continue;
            }
            const uint32_t ta = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)acc * (uint32_t)S2_ACC_STRIDE;
            uint32_t need_t[3] = {0u, 0u, 0u}, sign_t[3] = {0u, 0u, 0u};
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                if (t >= nt) break;
                // two halves of 16 columns: 32 live accumulator registers instead of 64, so that the CTA leaves room in the
                // register file for the other kernels' CTAs on this SM
                const int q_need = J.q_need[t], q_sign = J.q_sign[t];
                const bool is_tail = J.j.feat[t] == LM_TAIL;   // warp-uniform: only the tail consumes the "provably positive" map
                uint32_t need = 0, sign = 0;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    uint32_t hi[16], lo[16];
                    tmem_ld16(ta + (uint32_t)(J.j.col_hi[nar][t] + 16 * h), hi);
                    tmem_ld16(ta + (uint32_t)(J.j.col_lo[nar][t] + 16 * h), lo);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    if (is_tail) {
#pragma unroll
                        for (int c = 0; c < 16; ++c) {
                            const int H = (int)hi[c] + ((int)lo[c] >> 8);
                            if (H >= q_need) need |= 1u << (16 * h + c);
                            if (H > q_sign) sign |= 1u << (16 * h + c);
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < 16; ++c) {
                            const int H = (int)hi[c] + ((int)lo[c] >> 8);
                            if (H >= q_need) need |= 1u << (16 * h + c);
                        }
                    }
                }
                const int wvalid = J.out_w[t] - x0;
                const uint32_t colmask = wvalid >= 32 ? 0xffffffffu : (wvalid <= 0 ? 0u : ((1u << wvalid) - 1u));
                need_t[t] = rowok ? (need & colmask) : 0u;
                sign_t[t] = sign;
            }
            // every lane's tcgen05.ld has completed (wait::ld above); one arrival per warp: 128 remote arrivals per unit on the
            // leader's barrier cost more than the unit's MMAs (the accumulator came back ~6 k cycles after its commit)
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(d_empty(acc), 0);  // the leader's barrier counts both CTAs' epilogues
            if (P.whatif & 2) continue;
            uint32_t cmask = 0;
            if (any_point) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const uint32_t x = __funnelshift_r(cw[q], cw[q + 1], csh);
                    const uint32_t gt = (((x & 0x7f7f7f7fu) + 0x66666666u) | x) & 0x80808080u;  // bit 7 of each byte: byte >= 26
                    cmask |= ((gt * 0x00204081u) >> 28) << (4 * q);
                }
            }
            // pass 1: final "undecided" masks, tail sign rows, per-lane task counts and their warp prefix sums
            uint32_t pf_t[3] = {0u, 0u, 0u};
            int cnt_t[3] = {0, 0, 0}, incl_t[3] = {0, 0, 0}, total_t[3] = {0, 0, 0};
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                if (t >= nt) break;
                uint32_t need = need_t[t];
                if (J.j.feat[t] == LM_TAIL) {
                    if (x0 >= J.out_w[t]) continue;  // warp-uniform: no tail columns in this x tile
                    if (rowok) {
                        const uint32_t sign0 = sign_t[t];
                        uint8_t *tb = P.tailbin[v] + (int64_t)f * P.tailbin_stride[v] + (int64_t)y * P.tail_pitch + x0;
                        uint32_t w[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const uint32_t nib = (sign0 >> (4 * q)) & 0xfu;
                            w[q] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
                        }
                        reinterpret_cast<uint4 *>(tb)[0] = make_uint4(w[0], w[1], w[2], w[3]);
                        reinterpret_cast<uint4 *>(tb)[1] = make_uint4(w[4], w[5], w[6], w[7]);
                    }
                    need &= ~sign_t[t];
                } else {
                    need &= cmask;
                }
                uint32_t pf = lm_nibble_any(need);   // 2x4 patches: bit q = columns 4q .. 4q+3, rows y and y ^ 1 combined below
                pf |= __shfl_xor_sync(0xffffffffu, pf, 1);
                const int cnt = ((lane & 1) == 0) ? __popc(pf) : 0;
                int incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int w2 = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += w2;
                }
                pf_t[t] = pf;
                cnt_t[t] = cnt;
                incl_t[t] = incl;
                total_t[t] = __shfl_sync(0xffffffffu, incl, 31);
            }
            // pass 2: one reservation per non-empty list, issued together (independent round trips to L2)
            int base_t[3] = {0, 0, 0};
            if (P.whatif & 4) continue;
            if (lane == 31) {
#pragma unroll
                for (int t = 0; t < 3; ++t)
                    if (t < nt && total_t[t]) base_t[t] = atomicAdd(J.j.ntasks[t], total_t[t]);
            }
            // pass 3: the task words
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                if (t >= nt) break;
                if (!total_t[t]) continue;   // warp-uniform
                const int base = __shfl_sync(0xffffffffu, base_t[t], 31);
                if (cnt_t[t]) {
                    int o = base + incl_t[t] - cnt_t[t];
                    const uint32_t head = ((uint32_t)f << 16) | ((uint32_t)(y >> 1) << 8);
                    uint32_t m = pf_t[t];
                    while (m) {
                        const int q = __ffs(m) - 1;
                        m &= m - 1;
                        if (o < J.j.task_cap[t]) J.j.tasks[t][o] = head | (uint32_t)((x0 >> 2) + q);
                        ++o;
                    }
                }
            }
        }
    }
    // ---- teardown: nobody may free TMEM (or exit, its barriers are remote targets) before the peer is done ----
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();
    if (warp == S2_WARP_MMA) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(S2_TMEM_COLS));
    }
}

}  // namespace

size_t lm_screen2_smem_bytes(int KH, int ks, int rows, int nhalf, int stages) {
    return (size_t)KH * 2 * ks * nhalf * 16 + (size_t)stages * 2 * ks * rows * 16;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static const EncodeTiledFn fn = [] {  // initialised once, also when several host threads launch at once
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            return reinterpret_cast<EncodeTiledFn>(p);
        return (EncodeTiledFn) nullptr;
    }();
    return fn;
}
// One K panel of a window tile = a box of 16 bytes x `rows` rows; out-of-range rows / columns / frames read as zero.
static bool encode_window_map(CUtensorMap *tm, const uint8_t *win, int pitch, int win_h, int64_t win_stride, int frames, int rows, bool stacked) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc || rows > 256 || (pitch & 15) || (win_stride & 15)) return false;
    const cuuint32_t estr[3] = {1, 1, 1};
    if (stacked) {  // frames are win_h rows apart (win_stride == pitch * win_h): one tall image
        const cuuint64_t dim[2] = {(cuuint64_t)pitch, (cuuint64_t)win_h * (cuuint64_t)frames};
        const cuuint64_t str[1] = {(cuuint64_t)pitch};
        const cuuint32_t box[2] = {16, (cuuint32_t)rows};
        return enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t *>(win), dim, str, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    }
    const cuuint64_t dim[3] = {(cuuint64_t)pitch, (cuuint64_t)win_h, (cuuint64_t)frames};
    const cuuint64_t str[2] = {(cuuint64_t)pitch, (cuuint64_t)win_stride};
    const cuuint32_t box[3] = {16, (cuuint32_t)rows, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t *>(win), dim, str, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Launches k_screen2 for the pair-level jobs; the caller has zeroed the task counters.
int lm_launch_screen2_kernel(const LmBatch &b, cudaStream_t s) {
    const int n_sm = lm_sm_count();
    const int npairs_total = n_sm / 2;
    Screen2Params P{};
    size_t smem = 0;
    double work[6], total = 0.0;
    long long macs = 0;
    auto icost = [](int N) { return std::max(43.0, N / 2.0); };  // cycles per pair instruction (tools/umma_pair_probe.cu: the tensor pipe's rate down to N = 64)
    for (int v = 0; v < 2; ++v)
        for (int q = 0; q < 3; ++q) {
            const LmScreen2Job &sj = b.scr.job2[v][q];
            if (!sj.Bimg[0]) continue;  // no tail box
            Screen2JobDev &J = P.job[P.njobs];
            J.j = sj;
            int ow = 0;
            for (int t = 0; t < sj.ntmpl; ++t) {
                J.out_w[t] = sj.feat[t] == LM_TAIL ? b.tail_w : b.view[v].box_w;
                ow = std::max(ow, J.out_w[t]);
            }
            J.out_h = b.view[v].box_h;
            J.next_unit = b.scr.ntasks + 8 + P.njobs;
            J.nxt = (ow + S2_TILE_X - 1) / S2_TILE_X;
            const int nytp = ((J.out_h + S2_TILE_M - 1) / S2_TILE_M + 1) / 2;
            J.VH = sj.stacked ? b.view[v].win_h : 2 * S2_TILE_M * nytp;
            J.ntp = (int)(((int64_t)b.B * J.VH + 2 * S2_TILE_M - 1) / (2 * S2_TILE_M));
            J.halo_x = b.view[v].halo_x;
            J.halo_y = b.view[v].halo_y;
            for (int t = 0; t < sj.ntmpl; ++t) {
                auto fdiv256 = [](long long x) { return x >= 0 ? x / 256 : -((-x + 255) / 256); };  // floor
                auto clampi = [](long long x) { return (int)std::max<long long>(INT_MIN + 1LL, std::min<long long>(INT_MAX - 1LL, x)); };
                J.q_need[t] = clampi(fdiv256(sj.t_lo[t]));
                J.q_sign[t] = clampi(fdiv256(sj.t_hi[t]));
            }
            int n_narrow = 0;
            for (int xt = 0; xt < J.nxt; ++xt) n_narrow += (xt * S2_TILE_X >= sj.narrow_x0);
            work[P.njobs] = (double)J.ntp * sj.KH * sj.ks * ((J.nxt - n_narrow) * icost(2 * sj.nhalf) + n_narrow * icost(2 * sj.nhalf_narrow));
            total += work[P.njobs];
            macs += (long long)J.ntp * sj.KH * sj.ks * 256LL * 32LL * ((long long)(J.nxt - n_narrow) * 2 * sj.nhalf + (long long)n_narrow * 2 * sj.nhalf_narrow);
            smem = std::max(smem, lm_screen2_smem_bytes(sj.KH, sj.ks, sj.rows, sj.nhalf, sj.stages));
            if (sj.stacked && b.view[v].win_stride != (int64_t)b.view[v].win_pitch * b.view[v].win_h) return -1;
            if (!encode_window_map(&P.tmap[P.njobs], b.win[v], b.view[v].win_pitch, b.view[v].win_h, b.view[v].win_stride, b.B, sj.rows, sj.stacked != 0))
                return -1;
            ++P.njobs;
        }
    if (!P.njobs) return 0;
    {
        int left = npairs_total, pr = 0;
        double wleft = total;
        for (int q = 0; q < P.njobs; ++q) {
            int n = (q == P.njobs - 1) ? left : (int)std::lround(left * work[q] / wleft);
            n = std::max(1, std::min(n, left - (P.njobs - 1 - q)));
            P.job[q].pair_begin = pr;
            P.job[q].npair = n;
            pr += n;
            left -= n;
            wleft -= work[q];
        }
    }
    P.B = b.B;
    for (int v = 0; v < 2; ++v) {
        P.win[v] = b.win[v];
        P.win_h[v] = b.view[v].win_h;
        P.win_pitch[v] = b.view[v].win_pitch;
        P.win_stride[v] = b.view[v].win_stride;
        P.tailbin[v] = b.tailbin[v];
        P.tailbin_stride[v] = (int64_t)b.bb_h[v] * b.tail_pitch;
    }
    P.tail_pitch = b.tail_pitch;
    {
        static const int whatif = getenv("LM_WHATIF_S2") ? atoi(getenv("LM_WHATIF_S2")) : 0;
        P.whatif = whatif;
    }
    static_assert(sizeof(Screen2Params) <= 4000, "kernel parameter space");
    static LmDevOnce once;
    if (auto setup = once.first()) {
        if (cudaFuncSetAttribute(k_screen2, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024) != cudaSuccess) return -1;
    }
    if (P.whatif & 64) {
        for (int q = 0; q < P.njobs; ++q) {
            const Screen2JobDev &J = P.job[q];
            fprintf(stderr, "k_screen2 job %d: view %d ntmpl %d KH %d ks %d rows %d nhalf %d nhalf_narrow %d narrow_x0 %d nxt %d ntp %d VH %d npair %d stages %d stacked %d smem %zu\n", q,
                    J.j.view, J.j.ntmpl, J.j.KH, J.j.ks, J.j.rows, J.j.nhalf, J.j.nhalf_narrow, J.j.narrow_x0, J.nxt, J.ntp, J.VH, J.npair, J.j.stages, J.j.stacked, smem);
        }
    }
    // int8 multiply-accumulates this launch issues to the tensor cores (all instructions: M = 256 x N x K = 32 each), for
    // bench.py's executed-work figure beside the algorithmic one
    if (b.screen_macs) *b.screen_macs = macs;
    const int pairs = P.job[P.njobs - 1].pair_begin + P.job[P.njobs - 1].npair;
    k_screen2<<<2 * pairs, S2_THREADS, smem, s>>>(P);
    if (P.whatif & 128) {
        long long h[3 * 80];
        cudaStreamSynchronize(s);
        cudaMemcpyFromSymbol(h, g_s2_dbg, sizeof(h));
        for (int q = 0; q < pairs; q += 6)
            fprintf(stderr, "k_screen2 pair %d: setup %lld cycles, MMA loop %lld cycles for %lld units = %.1f per MMA\n", q, h[3 * q], h[3 * q + 1], h[3 * q + 2],
                    (double)h[3 * q + 1] / (60.0 * (double)h[3 * q + 2]));
    }
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}
