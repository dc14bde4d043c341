// k_pair.cu — bottom-to-side candidate pairing: one warp per (frame, feature).
//
// Replaces LocoMouse::matchBottomSideCandidates -> matchingWithVelocityConstraint -> xDist +
// matchViews + checkVelCriterion (LocoMouse_class.cpp:999-1267) and the P22D records it appends
// (Candidates/Candidates.cpp:40-156):
//   ovlp = (int)(w_bottom*(1-T)); D = |xb - xs|; boolD = D <= ovlp, then the reference's
//   normalize(boolD, 0, 1, MINMAX) which zeroes an all-equal matrix (SURVEY Q7); colsum/rowsum of
//   boolD; per bottom candidate the side candidates are visited in list order and accepted unless
//   (colsum > 1 & vel_check) and the two "moving" flags differ (Q8); accepted side candidates carry
//   score * (D * (-(1/ovlp)) + 1) (the cv::MatExpr evaluation order of 1 - D/ovlp, Q9).
// checkVelCriterion needs the previous frame inside the CURRENT frame's crop (class.cpp:1469-1470):
// current pixels come from the pre-processed window, previous ones are re-derived on the fly from
// the previous raw frame with that frame's own LUT (k_pre.cu), so no "previous canvas" is stored.
// The reference evaluates the moving flags lazily; they are pure functions, so evaluating each
// needed flag once up front gives identical results.
#include "lm_internal.h"

namespace {

constexpr int PAIR_WARPS = 4;

struct MatchBox {
    int tlx, tly, w, h;
};
// LocoMouse_Feature ctor (class.cpp:2954-2969); round(x/2) for non-negative ints = (x + 1) / 2
__device__ __forceinline__ MatchBox match_box(int tw, int th) {
    MatchBox m;
    m.w = (tw + 1) / 2;
    m.h = (th + 1) / 2;
    m.tlx = -(m.w / 2);
    m.tly = -(m.h / 2);
    return m;
}

// warp-cooperative checkVelCriterion: #( sat(cur - prev) > 25 ) >= template_area * alpha
__device__ bool check_vel(const LmBatch &b, int f, int view, int cx, int cy, const MatchBox &mb, int area,
                          double alpha, int lane) {
    const LmView &V = b.view[view];
    const uint8_t *W = b.win[view] + (int64_t)f * V.win_stride;
    const uint8_t *Fp = f > 0 ? b.frames + (int64_t)(f - 1) * b.frame_bytes : b.prev;
    const uint8_t *lutp = b.lut + f * 256;  // slot f == frame f-1
    const int x0 = (int)b.bb_x[f] - b.bb_w + 1;
    const int ypos = (int)(view == LM_BOTTOM ? b.bb_y_bottom[f] : b.bb_y_side[f]);
    const int y0 = ypos - V.box_h + 1;
    int cnt = 0;
    const int npx = mb.w * mb.h;
    for (int q = lane; q < npx; q += 32) {
        const int r = q / mb.w, c = q - r * mb.w;
        const int bx = cx + mb.tlx + c, by = cy + mb.tly + r;  // crop coordinates
        const int wc = bx + V.halo_x, wr = by + V.halo_y;
        int cur = 0;
        if (wc >= 0 && wc < V.win_w && wr >= 0 && wr < V.win_h) cur = W[(int64_t)wr * V.win_pitch + wc];
        const int xx = x0 + bx, yy = y0 + by;
        int prev = 0;
        if (xx >= 0 && xx < b.n_cols && yy >= 0 && yy < b.n_rows) {
            const int64_t at = (int64_t)yy * b.n_cols + xx;   // mirror folded into calib_flip / bkg_warp (k_fold_calib)
            int d = (int)Fp[b.calib_flip[at]] - (int)b.bkg_warp[at];
            prev = lutp[d < 0 ? 0 : d];
        }
        int diff = cur - prev;
        cnt += (diff > 25) ? 1 : 0;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    return (double)cnt >= __dmul_rn((double)area, alpha);
}

__global__ void __launch_bounds__(PAIR_WARPS * 32) k_pair(const __grid_constant__ LmBatch b) {
    extern __shared__ __align__(8) unsigned char raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int unit = blockIdx.x * PAIR_WARPS + warp;  // (frame, feature)
    if (unit >= b.B * 2) return;
    const int f = unit >> 1, feat = unit & 1;
    const int cap = b.cand_cap, mcap = b.match_cap;
    // per-warp shared arrays
    const size_t per_warp = (size_t)cap * (sizeof(double) + 6 * sizeof(int));
    unsigned char *base = raw + warp * per_warp;
    double *ss = reinterpret_cast<double *>(base);
    int *xb = reinterpret_cast<int *>(ss + cap);
    int *yb = xb + cap, *xs = yb + cap, *ys = xs + cap, *colsum = ys + cap, *mov = colsum + cap;
    // mov[j] bit0 = mov_t[j] (side), mov[i] bit1 = mov_b[i] (bottom)

    const int nb = b.n_bottom[unit], ns = b.n_side[unit];
    int32_t *mn = b.match_n + (int64_t)unit * cap;
    int32_t *my = b.match_y + (int64_t)unit * mcap;
    double *ms = b.match_s + (int64_t)unit * mcap;
    for (int i = lane; i < cap; i += 32) mn[i] = 0;
    for (int i = lane; i < mcap; i += 32) {
        my[i] = -1;
        ms[i] = -1.0;
    }
    if (nb == 0 || ns == 0) return;

    const lm_cand *cb = b.bottom + (int64_t)unit * cap, *cs = b.side + (int64_t)unit * cap;
    for (int i = lane; i < nb; i += 32) {
        xb[i] = cb[i].x;
        yb[i] = cb[i].y;
        mov[i] = 0;
    }
    for (int j = lane; j < ns; j += 32) {
        xs[j] = cs[j].x;
        ys[j] = cs[j].y;
        ss[j] = cs[j].s;
        if (j >= nb) mov[j] = 0;
    }
    __syncwarp();
    const LmTemplateDev &Tb = b.tmpl[LM_BOTTOM][feat], &Ts = b.tmpl[LM_SIDE][feat];
    const int ovlp = b.ovlp[feat];  // (int)(w_bottom * (1 - T)), class.cpp:1047
    // boolD min/max (normalize quirk)
    bool any_t = false, any_f = false;
    for (int q = lane; q < nb * ns; q += 32) {
        const int i = q / ns, j = q - i * ns;
        const bool t = abs(xb[i] - xs[j]) <= ovlp;
        any_t |= t;
        any_f |= !t;
    }
    const bool mixed = __any_sync(0xffffffffu, any_t) && __any_sync(0xffffffffu, any_f);
    if (!mixed) return;  // boolD normalised to all zeros -> every bottom candidate unmatched
    for (int j = lane; j < ns; j += 32) {
        int c = 0;
        for (int i = 0; i < nb; ++i) c += (abs(xb[i] - xs[j]) <= ovlp) ? 1 : 0;
        colsum[j] = c;
    }
    __syncwarp();
    const bool vel = (b.first_index + f) > 0;
    if (vel) {
        const MatchBox mbs = match_box(Ts.kw, Ts.kh), mbb = match_box(Tb.kw, Tb.kh);
        for (int j = 0; j < ns; ++j) {
            if (colsum[j] > 1) {
                bool mv = check_vel(b, f, LM_SIDE, xs[j], ys[j], mbs, Ts.kw * Ts.kh, 0.05, lane);
                if (lane == 0) mov[j] |= mv ? 1 : 0;
            }
        }
        for (int i = 0; i < nb; ++i) {
            bool need = false;
            for (int j = lane; j < ns; j += 32) need |= (colsum[j] > 1) && (abs(xb[i] - xs[j]) <= ovlp);
            if (__any_sync(0xffffffffu, need)) {
                bool mv = check_vel(b, f, LM_BOTTOM, xb[i], yb[i], mbb, Tb.kw * Tb.kh, 0.02, lane);
                if (lane == 0) mov[i] |= mv ? 2 : 0;
            }
        }
        __syncwarp();
    }
    const double alpha = -__ddiv_rn(1.0, (double)ovlp);
    int basei = 0;
    for (int i0 = 0; i0 < nb; i0 += 32) {
        const int i = i0 + lane;
        int cnt = 0;
        if (i < nb)
            for (int j = 0; j < ns; ++j) {
                if (abs(xb[i] - xs[j]) > ovlp) continue;
                bool match = true;
                if (colsum[j] > 1 && vel) match = ((mov[i] >> 1) & 1) == (mov[j] & 1);
                cnt += match ? 1 : 0;
            }
        int incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += v;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        int o = basei + incl - cnt;
        if (i < nb) {
            mn[i] = cnt;
            for (int j = 0; j < ns; ++j) {
                const int D = abs(xb[i] - xs[j]);
                if (D > ovlp) continue;
                bool match = true;
                if (colsum[j] > 1 && vel) match = ((mov[i] >> 1) & 1) == (mov[j] & 1);
                if (!match) continue;
                if (o < mcap) {
                    my[o] = ys[j];
                    ms[o] = __dmul_rn(ss[j], __dadd_rn(__dmul_rn((double)D, alpha), 1.0));
                }
                ++o;
            }
        }
        basei += total;
    }
    if (lane == 0 && basei > mcap) atomicOr(&b.flags[f], LM_FLAG_MATCH_OVERFLOW);
}

}  // namespace

int lm_launch_pair(const LmBatch &b, cudaStream_t s) {
    const size_t per_warp = (size_t)b.cand_cap * (sizeof(double) + 6 * sizeof(int));
    const int units = b.B * 2;
    static LmDevOnce once;  // cand_cap > 384 needs more than the default 48 kB of dynamic shared memory
    if (auto setup = once.first()) {
        if (cudaFuncSetAttribute(k_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024) != cudaSuccess) return -1;
        lm_prefer_max_shared(k_pair);
    }
    k_pair<<<(units + PAIR_WARPS - 1) / PAIR_WARPS, PAIR_WARPS * 32, per_warp * PAIR_WARPS, s>>>(b);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}
