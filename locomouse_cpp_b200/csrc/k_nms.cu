// k_nms.cu — candidate extraction from the positive-pixel lists: one CTA per (frame, feature).
//
//  k_nms_bottom = nmsMax          (LocoMouse_class.cpp:1610-1747) after detectPointCandidatesBottom's
//                                  tail masking (783, 849)
//  k_nms_side   = peakClustering  (LocoMouse_class.cpp:1749-1905), skipped when the feature's bottom
//                                  list is empty (820, 828)
//
// Keys: (~score_bits << 32) | (y << 16 | x).  Ascending key order == score descending, row-major pixel index ascending
// == the oracle's total order (SURVEY Q5); keys of one list are distinct.
// Overlap predicate inter/(2wh - inter) > 0.5  <=>  3*(w-|dx|)*(h-|dy|) > 2*w*h (exact in integers).  With h-|dy| <= h
// it implies |dx| < w/3, and likewise |dy| < h/3: with grid cells of at least ceil(w/3) x ceil(h/3) pixels, every
// overlapping pair lies in the same or an adjacent cell.  The front end therefore buckets each list by cell (counting
// sort in shared memory) instead of ranking it, and every overlap search reads 3 x 3 cells only.
//
// nmsMax's chain suppression (discarded detections keep suppressing, Q3) is equivalent to
//   parent(j) = the best-ranked i whose box overlaps j's by more than 0.5 (j itself included), root = parent chain end:
// j is discarded by the FIRST overlapping i met in rank order, discarded or not, and inherits that i's root.  Overlap is
// symmetric, so the parent is the neighbourhood's minimum key; roots need no global order.
// peakClustering is truly greedy: maxima are confirmed one at a time in rank order (the minimum free key), each
// confirmation claiming the free detections it overlaps in its 3 x 3 cells.
// Candidate slots are the roots / maxima in rank order.  Each cluster's sums are accumulated in double IN RANK ORDER, as
// the reference's loops do (1731-1739, 1865-1869), because double addition is not associative: the members are bucketed
// by slot and each bucket is merge-sorted by key.
#include "lm_internal.h"

namespace {

constexpr int NMS_T = 256;
constexpr int NMS_NWARPS = NMS_T / 32;
// Lists of up to NMS_SMEM_LIST entries keep their arrays in shared memory (20 B per entry); longer ones use this CTA's slice
// of the global scratch array.  With the cell / slot table the CTA stays below 20 kB, so it fits beside a resident k_screen2
// CTA of a neighbouring sub-batch.
constexpr int NMS_SMEM_LIST = 768;
constexpr int NMS_MAX_CELLS = 1024;  // cells are widened (by powers of two) until the grid has at most this many

__host__ __device__ __forceinline__ int nms_table_ints(int cand_cap) {
    return (cand_cap > NMS_MAX_CELLS ? cand_cap : NMS_MAX_CELLS) + 1;
}
__host__ __device__ __forceinline__ size_t nms_table_bytes(int cand_cap) { return ((size_t)nms_table_ints(cand_cap) * 4 + 15) & ~(size_t)15; }

// Per-list arrays (capacity C entries): key, a second key buffer (load order / root scratch / merge ping-pong), link.
struct NmsLists {
    unsigned long long *key;  // [C]  cell-major keys
    unsigned long long *buf;  // [C]  scratch; as ints [2C]
    int *link;                // [C]  parent / root / slot
    __device__ __forceinline__ int *bufi() const { return reinterpret_cast<int *>(buf); }
};

__device__ __forceinline__ NmsLists carve(unsigned char *base, int C) {
    NmsLists m;
    m.key = reinterpret_cast<unsigned long long *>(base);
    m.buf = m.key + C;
    m.link = reinterpret_cast<int *>(m.buf + C);
    return m;
}

struct NmsGrid {
    int cw, ch, gx, gy;
};

__device__ __forceinline__ NmsGrid make_grid(int w, int h, int bw, int bh) {
    NmsGrid g;
    g.cw = (w + 2) / 3;
    g.ch = (h + 2) / 3;
    for (;;) {
        g.gx = (bw + g.cw - 1) / g.cw;
        g.gy = (bh + g.ch - 1) / g.ch;
        if (g.gx * g.gy <= NMS_MAX_CELLS) return g;
        if (g.gx >= g.gy)
            g.cw *= 2;
        else
            g.ch *= 2;
    }
}

__device__ __forceinline__ int key_x(unsigned long long k) { return (int)(k & 0xffffu); }
__device__ __forceinline__ int key_y(unsigned long long k) { return (int)((k >> 16) & 0xffffu); }
__device__ __forceinline__ float key_score(unsigned long long k) { return __uint_as_float(~(unsigned)(k >> 32)); }

__device__ __forceinline__ bool overlaps(int dx, int dy, int w, int h, int wh2) {
    dx = dx < 0 ? -dx : dx;
    dy = dy < 0 ? -dy : dy;
    return dx < w && dy < h && 3 * (w - dx) * (h - dy) > wh2;
}

// In-place exclusive prefix sum of a[0, len) by the whole block; returns the total.  Ends with a barrier.
__device__ int block_exclusive_scan(int *a, int len) {
    __shared__ int warp_sum[NMS_NWARPS];
    __shared__ int total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (len + NMS_T - 1) / NMS_T, lo = min(tid * per, len), hi = min(lo + per, len);
    int s = 0;
    for (int i = lo; i < hi; ++i) s += a[i];
    int incl = s;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int v = lane < NMS_NWARPS ? warp_sum[lane] : 0;
        int x = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += u;
        }
        if (lane < NMS_NWARPS) warp_sum[lane] = x - v;
        if (lane == NMS_NWARPS - 1) total = x;
    }
    __syncthreads();
    int base = warp_sum[warp] + incl - s;
    for (int i = lo; i < hi; ++i) {
        const int t = a[i];
        a[i] = base;
        base += t;
    }
    __syncthreads();
    return total;
}

// Front end: loads the list, drops tail-masked pixels (bottom only: setTo(255, TAIL_MASK)) and stores the keys cell-major
// in m.key (counting sort: histogram, scan, scatter).  Afterwards cell_end[c] is the end of cell c's range (its start is
// cell_end[c - 1], 0 for c = 0).  Returns the number of detections n (<= det_cap); sets *overflow.
__device__ int load_bucketed(const LmBatch &b, int f, int feat, int view, const NmsGrid &g, const NmsLists &m, int *cell_end,
                             bool *overflow) {
    const int tid = threadIdx.x;
    const int list = (f * 2 + feat) * 2 + view;
    int cnt = b.det_count[list];
    *overflow = cnt > b.det_cap;
    if (cnt > b.det_cap) cnt = b.det_cap;
    const LmDet *d = b.det + (int64_t)list * b.det_cap;
    const int bw = b.bb_w, G = g.gx * g.gy;
    const uint8_t *tm = (view == LM_BOTTOM && b.tail_w > 0)
                            ? b.tailmask + (int64_t)f * b.bb_h[LM_BOTTOM] * b.tail_pitch
                            : nullptr;
    for (int c = tid; c < G; c += NMS_T) cell_end[c] = 0;
    __syncthreads();
    // keys in load order in buf; a tail-masked entry gets ~0, which no detection's key equals (its score word would be 0)
    for (int i = tid; i < cnt; i += NMS_T) {
        const LmDet e = d[i];
        const int y = e.idx / bw, x = e.idx - y * bw;
        unsigned long long k = ~0ull;
        if (!(tm && x < b.tail_w && tm[y * b.tail_pitch + x])) {
            k = ((unsigned long long)(~__float_as_uint(e.score)) << 32) | ((uint32_t)y << 16) | (uint32_t)x;
            atomicAdd(&cell_end[(y / g.ch) * g.gx + x / g.cw], 1);
        }
        m.buf[i] = k;
    }
    __syncthreads();
    const int n = block_exclusive_scan(cell_end, G);
    for (int i = tid; i < cnt; i += NMS_T) {
        const unsigned long long k = m.buf[i];
        if (k != ~0ull) m.key[atomicAdd(&cell_end[(key_y(k) / g.ch) * g.gx + key_x(k) / g.cw], 1)] = k;
    }
    __syncthreads();
    return n;
}

// Calls fn(i) for every entry i of the 3 x 3 cells around pixel (x, y).  A cell row's three cells are one contiguous range.
template <class F>
__device__ __forceinline__ void for_neighbourhood(const NmsGrid &g, const int *cell_end, int x, int y, int first, int step, F fn) {
    const int cx = x / g.cw, cy = y / g.ch;
    const int x0 = cx > 0 ? cx - 1 : 0, x1 = cx + 1 < g.gx ? cx + 1 : g.gx - 1;
    const int y0 = cy > 0 ? cy - 1 : 0, y1 = cy + 1 < g.gy ? cy + 1 : g.gy - 1;
    for (int r = y0; r <= y1; ++r) {
        const int c0 = r * g.gx + x0, c1 = r * g.gx + x1;
        const int lo = c0 > 0 ? cell_end[c0 - 1] : 0, hi = cell_end[c1];
        for (int i = lo + first; i < hi; i += step) fn(i);
    }
}

// Common back end.  On entry link[j] holds the cluster head (root / confirmed maximum) of detection j and bufi()[h] the
// candidate slot of head h; ncand = number of clusters.  Buckets the members of the first cand_cap clusters by slot, merge-
// sorts each bucket by key and writes one candidate per slot: the rank-ordered double sums, and the head's score.
template <bool HALF_EVEN>
__device__ void write_candidates(const NmsLists &m, int n, int ncw, int cap, int *slot_end, lm_cand *out) {
    const int tid = threadIdx.x;
    __shared__ int s_maxlen;
    for (int j = tid; j < n; j += NMS_T) m.link[j] = m.bufi()[m.link[j]];
    for (int k = tid; k < ncw; k += NMS_T) slot_end[k] = 0;
    if (tid == 0) s_maxlen = 0;
    __syncthreads();
    for (int j = tid; j < n; j += NMS_T)
        if (m.link[j] < ncw) atomicAdd(&slot_end[m.link[j]], 1);
    __syncthreads();
    for (int k = tid; k < ncw; k += NMS_T) atomicMax(&s_maxlen, slot_end[k]);
    const int total = block_exclusive_scan(slot_end, ncw);
    for (int j = tid; j < n; j += NMS_T)
        if (m.link[j] < ncw) m.buf[atomicAdd(&slot_end[m.link[j]], 1)] = m.key[j];
    __syncthreads();
    // Segmented merge sort of buf: in a pass with run length L, an element's place in the merged pair of runs is its index
    // in its own run plus the number of smaller keys in the partner run (keys are distinct).
    unsigned long long *src = m.buf, *dst = m.key;
    const int maxlen = s_maxlen;
    for (int L = 1; L < maxlen; L <<= 1) {
        for (int p = tid; p < total; p += NMS_T) {
            int lo = 0, hi = ncw - 1;  // slot of position p: first k with slot_end[k] > p
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (slot_end[mid] > p) hi = mid; else lo = mid + 1;
            }
            const int s0 = lo > 0 ? slot_end[lo - 1] : 0, e0 = slot_end[lo];
            const int q = p - s0, r = q / L;
            const int ps = s0 + (r ^ 1) * L;
            const unsigned long long k = src[p];
            if (ps >= e0) {
                dst[p] = k;
                continue;
            }
            int a = ps, z = min(ps + L, e0);  // number of partner keys < k: lower bound in [ps, pe)
            while (a < z) {
                const int mid = (a + z) >> 1;
                if (src[mid] < k) a = mid + 1; else z = mid;
            }
            dst[s0 + (r & ~1) * L + (q - r * L) + (a - ps)] = k;
        }
        __syncthreads();
        unsigned long long *t = src;
        src = dst;
        dst = t;
    }
    for (int k = tid; k < cap; k += NMS_T) {
        lm_cand c;
        c.x = -1;
        c.y = -1;
        c.s = -1.0;
        if (k < ncw) {
            const int s0 = k > 0 ? slot_end[k - 1] : 0, e0 = slot_end[k];
            double wx = 0.0, wy = 0.0, ss = 0.0;
            for (int i = s0; i < e0; ++i) {
                const unsigned long long q = src[i];
                const double s = (double)key_score(q);
                wx = __dadd_rn(wx, __dmul_rn((double)key_x(q), s));
                wy = __dadd_rn(wy, __dmul_rn((double)key_y(q), s));
                ss = __dadd_rn(ss, s);
            }
            const double qx = __ddiv_rn(wx, ss), qy = __ddiv_rn(wy, ss);
            if (HALF_EVEN) {
                c.x = __double2int_rn(qx);
                c.y = __double2int_rn(qy);
            } else {
                c.x = (int)round(qx);
                c.y = (int)round(qy);
            }
            c.s = (double)key_score(src[s0]);  // the head has the cluster's smallest key
        }
        out[k] = c;
    }
}

__device__ __forceinline__ NmsLists lists_for(const LmBatch &b, unsigned char *raw, int list) {
    int c = b.det_count[list];
    c = c > b.det_cap ? b.det_cap : c;
    return c <= NMS_SMEM_LIST ? carve(raw + nms_table_bytes(b.cand_cap), NMS_SMEM_LIST)
                              : carve(b.nms_scratch + (size_t)blockIdx.x * lm_nms_scratch_bytes(b.det_cap), b.det_cap);
}

__device__ __forceinline__ void set_flags(const LmBatch &b, int f, bool overflow, int nc) {
    unsigned fl = 0;
    if (overflow) fl |= LM_FLAG_DET_OVERFLOW;
    if (nc > b.cand_cap) fl |= LM_FLAG_CAND_OVERFLOW;
    if (fl) atomicOr(&b.flags[f], fl);
}

// ---- nmsMax ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NMS_T) k_nms_bottom(const __grid_constant__ LmBatch b) {
    extern __shared__ __align__(16) unsigned char raw[];
    int *table = reinterpret_cast<int *>(raw);  // cell ends, later slot ends
    __shared__ int s_nr;
    const int f = blockIdx.x >> 1, feat = blockIdx.x & 1, tid = threadIdx.x;
    const NmsLists m = lists_for(b, raw, (f * 2 + feat) * 2 + LM_BOTTOM);
    const LmTemplateDev &T = b.tmpl[LM_BOTTOM][feat];
    const int w = T.kw, h = T.kh, wh2 = 2 * w * h;
    const NmsGrid g = make_grid(w, h, b.bb_w, b.bb_h[LM_BOTTOM]);
    bool overflow;
    const int n = load_bucketed(b, f, feat, LM_BOTTOM, g, m, table, &overflow);
    if (tid == 0) s_nr = 0;
    // parent = the overlapping detection with the smallest key (j itself when none is better)
    for (int j = tid; j < n; j += NMS_T) {
        const unsigned long long kj = m.key[j];
        const int xj = key_x(kj), yj = key_y(kj);
        unsigned long long best = kj;
        int par = j;
        for_neighbourhood(g, table, xj, yj, 0, 1, [&](int i) {
            const unsigned long long ki = m.key[i];
            if (ki < best && overlaps(key_x(ki) - xj, key_y(ki) - yj, w, h, wh2)) {
                best = ki;
                par = i;
            }
        });
        m.link[j] = par;
    }
    __syncthreads();
    // roots by pointer chasing (parents have smaller keys, so chains end); the roots are listed in bufi()[n, 2n)
    int *root_of = m.bufi(), *roots = m.bufi() + n;
    for (int j = tid; j < n; j += NMS_T) {
        int r = j;
        while (m.link[r] != r) r = m.link[r];
        root_of[j] = r;
        if (r == j) roots[atomicAdd(&s_nr, 1)] = j;
    }
    __syncthreads();
    const int nr = s_nr;
    for (int j = tid; j < n; j += NMS_T) m.link[j] = root_of[j];
    __syncthreads();
    // candidate slot of a root = its rank among the roots (few per list), stored at bufi()[root]
    for (int t = tid; t < nr; t += NMS_T) {
        const int p = roots[t];
        const unsigned long long kp = m.key[p];
        int rank = 0;
        for (int u = 0; u < nr; ++u) rank += m.key[roots[u]] < kp;
        root_of[p] = rank;
    }
    __syncthreads();
    const int ncw = nr < b.cand_cap ? nr : b.cand_cap;
    write_candidates<true>(m, n, ncw, b.cand_cap, table, b.bottom + (int64_t)(f * 2 + feat) * b.cand_cap);
    if (tid == 0) {
        b.n_bottom[f * 2 + feat] = ncw;
        set_flags(b, f, overflow, nr);
    }
}

// ---- peakClustering ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(NMS_T) k_nms_side(const __grid_constant__ LmBatch b) {
    extern __shared__ __align__(16) unsigned char raw[];
    int *table = reinterpret_cast<int *>(raw);
    __shared__ int s_nc;
    const int f = blockIdx.x >> 1, feat = blockIdx.x & 1, tid = threadIdx.x;
    lm_cand *out = b.side + (int64_t)(f * 2 + feat) * b.cand_cap;
    if (b.n_bottom[f * 2 + feat] == 0) {  // Q6
        for (int k = tid; k < b.cand_cap; k += NMS_T) {
            lm_cand c;
            c.x = -1;
            c.y = -1;
            c.s = -1.0;
            out[k] = c;
        }
        if (tid == 0) b.n_side[f * 2 + feat] = 0;
        return;
    }
    const NmsLists m = lists_for(b, raw, (f * 2 + feat) * 2 + LM_SIDE);
    const LmTemplateDev &T = b.tmpl[LM_SIDE][feat];
    const int w = T.kw, h = T.kh, wh2 = 2 * w * h;
    const NmsGrid g = make_grid(w, h, b.bb_w, b.bb_h[LM_SIDE]);
    bool overflow;
    const int n = load_bucketed(b, f, feat, LM_SIDE, g, m, table, &overflow);
    for (int j = tid; j < n; j += NMS_T) m.link[j] = -1;  // -1 = free
    __syncthreads();
    // Greedy, by one warp (no block barriers): the next maximum is the free detection with the smallest key; it claims the
    // free detections of its 3 x 3 cells that it overlaps.  bufi()[c] = slot of maximum c.
    // Each lane owns the entries lane, lane + 32, ... and keeps the minimum of its free ones between confirmations: the free
    // set only shrinks, so that minimum stays valid until it is claimed.  Only then does the lane rescan, starting after the
    // claimed prefix of its entries.
    if (tid < 32) {
        const int lane = tid;
        int nc = 0, first = lane;
        unsigned long long mine = ~0ull;
        int mi = -1;
        for (;;) {
            if (mi < 0 || m.link[mi] >= 0) {
                while (first < n && m.link[first] >= 0) first += 32;
                mine = ~0ull;
                mi = -1;
                for (int j = first; j < n; j += 32)
                    if (m.link[j] < 0 && m.key[j] < mine) {
                        mine = m.key[j];
                        mi = j;
                    }
            }
            unsigned long long best = mine;
            int bi = mi;
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long ob = __shfl_xor_sync(0xffffffffu, best, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ob < best) {
                    best = ob;
                    bi = oi;
                }
            }
            if (bi < 0) break;
            const int xc = key_x(best), yc = key_y(best);
            for_neighbourhood(g, table, xc, yc, lane, 32, [&](int j) {
                if (m.link[j] < 0) {
                    const unsigned long long kq = m.key[j];
                    if (overlaps(key_x(kq) - xc, key_y(kq) - yc, w, h, wh2)) m.link[j] = bi;
                }
            });
            if (lane == 0) m.bufi()[bi] = nc;
            ++nc;
            __syncwarp();
        }
        if (lane == 0) s_nc = nc;
    }
    __syncthreads();
    const int nc = s_nc;
    const int ncw = nc < b.cand_cap ? nc : b.cand_cap;
    write_candidates<false>(m, n, ncw, b.cand_cap, table, out);
    if (tid == 0) {
        b.n_side[f * 2 + feat] = ncw;
        set_flags(b, f, overflow, nc);
    }
}

}  // namespace

int lm_launch_nms(const LmBatch &b, cudaStream_t s) {
    static LmDevOnce once;
    if (auto setup = once.first()) {
        lm_prefer_max_shared(k_nms_bottom);
        lm_prefer_max_shared(k_nms_side);
    }
    if (!b.nms_scratch) return -1;
    const size_t smem = nms_table_bytes(b.cand_cap) + (size_t)NMS_SMEM_LIST * 20;
    k_nms_bottom<<<b.B * 2, NMS_T, smem, s>>>(b);
    k_nms_side<<<b.B * 2, NMS_T, smem, s>>>(b);
    return 2;
}
