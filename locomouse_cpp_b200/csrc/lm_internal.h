// lm_internal.h — shared declarations of the sm_100a kernels behind include/locomouse_b200.h.
// Data layout in HBM for one sub-batch of B frames (see DESIGN.md §3):
//   raw frames      u8  [B(+1 halo)][vid_rows][vid_cols]     (caller's device memory or staging)
//   minmax          i32 [B+1][2]            (255 - min, max) of sat(F - BKG); slot 0 = halo frame
//   lut             u8  [B+1][256]          normalize ∘ imadjust per frame
//   win[view]       u8  [B][win_h][win_pitch]   pre-processed crop + template halo, zero extended
//   tailbin[view]   u8  [B][box_h][tail_pitch]  tail score > 0
//   tailmask        u8  [B][bb_h_bottom][tail_pitch]  largest bottom region (TAIL_MASK) 0/1
//   cc scratch      i32 [B][3][max_h * tail_w]  labels / area / key
//   det lists       {u32 idx; f32 score} [B][2 feat][2 view][det_cap] + counts i32 [B][4]
//   results         same struct-of-arrays as lm_results, for B frames
#pragma once
#include <cstdlib>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "../../include/locomouse_b200.h"

#define LM_MAX_KW 64  // widest template row the correlation kernel is instantiated for

struct LmDet {
    uint32_t idx;  // y * box_w + x in the unpadded crop
    float score;
};

// geometry of one view's pre-processed window and of the three correlations run on it
struct LmView {
    int box_w, box_h;      // unpadded crop (bb_w x bb_h_*)
    int halo_x, halo_y;    // window origin = crop origin - halo  (max anchor over the view's templates)
    int win_w, win_h, win_pitch;
    int64_t win_stride;    // bytes per frame
};

struct LmTemplateDev {
    const float *w;  // device, row-major, row stride = kwp floats (zero padded), rows = kh
    int kh, kw, kwp;
    int ax, ay;      // anchor = (kw/2, kh/2)
    float init;      // float(-rho)
};

struct LmGeom {
    int spre_b_w, spre_b_h, spost_b_w, spost_b_h;
    int spre_s_w, spre_s_h, spost_s_w, spost_s_h;
    int pad_pre_cols, pad_pre_rows, pad_post_cols, pad_post_rows;
};

// Tensor-core screen (k_screen.cu): per (view, template) job, the int8 banded-Toeplitz B operand, the
// integer decision thresholds and the list of 4x8 output patches the exact kernel must re-evaluate.
struct LmScreenJob {
    const int8_t *Bimg;   // device, [kh][2*ks chunks][64 rows][16 B]   (N = 64: 32 columns x {hi, lo} digit)
    int kh, ks;           // kernel rows, K steps of 32 window bytes
    int dx, dy;           // window column / row of tap (0,0) for output (0,0): halo - anchor
    int rows;             // window rows staged per 128-row tile: 128 + kh - 1 + dy, rounded up to 8
    long long t_lo, t_hi; // V <= t_lo: score provably <= 0;  V > t_hi: score provably > 0
    uint32_t *tasks;      // device, [task_cap]: frame << 16 | patch_row << 8 | patch_col (2x4 patches)
    int task_cap;
};
// CTA-pair variant (k_screen2.cu).  A job decides up to three templates of one view with one resident B operand per
// CTA: B rows are 32-row "planes" (one weight digit of one template for the tile's 32 output columns); CTA rank r holds
// nhalf / 32 planes, and plane g of rank r lands in accumulator columns 32 * (r * nhalf / 32 + g).
//   paw + snout + tail (N = 192): rank 0 = [paw hi | paw lo | tail hi], rank 1 = [snout hi | snout lo | tail lo];
//                                 x tiles right of the tail box use only the first nhalf_narrow = 64 rows (N = 128)
//   paw + snout        (N = 128): rank 0 = [paw hi | paw lo], rank 1 = [snout hi | snout lo]
//   one template       (N = 64) : rank 0 = [hi], rank 1 = [lo]   (tail alone, or templates too large to share)
struct LmScreen2Job {
    const int8_t *Bimg[2];  // device, per CTA rank: [KH][2*ks chunks][nhalf rows][16 B]
    int view, ntmpl;
    int feat[3];            // LM_PAW / LM_SNOUT / LM_TAIL of template slot t
    int KH, ks, rows, nhalf, nhalf_narrow;
    int narrow_x0;          // x tiles starting at or right of this column run the narrow instruction (INT_MAX: never)
    int ntmpl_narrow;       // template slots decided by the narrow instruction (the leading ones)
    int col_hi[2][3], col_lo[2][3];  // accumulator column of the hi / lo plane of slot t, [0] wide, [1] narrow
    int stages;             // window-tile ring depth that fits next to the resident B operand (2..4)
    int stacked;            // 1: y tiles run over the frames of the sub-batch stacked at the window pitch
    long long t_lo[3], t_hi[3];   // per template decided by this job
    uint32_t *tasks[3];
    int task_cap[3];
    int *ntasks[3];
};
struct LmScreen {
    int enabled;          // 0: dense exact kernel, 1: k_screen (one CTA per tile), 2: k_screen2 (CTA pairs)
    LmScreenJob job[2][3];
    LmScreen2Job job2[2][3];  // [view][0 = paw + snout (+ tail) (or paw alone), 1 = tail, 2 = snout alone]; unused: Bimg[0] == null
    int *ntasks;          // device, [6] = [view][feat]
};

// everything a kernel needs to know about the current sub-batch
struct LmBatch {
    // inputs
    const uint8_t *frames;      // frame i (0..B-1) at frames + i*frame_bytes
    const uint8_t *prev;        // frame -1 (halo); may be null when first_index == 0
    int64_t frame_bytes;
    int B;
    int64_t first_index;        // CURRENT_FRAME of frame 0 of this sub-batch
    const uint8_t *bkg;
    const int32_t *calib;
    const int32_t *calib_flip;  // [n_rows][n_cols] calib with the mirror folded in (k_fold_calib); detection path only
    const uint8_t *bkg_warp;    // [n_rows][n_cols] bkg[calib_flip], 4-byte aligned, >= 8 bytes of padding behind it
    const uint8_t *run_mode;    // [n_rows][n_cols] 1 / 2: pixels c..c+3 come from four consecutive raw bytes (ascending / descending); 0: no run
    const uint32_t *bb_x, *bb_y_side, *bb_y_bottom;  // device, [B]
    // config
    int vid_rows, vid_cols, n_rows, n_cols;
    int bb_w, bb_h[2], tail_w, tail_pitch;
    int flip, imadjust, conn, n_tail_points, fma_mode;
    int cand_cap, det_cap, match_cap;
    unsigned char *nms_scratch;  // device, [2 B lists][lm_nms_scratch_bytes(det_cap)]: lists too long for the NMS kernels' shared memory
    int ovlp[2];                // (int)(w_bottom * (1 - T)) per feature (class.cpp:1047), host computed
    LmView view[2];
    LmTemplateDev tmpl[2][3];
    // scratch
    int32_t *minmax;            // [B+1][2]
    uint8_t *lut;               // [B+1][256]
    uint8_t *win[2];
    uint8_t *tailbin[2];
    uint8_t *tailmask;
    uint8_t *sidemask;
    int32_t *cc;                // [B][3][cc_stride]
    int64_t cc_stride;
    int32_t *cc_flag;           // [B] 1 = frame exceeded the run capacity of k_tail and takes k_tail_slow
    LmScreen scr;
    cudaEvent_t ev_screen_done; // recorded by lm_launch_screen between k_screen and k_corr_sparse (may be null)
    cudaStream_t screen_stream; // when set (with ev_screen_go and ev_screen_done): the screen kernel runs on this (high-priority) stream
    cudaEvent_t ev_screen_start;  // recorded on the screen's stream right before the kernel (device timeline)
    cudaEvent_t ev_screen_go;
    long long *screen_macs;     // host, may be null: receives the int8 MACs of the k_screen2 launch (the context's lm_get_info("screen_macs"))
    LmDet *det;                 // [B][2][2][det_cap]   index: ((f*2+feat)*2+view)
    int32_t *det_count;         // [B][2][2]
    // results (device mirrors of lm_results)
    int32_t *n_bottom, *n_side;
    lm_cand *bottom, *side;
    int32_t *match_n, *match_y;
    double *match_s;
    int32_t *tail;
    uint32_t *flags;
};

// launchers (each returns the number of kernels it launched)
int lm_launch_minmax(const LmBatch &b, cudaStream_t s);
int lm_launch_prep(const LmBatch &b, cudaStream_t s);
int lm_launch_fold_calib(const int32_t *calib, const uint8_t *bkg, int n_rows, int n_cols, int flip, int32_t *calib_flip, uint8_t *bkg_warp, uint8_t *run_mode,
                         cudaStream_t s);
int lm_launch_corr(const LmBatch &b, cudaStream_t s);
int lm_launch_tail(const LmBatch &b, cudaStream_t s);
int lm_launch_nms(const LmBatch &b, cudaStream_t s);
// bytes of nms_scratch per list: 8 + 8 + 4 bytes per entry (two key arrays, one link array), 16-byte aligned slices
__host__ __device__ inline size_t lm_nms_scratch_bytes(int det_cap) { return ((size_t)det_cap * 20 + 15) & ~(size_t)15; }
int lm_launch_pair(const LmBatch &b, cudaStream_t s);
// sums (may be null): [B][side_w] per-column counts of the thresholded side view
int lm_launch_bbox_tm_de(const LmBatch &b, const lm_bb_de_params &p, uint32_t *hist, uint8_t *pred, double *bb_x, int32_t *lims,
                         int32_t *sums, cudaStream_t s, uint8_t *diff = nullptr);

// pass 1 of the base class (k_bbox_base.cu)
int lm_launch_bbox_pred(const LmBatch &b, const lm_bb_de_params &p, uint32_t *hist, uint8_t *pred, cudaStream_t s, uint8_t *diff = nullptr);
// pass 1 of LocoMouse_TM (k_bbox_tm.cu); returns the number of launches, -1 on a launch error, -2 when the side view's bit
// image does not fit into shared memory.  sums (may be null): [B][side_w] CV_32S column sums of the filled image.
size_t lm_bbox_tm_bits_bytes(const lm_bb_tm_params &p, int B);
size_t lm_bbox_tm_slow_runs(const lm_bb_tm_params &p);
int lm_launch_bbox_tm(const LmBatch &b, const lm_bb_tm_params &p, const float *d_disk, uint32_t *hist, uint8_t *pred, uint32_t *bits_a,
                      uint32_t *bits_b, int *need_slow, unsigned char *g_runs, int g_slots, uint32_t *level_mask /* 512 words */, double *bb_x, int32_t *lims,
                      int32_t *sums, cudaStream_t s);
size_t lm_bbox_base_bits_bytes(int n_rows, int n_cols, int B);
size_t lm_bbox_base_slow_ints(const lm_bb_base_params &p);
constexpr int LM_BBOX_SLOW_SLOTS = 8;
// sums (may be null): [B][lm_bbox_base_sums(p)] = Row_side[side_w] | Row_bottom[bottom_w] | Col_side[side_h] | Col_bottom[bottom_h], 255 per
// pixel of each view's largest component
inline int lm_bbox_base_sums(const lm_bb_base_params &p) { return p.side_w + p.bottom_w + p.side_h + p.bottom_h; }
int lm_launch_bbox_base(const LmBatch &b, const lm_bb_base_params &p, uint32_t *bits, uint32_t *major, int32_t *cc, uint8_t *vmap, uint8_t *vmask,
                        int *need_slow, int32_t *lims, int32_t *sums, cudaStream_t s);

// cost builders (k_cost.cu); all pointers are device memory.  Pairwise: phase 0 = count + scan (fills jc, nnz, offs),
// phase 1 = fill (ir, pr)
int lm_launch_unary(const lm_cand *cand, const int32_t *ncand, int64_t n, int cand_cap, int feat, int bb_w, int bb_h,
                    const lm_location_prior *pri, int np, double *out, cudaStream_t s);
int lm_launch_pairwise(const lm_cand *cand, const int32_t *ncand, int64_t n, int cand_cap, int feat, const lm_pairwise_params &p,
                       int32_t *jc, int64_t *nnz, int64_t *offs, int32_t *ir, double *pr, int64_t cap, int phase, cudaStream_t s);

// tensor-core screen + sparse exact re-evaluation (k_screen.cu); returns kernels launched or -1
int lm_launch_screen(const LmBatch &b, cudaStream_t s);
// Host-side preparation of one screen job from the fp32 template: quantisation to two int8 digits, the
// Toeplitz operand image and the thresholds.  Returns false when the job cannot be screened (operand does
// not fit in shared memory, non-finite weights); `img` receives kh * ks * 2048 bytes.
struct LmScreenHost {
    int kh, ks, dx, dy, rows;
    long long t_lo, t_hi;
    double scale, eps;
};
bool lm_screen_build(const float *w, int kh, int kw, float init, int halo_x, int halo_y, int fma_mode,
                     LmScreenHost *out, std::vector<int8_t> *img);
size_t lm_screen_smem_bytes(int kh, int ks, int rows, int stages);
// CTA-pair variant: writes ONE plane (32 rows: one weight digit, 0 = hi / 1 = lo, of one template) of a rank's B image
// in the common geometry of its job (KH kernel-row steps, ks K steps, nplanes planes per rank; the template's own row
// offset dy folded in as leading zero rows).  `img` must hold KH * 2 * ks * nplanes * 512 bytes, zero initialised.
// Thresholds / scale / eps as lm_screen_build.
bool lm_screen_build_plane(const float *w, int kh, int kw, float init, int dx, int dy, int KH, int ks, int digit, int plane,
                           int nplanes, LmScreenHost *out, std::vector<int8_t> *img);
size_t lm_screen2_smem_bytes(int KH, int ks, int rows, int nhalf, int stages);
// thresholds / scale / eps of one template (no image); false for non-finite weights
bool lm_screen_quantize(const float *w, int kh, int kw, float init, LmScreenHost *out);
int lm_launch_screen2_kernel(const LmBatch &b, cudaStream_t s);
// timing experiments only (tools/whatif.py): bit mask from the environment variable LM_WHATIF_SKIP of stages NOT launched
// (1 minmax, 2 prep, 4 screen kernel, 8 sparse exact pass, 16 tail, 32 nms, 64 pairing); results are then meaningless
inline int lm_whatif_skip() {
    const char *e = getenv("LM_WHATIF_SKIP");
    return e ? atoi(e) : 0;
}

// PNG frame decode (k_png.cu).  Per-frame status codes of k_png_decode:
enum {
    LM_PNG_OK = 0, LM_PNG_HEADER, LM_PNG_TRUNCATED, LM_PNG_ZLIB, LM_PNG_BLOCK_TYPE, LM_PNG_CODES, LM_PNG_SYMBOL, LM_PNG_DISTANCE,
    LM_PNG_TOO_LONG, LM_PNG_TOO_SHORT, LM_PNG_STORED, LM_PNG_FILTER, LM_PNG_NO_IDAT, LM_PNG_NOT_RUN
};
constexpr int LM_PNG_HDR_BYTES = 33;  // signature + IHDR chunk
// Frame j of the launch is payload[offs[j] - base, offs[j + 1] - base); its filtered stream goes to scratch + j * slot, its
// pixels to out + j * rows * cols, its LM_PNG_* code to status[j].
int lm_launch_png_decode(const uint8_t *payload, const int64_t *offs, int64_t base, int n, int rows, int cols, uint8_t *scratch, int64_t slot,
                         uint8_t *out, int32_t *status, cudaStream_t s);
// hdr[j][LM_PNG_HDR_BYTES] = the first bytes of frame j, zero-padded
int lm_launch_png_headers(const uint8_t *payload, const int64_t *offs, int64_t base, int64_t n, uint8_t *hdr, cudaStream_t s);
const char *lm_png_status_text(int st);

// FFV1 frame decode (k_ffv1.cu, format in ffv1_format.h).  One (GOP, slice) chain: slice s of frames f0 .. f0 + nf - 1.
namespace ffv1 {
struct Record;
}
struct LmFfv1Chain {
    int64_t f0;
    int32_t nf, s;
};
constexpr int LM_FFV1_CHAINS_PER_CTA = 32;
size_t lm_ffv1_smem_tables();  // shared memory of the record's tables in k_ffv1_decode
// Slice f * S + s of frame f (payload[offs[f] - base, offs[f + 1] - base)) is located at payload + soff[.], slen[.] bytes;
// a broken footer chain sets status[.] = LM_FFV1_FOOTER for the whole frame.
int lm_launch_ffv1_locate(const uint8_t *payload, const int64_t *offs, int64_t base, int64_t n, int S, int ec, int64_t *soff, int32_t *slen,
                          int32_t *status, cudaStream_t s);
int lm_launch_ffv1_crc(const uint8_t *payload, const int64_t *soff, const int32_t *slen, int64_t ns, int32_t *status, cudaStream_t s);
// work: work_bytes per chain (global slots, or shared memory when work_in_smem)
int lm_launch_ffv1_decode(const ffv1::Record *rec, int ac, const uint8_t *initial, const uint8_t *payload, const int64_t *soff,
                          const int32_t *slen, int32_t *status, uint8_t *out, int rows, int cols, const LmFfv1Chain *chains, int nchains,
                          uint8_t *work, int64_t work_bytes, int work_in_smem, cudaStream_t s);

// Motion-JPEG frame decode (k_mjpeg.cu, format in mjpeg_format.h).  Frame j of the launch is payload[offs[j] - base,
// offs[j + 1] - base); its header goes to hdr + j * lm_mjpeg_header_bytes(), its coefficients to coef + j *
// mjpeg::max_blocks(rows, cols) * 64, its pixels to out + j * rows * cols, its LM_MJPEG_* code to status[j].  *dht0 holds the
// Huffman tables the call's frame 0 defines (written by the launch with first_piece set), which every frame must match.
// A CTA of the entropy kernel takes 8 frames (4 kB of lookahead tables each), so several CTAs share an SM.
constexpr int LM_MJPEG_FRAMES_PER_CTA = 8;
size_t lm_mjpeg_header_bytes();
int lm_launch_mjpeg_decode(const uint8_t *payload, const int64_t *offs, int64_t base, int n, int rows, int cols, uint8_t *hdr, int16_t *coef,
                           int32_t *status, int32_t *dht0, int first_piece, uint8_t *out, cudaStream_t s);

// MPEG-4 Part 2 decode (k_mpeg4.cu, format in mpeg4_format.h).  Frame j of a launch is payload[offs[j] - base, offs[j + 1] -
// base) with its VOP header at vop + j * lm_mpeg4_vop_bytes() and its LM_MPEG4_* code in status[j] (0 on entry: headers
// good); its macroblock records go to info + j * nmb * lm_mpeg4_info_bytes(), its coefficients to coef + j * nmb * 320, its
// prediction state to lines + j * lm_mpeg4_lines_bytes(cols), its pixels to out + j * rows * cols.  seg: nseg pairs (first
// frame, frames) of the launch's segments, each reconstructed in the planes 2 s, 2 s + 1 (lm_mpeg4_plane_bytes each); a
// segment that starts with a P-VOP predicts its first frame from `carry`.  Entropy CTAs take 8 frames and 44 kB of
// shared lookahead tables.  lm_launch_mpeg4_locate fills vop / status of n frames already on the device (need_vol: *vol is
// invalid and becomes frame 0's VOL).
constexpr int LM_MPEG4_FRAMES_PER_CTA = 8;
size_t lm_mpeg4_vol_bytes();
size_t lm_mpeg4_vop_bytes();
size_t lm_mpeg4_info_bytes();
int64_t lm_mpeg4_lines_bytes(int cols);
inline int64_t lm_mpeg4_plane_bytes(int rows, int cols) { return (int64_t)((cols + 15) / 16) * ((rows + 15) / 16) * 320; }
int lm_launch_mpeg4_locate(const uint8_t *payload, const int64_t *offs, int n, int rows, int cols, uint8_t *vol, int need_vol, uint8_t *vop,
                           int32_t *status, cudaStream_t s);
int lm_launch_mpeg4_decode(const uint8_t *payload, const int64_t *offs, int64_t base, int n, const uint8_t *vop, int rows, int cols, uint8_t *info,
                           int16_t *coef, uint8_t *lines, const int32_t *seg, int nseg, int seg_len, uint8_t *planes, const uint8_t *carry,
                           int32_t *status, uint8_t *out, cudaStream_t s);

// pick the padded kernel-row width the correlation kernel is instantiated for (>= kw), or -1
int lm_corr_kwp(int kw);
// dynamic shared memory the correlation kernel needs for a view/template (for capability checks)
size_t lm_corr_smem_bytes(const LmBatch &b, int view, int feat);

// Per-device one-time set-up of the launchers (function attributes are per device; a process may own several contexts, driven
// from several host threads).  `if (auto setup = once.first()) { ... }`: exactly one caller per current device gets an open gate
// and runs the block; a concurrent caller on the same device waits until that block has finished (it must not launch a kernel
// whose shared-memory attribute is not set yet), later callers pass at the cost of one atomic load.
struct LmDevOnce {
    std::atomic<bool> done[64] = {};
    std::mutex m;
    struct Gate {
        std::unique_lock<std::mutex> lock;
        std::atomic<bool> *flag = nullptr;
        Gate() = default;
        Gate(Gate &&o) noexcept : lock(std::move(o.lock)), flag(o.flag) { o.flag = nullptr; }
        explicit operator bool() const { return flag != nullptr; }
        ~Gate() {
            if (flag) flag->store(true, std::memory_order_release);
        }
    };
    Gate first(void) {
        int dev = 0;
        cudaGetDevice(&dev);
        dev &= 63;
        Gate g;
        if (done[dev].load(std::memory_order_acquire)) return g;
        g.lock = std::unique_lock<std::mutex>(m);
        if (!done[dev].load(std::memory_order_acquire)) g.flag = &done[dev];
        else g.lock.unlock();
        return g;
    }
};
// Raises a kernel's dynamic shared-memory limit to all the device allows one block.  The attribute belongs to the function on the
// device, shared by every context and host thread there: it is set once (under an LmDevOnce), never per call to a call-dependent
// value that another thread's launch could overwrite between its own set and launch.
template <class F>
inline cudaError_t lm_allow_max_dynamic_smem(F *kernel) {
    int dev = 0, optin = 0;
    cudaGetDevice(&dev);
    cudaError_t e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaFuncAttributes a{};
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, kernel);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)a.sharedSizeBytes);
}
// The SM's L1 / shared-memory split is a per-SM setting.  Hypothesis tested in round 2: a kernel that prefers another split than
// k_screen2's (the largest shared-memory carve-out) cannot join an SM the screen runs on.  Measured: it can (tools/
// coresidency_probe.cu; what decides is registers per SM sub-partition and the shared memory left), and asking every kernel of the
// pipeline for the screen's split changed nothing (0.900 vs 0.904 ms per sub-batch) while taking L1 away from k_prep's gathers.
// The preference is therefore OFF by default; LM_CARVEOUT=1 turns it on for what-if runs.
template <class F>
inline void lm_prefer_max_shared(F *kernel) {
    static const bool on = getenv("LM_CARVEOUT") && atoi(getenv("LM_CARVEOUT")) != 0;
    if (on) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}
inline int lm_sm_count() {
    int dev = 0, n = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
}

#define LM_CUDA_CHECK(x)                                                            \
    do {                                                                            \
        cudaError_t _e = (x);                                                       \
        if (_e != cudaSuccess) return lm_fail_cuda(_e, #x, __FILE__, __LINE__);     \
    } while (0)
