/*
 * locomouse_b200.h — C ABI of the B200-native LocoMouse per-frame detection path.
 *
 * This is the drop-in boundary for the hot loop of the reference program
 * (reference main.cpp:54-82): every entry point below replaces one or more methods of the
 * reference's `LocoMouse` / `LocoMouse_TM` / `LocoMouse_TM_DE` classes for a *batch* of frames:
 *
 *   lm_set_model        <- LocoMouse_Model(file)            LocoMouse_class.cpp:3095-3162, 2941-2990
 *   lm_set_background   <- LocoMouse::loadBackground        LocoMouse_class.cpp:402-417
 *   lm_set_calibration  <- LocoMouse::loadCalibration       LocoMouse_class.cpp:419-463
 *   lm_detect_batch     <- readFrame + cropBoundingBox + detectTail + detectBottomCandidates +
 *                          detectSideCandidates + matchBottomSideCandidates + storePreviousImage
 *                          (LocoMouse_class.cpp:1273-1333, LocoMouse_TM.cpp:243-249,
 *                           1408-1478, 2541-2767, 771-870, 1610-1905, 999-1267, 1508-1513)
 *
 * Plain pointers and sizes only; no C++ or torch types. All functions return LM_OK (0) or a
 * negative lm_status; lm_last_error() gives the message. The host C++ mirror of the reference
 * classes (locomouse_cpp_b200/host) turns non-zero codes into std::runtime_error /
 * std::invalid_argument like reference main.cpp:94-101 expects.
 *
 * There is no CPU fallback: if no CUDA device is usable lm_create fails.
 */
#ifndef LOCOMOUSE_B200_H
#define LOCOMOUSE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LM_ABI_VERSION 5  /* 5: lm_bounding_box_tm, and (backward compatible additions) lm_decode_png, lm_decode_ffv1, lm_device_alloc / lm_device_free / lm_device_copy, lm_get_info("ms_decode"), lm_get_info("device_allocs"); 4: lm_bounding_box_base, lm_mouse_box_size; 2: lm_set_option, lm_get_info, lm_debug_nms, lm_bounding_box_tm_de, lm_moving_average; 3: lm_host_alloc / lm_host_free, lm_unary_costs / lm_pairwise_costs, options streams 1..4, screen_layout, screen_priority */

/* feature / view indices used in every [2] / [3] array below */
enum { LM_PAW = 0, LM_SNOUT = 1, LM_TAIL = 2 };
enum { LM_BOTTOM = 0, LM_SIDE = 1 };

typedef enum {
    LM_OK = 0,
    LM_ERR_INVALID = -1,   /* bad argument / configuration  (reference: std::invalid_argument) */
    LM_ERR_RUNTIME = -2,   /* CUDA failure, out of memory   (reference: std::runtime_error)    */
    LM_ERR_ROI = -3,       /* a frame's bounding box leaves the padded canvas
                              (reference: uncaught cv::Exception from Mat ROI, class.cpp:1433,1465) */
    LM_ERR_OVERFLOW = -4,  /* a fixed-capacity list overflowed; see lm_results.flags           */
    LM_ERR_STATE = -5      /* call order (model/background/calibration not set)                */
} lm_status;

/* per-frame flag bits in lm_results.flags */
#define LM_FLAG_DET_OVERFLOW   0x1u  /* > det_cap positive pixels in one (feature, view)        */
#define LM_FLAG_CAND_OVERFLOW  0x2u  /* > cand_cap candidates after NMS                         */
#define LM_FLAG_MATCH_OVERFLOW 0x4u  /* > match_cap side matches for one feature                */

/* One detector template = LocoMouse_Feature::w_b / w_s + rho (class.hpp:110-146).
 * w is row-major float32, rows x cols; the correlation anchor is (cols/2, rows/2)
 * as in cv::filter2D with anchor (-1,-1) (class.cpp:845,860,2575). */
typedef struct {
    const float *w;
    int32_t rows, cols;
    double rho;
} lm_template;

/* Everything the kernels need besides pixel data.  Field <- reference source:            */
typedef struct {
    int32_t vid_rows, vid_cols;  /* raw frame / background size      (class.cpp:494-500)   */
    int32_t n_rows, n_cols;      /* calibrated image = CALIBRATION size (class.cpp:489-490)*/
    int32_t bb_w;                /* BB_BOTTOM_MOUSE.width == BB_SIDE_MOUSE.width           */
    int32_t bb_h_bottom;         /* BB_BOTTOM_MOUSE.height                                 */
    int32_t bb_h_side;           /* BB_SIDE_MOUSE.height (TM: 150, TM_DE: side view height)*/
    int32_t tail_w;              /* (int)(bb_w * tail_sub_bounding_box)  (class.cpp:711)   */
    int32_t flip;                /* IMAGE_FLIP: side char 'L'            (class.cpp:465-484)*/
    int32_t imadjust;            /* 1: LocoMouse_TM::readFrame imadjust(0,0.6,0,1)         */
    int32_t conn;                /* conn_comp_connectivity 4|8           (class.hpp:53)    */
    int32_t n_tail_points;       /* N_tail_points = 15                   (class.hpp:86)    */
    double min_overlap;          /* side_bottom_min_overlap T            (class.hpp:56)    */
    int32_t fma_mode;            /* 1: acc=fma(w,px,acc)   0: acc=acc+w*px (two roundings, the
                                    OpenCV direct-path order; SURVEY Q1)                   */
    int32_t cand_cap;            /* capacity of every candidate list (default 64)          */
    int32_t det_cap;             /* capacity of every positive-pixel list (default 8192)   */
    int32_t match_cap;           /* capacity of the side-match pool per feature            */
} lm_config;

/* Candidate (Candidates.hpp:16-34): Point_<int> p; double s */
typedef struct {
    int32_t x, y;
    double s;
} lm_cand;

/* Host result buffers, caller-allocated, struct-of-arrays, n = number of frames in the call.
 * P22D (Candidates.hpp:63-105) for bottom candidate i of feature k in frame f is
 *   CB = bottom[f][k][i];  its side list = match_y/match_s[f][k][o .. o+match_n[f][k][i])
 *   with o = sum of match_n[f][k][0..i);  match_n == 0  <=>  the reference's sentinel
 *   yt[0] = st[0] = -1 ("no side match", Candidates.cpp:40-45,148-156).
 * number of P22D per frame/feature == n_bottom[f][k] (class.cpp:1154-1251). */
typedef struct {
    int64_t n_frames;
    int32_t cand_cap, match_cap, n_tail_points;
    int32_t *n_bottom;   /* [n][2]            CANDIDATES_BOTTOM_{PAW,SNOUT}[f].size()        */
    int32_t *n_side;     /* [n][2]            CANDIDATES_SIDE_{PAW,SNOUT}[f].size()          */
    lm_cand *bottom;     /* [n][2][cand_cap]                                                 */
    lm_cand *side;       /* [n][2][cand_cap]                                                 */
    int32_t *match_n;    /* [n][2][cand_cap]                                                 */
    int32_t *match_y;    /* [n][2][match_cap]                                                */
    double *match_s;     /* [n][2][match_cap]                                                */
    int32_t *tail;       /* [n][3][n_tail_points]   TRACKS_TAIL[f] (x, y, z; -1 = missing)   */
    uint32_t *flags;     /* [n]                                                              */
} lm_results;

typedef struct lm_ctx lm_ctx;

/* lifetime ------------------------------------------------------------------------------- *
 * Concurrency: different contexts may be used concurrently from different host threads, also on the same device; a context
 * waits only for its own streams (no call synchronises the whole device), and the library's per-device one-time set-up is
 * thread-safe.  One context is used by one thread at a time (it may move between threads between calls).
 * Re-configuration keeps the context's device allocations: lm_configure / lm_set_model / lm_set_option only mark the
 * scratch free, and the next call that needs scratch re-derives the layout from the new geometry and reuses every block
 * that is large enough; it allocates (and returns the blocks it no longer fits to the driver) only when the geometry grew. */
int lm_abi_version(void);
int lm_create(lm_ctx **out, int device);            /* binds a CUDA device, creates streams   */
int lm_destroy(lm_ctx *ctx);
const char *lm_last_error(const lm_ctx *ctx);       /* ctx may be NULL: last create error     */

/* per-video state ------------------------------------------------------------------------ */
int lm_configure(lm_ctx *ctx, const lm_config *cfg);
/* t[view][feature]: t[LM_BOTTOM][LM_PAW] ... t[LM_SIDE][LM_TAIL] */
int lm_set_model(lm_ctx *ctx, const lm_template t[2][3]);
int lm_set_background(lm_ctx *ctx, const uint8_t *bkg);          /* vid_rows*vid_cols u8     */
int lm_set_calibration(lm_ctx *ctx, const int32_t *ind_warp_mapping); /* n_rows*n_cols i32   */

/* geometry the reference derives in initializeFeatureLoop (class.cpp:655-721), for callers
 * that want to validate boxes themselves: pads[8] = spre_b.w, spre_b.h, spost_b.w, spost_b.h,
 * spre_s.w, spre_s.h, spost_s.w, spost_s.h ; canvas[4] = PAD_PRE_COLS, PAD_PRE_ROWS,
 * PAD_POST_COLS, PAD_POST_ROWS */
int lm_get_geometry(const lm_ctx *ctx, int32_t pads[8], int32_t canvas[4]);

/* frames --------------------------------------------------------------------------------- *
 * Frames are raw 8-bit grayscale (channel 0 of the decoded video frame, class.cpp:1293),
 * contiguous [n][vid_rows][vid_cols].
 *  - frames            : n frames, host memory (pinned or pageable) or device memory,
 *                        chosen by frames_on_device.
 *  - prev_frame        : raw frame that precedes frames[0] in the video, same memory space;
 *                        required when first_frame_index > 0 (it plays I_PREV_PAD,
 *                        class.cpp:1469-1470,1510), ignored (may be NULL) otherwise.
 *  - first_frame_index : CURRENT_FRAME of frames[0]; the velocity check is off for video
 *                        frame 0 (class.cpp:1009).
 *  - bb_x, bb_y_side, bb_y_bottom : BB_X_POS / BB_Y_SIDE_POS / BB_Y_BOTTOM_POS for these n
 *                        frames (bottom-right box corners in calibrated-image coordinates,
 *                        class.cpp:1411-1423,1457-1458), host memory.
 * Results are written to the caller's host buffers when the call returns. */
int lm_detect_batch(lm_ctx *ctx, const uint8_t *frames, int frames_on_device,
                    const uint8_t *prev_frame, int64_t n, int64_t first_frame_index,
                    const uint32_t *bb_x, const uint32_t *bb_y_side, const uint32_t *bb_y_bottom,
                    lm_results *out);

/* tuning knobs that never change results ------------------------------------------------------ *
 *  "screen"   2 (default) / 1: the six correlations run as an int8 tensor-core screen (tcgen05; 2 = CTA pairs with
 *             cta_group::2, 1 = one CTA per tile) followed by an exact FP32 re-evaluation of the undecided
 *             outputs; 0: dense exact FP32 kernel only.  All three produce bit-identical results (the screen
 *             only discards outputs proven <= 0).
 *  "subbatch" frames per internal sub-batch (default 1024; frames in host memory use half of it, and a video shorter than two sub-batches is cut in two).
 *  "streams"  n = 2 .. 8 (default 4): n consecutive sub-batches are in flight on n streams with separate scratch (about
 *             1 GB each at the default sub-batch), so the latency-bound kernels of some overlap the tensor-core kernel of
 *             another; 1: all kernels strictly serial (used when timing a single kernel with events).
 *  "screen_stages"  2 (default) .. 4: depth of the CTA-pair screen's window-tile ring; 2 leaves 27 kB of each SM's shared
 *             memory to co-resident CTAs of the other sub-batches' small kernels.
 *  "screen_layout"  bit 0: the tail template shares the paw + snout operand of the CTA-pair screen (N = 192),
 *             bit 1: y tiles stacked over the frames of a sub-batch (default 3; never changes results).
 *  "screen_priority"  1 (default): the tensor-core screen kernels run on a high-priority stream.
 *  "back_priority"  1: everything after the crop kernel of a sub-batch runs on a medium-priority stream of its slot (default 0;
 *             measured neutral: the pipeline is bound by aggregate SM work, not by kernel ordering).
 * lm_get_info: "screen_active" (2/1/0 after the first lm_detect_batch, -1 before), "subbatch", "ms_screen"
 *             (device ms of the tensor-core kernel alone in the last call; ms[2] of lm_last_timing = screen + exact pass),
 *             "screen_eps_<view><feat>" / "screen_scale_<view><feat>" (error bound / weight quantum), "screen_macs" (int8
 *             multiply-accumulates the last CTA-pair screen launch issued: executed work, beside the algorithmic count),
 *             "device_allocs" (cudaMalloc calls this context has made so far; each one waits for the whole device, so a context
 *             re-configured for a video of the same geometry makes none; the stream-ordered allocations of lm_bounding_box_base /
 *             _tm / _tm_de and of the cost builders are not counted). */
int lm_set_option(lm_ctx *ctx, const char *name, int64_t value);
int lm_get_info(const lm_ctx *ctx, const char *name, double *value);

/* pass 1 (SURVEY §8f-1) -------------------------------------------------------------------------- *
 * LocoMouse_TM_DE::computeBoundingBox / computeMouseBox_DE (LocoMouse_TM_DE.cpp:8-113): per frame, the base-class
 * readFrame (no imadjust(0, 0.6)), imadjust_default on the side view (LocoMouse_class.cpp:3244-3311), zeroed border
 * bands, threshold, column sums, firstLastOverT (LocoMouse_class.hpp:411-442) and
 *     bb_x = min(side_w - 1, last * width_margin).
 * The whole-video smoothing that follows (vecmovingaverage, LocoMouse_class.cpp:1559-1608) is sequential host work:
 * lm_moving_average below.  Defaults = LocoMouse_TM_DE.hpp:27-29 and LocoMouse_TM_DE.cpp:68-71. */
typedef struct {
    int32_t side_x, side_y, side_w, side_h;   /* BB_SIDE_VIEW (calibration file view_boxes row 0)             */
    int32_t zero_col_pre, zero_col_post;      /* columns [0, pre) and [post, n_cols) of the side view -> 0: 46, 760 */
    int32_t zero_row_pre, zero_row_post;      /* rows    [0, pre) and [post, side_h) -> 0: 100, 149               */
    double threshold;                         /* SIDE_THRESHOLD = 255 * 0.05                                        */
    int32_t min_count;                        /* MIN_PIXEL_COUNT = 10 (column sum >= min_count)                     */
    double width_margin;                      /* WIDTH_MARGIN = 1.1                                                 */
} lm_bb_de_params;

/* frames: n raw frames (host or device memory, as lm_detect_batch).  bb_x_raw[n] receives the per-frame, unsmoothed
 * box position (double, may be -width_margin when no column qualifies); lims[n][2] (optional, may be NULL) the
 * first / last qualifying columns (-1, -1 when none; the reference leaves last = 0 when exactly one column qualifies).
 * Needs lm_configure, lm_set_background and lm_set_calibration; the model is not used. */
int lm_bounding_box_tm_de(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, int64_t n,
                          const lm_bb_de_params *p, double *bb_x_raw, int32_t *lims);
/* vecmovingaverage (LocoMouse_class.cpp:1559-1608): central moving average, partial windows copied, (uint32_t) casts */
int lm_moving_average(const double *v, int64_t n, int32_t window, uint32_t *out);

/* Pass 1 of the base class: LocoMouse::computeBoundingBox / computeMouseBox / largestBWAreaObject
 * (LocoMouse_class.cpp:579-653, 921-997): per frame, the base-class readFrame; medianBlur(median_filter_size) of the
 * zero-padded image; threshold(> 2.55 -> 1); the largest connected component of the side view and of the bottom view;
 * column sums (Row_*) and row sums (Col_*) of those 0 / 255 images as CV_32S; firstLastOverT on each; and from the four
 * (first, last) pairs the six per-frame numbers
 *     box[f] = { bb_x, bb_y_bottom (+ BB_BOTTOM_VIEW.y), bb_y_side, bb_width, bb_height_bottom, bb_height_side }.
 * The whole-video post-processing (computeMouseBoxSize, vecmovingaverage) is sequential host work: lm_mouse_box_size,
 * lm_moving_average.
 * sums_as_float = 1 is the reference: firstLastOverT reads its argument through a float pointer (LocoMouse_class.hpp:417)
 * although these sums are 32-bit integers, so a sum s is compared as the float with s's bit pattern (a denormal): with
 * min_pixel_visible >= 1 no entry ever qualifies and every limit is -1; with 0 every entry does.  sums_as_float = 0 compares
 * the integer sums themselves (what the code evidently intends; LocoMouse_TM_DE reduces to CV_32F and is not affected). */
typedef struct {
    int32_t side_x, side_y, side_w, side_h;         /* BB_SIDE_VIEW   (calibration file view_boxes row 0)               */
    int32_t bottom_x, bottom_y, bottom_w, bottom_h; /* BB_BOTTOM_VIEW (row 1)                                            */
    int32_t median_filter_size;                     /* odd; LocoMouse_class.hpp:54: 11                                   */
    int32_t min_pixel_visible;                      /* LocoMouse_class.hpp:55: 1                                         */
    int32_t sums_as_float;                          /* 1: as the reference (see above), 0: integer sums                   */
    int32_t reserved;
} lm_bb_base_params;
/* box: [n][6] doubles; lims (optional, may be NULL): [n][4][2] = (first, last) of Row_side, Row_bottom, Col_side, Col_bottom.
 * Needs lm_configure (its conn_comp_connectivity is used), lm_set_background and lm_set_calibration. */
int lm_bounding_box_base(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, int64_t n, const lm_bb_base_params *p,
                         double *box, int32_t *lims);
/* computeMouseBoxSize (LocoMouse_class.cpp:1481-1506) with medianvec / stdvec (1515-1556): size[3] = final width, bottom
 * height, side height = min(median + 3 std, max) per series.  The three arrays are sorted in place, as the reference's are. */
int lm_mouse_box_size(double *bb_w, double *bb_hb, double *bb_hs, int64_t n, int32_t size[3]);

/* Pass 1 of LocoMouse_TM: LocoMouse_TM::computeBoundingBox / computeMouseBox_DD / bwAreaOpen / imfill
 * (LocoMouse_TM.cpp:115-269): per frame, the base-class readFrame; on the side view imadjust_default
 * (LocoMouse_class.cpp:3244-3311); the four border bands set to zero; threshold(> bw_threshold_side -> 1); bwAreaOpen
 * (connected components of conn_comp_connectivity with fewer than min_pixel_count pixels removed); filter2D with the
 * DISK_FILTER matrix (8-bit result, anchor at the centre, BORDER_REPLICATE; float accumulation over the taps in row-major
 * order, rounded half to even -- OpenCV's direct path, which it uses for kernels of fewer than 130 taps; larger kernels go
 * through its DFT path, whose rounding at exact .5 ties is build-dependent); imfill (every pixel that a 4-connected flood
 * fill from pixel (0, 0) does not reach becomes 255); the CV_32S column sums; firstLastOverT with min_pixel_visible;
 * bb_x = the last qualifying column.  BB_Y_BOTTOM_POS = N_ROWS - 1 and BB_Y_SIDE_POS = 164 are constants of the method
 * (LocoMouse_TM.cpp:141-142); the moving average over the video is lm_moving_average.
 * sums_as_float: as for lm_bb_base_params -- 1 is the reference (firstLastOverT reads the integer sums through a float
 * pointer: with min_pixel_visible >= 1 nothing ever qualifies and bb_x = -1 for every frame; with 0 everything does and
 * bb_x = side_w - 1), 0 compares the integer sums themselves (the evident intent).
 * The reference requires BB_SIDE_VIEW to span the image width (colRange(ZERO_COL_POST, N_COLS) on the side view,
 * LocoMouse_TM.cpp:205): side_w != n_cols, zero_col_pre > zero_col_post-style inverted ranges and bands beyond the view are
 * rejected with LM_ERR_INVALID where OpenCV would throw. */
typedef struct {
    int32_t side_x, side_y, side_w, side_h;   /* BB_SIDE_VIEW                                                        */
    int32_t side_threshold;                   /* bw_threshold_side (SIDE_THRESHOLD, 0..255)                          */
    int32_t min_pixel_count;                  /* min_pixel_count (MIN_PIXEL_COUNT >= 1): bwAreaOpen                  */
    int32_t min_pixel_visible;                /* LM_PARAMS.min_pixel_visible: firstLastOverT threshold               */
    int32_t zero_col_pre, zero_col_post;      /* columns [0, pre) and [post, n_cols) of the side view are zeroed     */
    int32_t zero_row_pre, zero_row_post;      /* rows [0, pre) and [post, side_h)                                    */
    int32_t sums_as_float;                    /* 1: as the reference (see above), 0: integer sums                    */
    int32_t disk_size;                        /* DISK_FILTER is disk_size x disk_size (diskfilter.yml "H")           */
    int32_t reserved;
    const float *disk;                        /* host memory, row-major                                              */
} lm_bb_tm_params;
/* bb_x_raw[n]: per-frame, unsmoothed box position; lims (optional, may be NULL): [n][2] first / last qualifying column.
 * Needs lm_configure (its conn_comp_connectivity is used), lm_set_background and lm_set_calibration. */
int lm_bounding_box_tm(lm_ctx *ctx, const uint8_t *frames, int frames_on_device, int64_t n, const lm_bb_tm_params *p,
                       double *bb_x_raw, int32_t *lims);

/* cost builders of the host tracker (SURVEY §8f-2) --------------------------------------------------------------- *
 * LocoMouse::computeUnaryCostsBottom / unaryCostBox (LocoMouse_class.cpp:873-894, 1909-1952) and
 * computePairwiseCostsBottom / pairwisePotential (896-919, 1954-2070) + MATSPARSE(const MyMat*) (MyMat.cpp:141-178), for
 * ALL frames of a result set at once.  They feed match2nd, which stays on the host. */
typedef struct {              /* LocoMouse_LocationPrior (LocoMouse_class.hpp:33-45, .cpp:3196-3202)                    */
    double pos_x, pos_y;      /* POSITION, in box-normalised coordinates                                               */
    double max_distance;      /* MAX_DISTANCE                                                                          */
    double area_x, area_y, area_w, area_h; /* AREA = Rect_<double>(min_x, min_y, max_x - min_x, max_y - min_y)       */
} lm_location_prior;
typedef struct {
    double grid_x, grid_y;    /* ONG_BR_corner (LocoMouse_class.cpp:733)                                               */
    double grid_spacing;      /* occlusion_grid_spacing_pixels_bottom                                                  */
    int32_t ong_w, ong_h;     /* ONG_size (731); Nong = ong_w * ong_h occlusion-grid nodes                             */
    double max_displacement;  /* max_displacement_bottom                                                               */
    double alpha_vel;         /* alpha_vel_bottom                                                                      */
    double occluded_cost;     /* pairwise_occluded_cost                                                                */
} lm_pairwise_params;

/* UNARY_BOTTOM_{PAW,SNOUT}: for every frame f of `res` the MyMat unaryCostBox(CANDIDATES_BOTTOM_<feat>[f], BB, priors)
 * returns (N_candidates x n_priors, column-major, zeros where the candidate lies outside the prior's area or too far).
 * out[(f * n_priors + j) * cand_cap + i] = M(i, j); rows i >= n_bottom[f][feat] are 0.  bb_w / bb_h = BB_BOTTOM_MOUSE size. */
int lm_unary_costs(lm_ctx *ctx, const lm_results *res, int64_t n, int32_t feat, int32_t bb_w, int32_t bb_h,
                   const lm_location_prior *priors, int32_t n_priors, double *out);
/* PAIRWISE_BOTTOM_{PAW,SNOUT}: for every frame f >= 1 the MATSPARSE (MATLAB-style CSC) of
 * pairwisePotential(C[f-1], C[f], ...): (N_f + Nong) rows x (N_{f-1} + Nong) columns.
 *   jc[f * (cand_cap + Nong + 1) + c], c = 0 .. ncols: column starts relative to offs[f] (frame 0: all zero, no matrix);
 *   ir / pr [offs[f] + k]: row index / value of the k-th stored entry; entries equal to 0 are not stored, as in the
 *   reference; offs has n + 1 entries, offs[n] = total number of stored entries.  cap = capacity of ir / pr in entries; LM_ERR_OVERFLOW (with
 *   *total set to the required capacity) when it is too small. */
int lm_pairwise_costs(lm_ctx *ctx, const lm_results *res, int64_t n, int32_t feat, const lm_pairwise_params *p,
                      int64_t *offs, int32_t *jc, int32_t *ir, double *pr, int64_t cap, int64_t *total);

/* Page-locked host memory for frames and result arrays (optional).  When EVERY array of the lm_results passed to
 * lm_detect_batch lies in page-locked memory (from lm_host_alloc, cudaHostAlloc or cudaHostRegister), results are
 * copied device -> caller directly; otherwise they go through the library's pinned staging and one host memcpy per
 * sub-batch.  Frames in page-locked memory upload at full PCIe rate.  (The reference keeps results in std::vector
 * members of LocoMouse, LocoMouse_class.hpp:188-236; a binding backs those with this memory or accepts the copy.) */
int lm_host_alloc(void **ptr, size_t bytes);
int lm_host_free(void *ptr);

/* compressed video ------------------------------------------------------------------------------------------------------ *
 * PNG-coded AVI frames (fourcc 'MPNG' / 'png '): payload holds n complete PNG files, frame i = payload[offsets[i], offsets[i+1]),
 * offsets on the host; payload in host (pageable or page-locked) or device memory.  frames: device memory,
 * [n][vid_rows][vid_cols] of the configured geometry.  LM_ERR_INVALID names the first bad frame and why.
 * Each frame must be 8-bit grey, RGB or RGBA, not interlaced, of the configured size; the output is channel 0 of the frame
 * cv::VideoCapture delivers (grey, or blue), decoded on the device (inflate + the five row filters; checksums are not
 * verified).  Host payloads are copied in pieces on the copy stream, overlapped with the decode of the previous piece.
 * Needs lm_configure only.  lm_get_info("ms_decode"): device ms of the decode kernels in the last call. */
int lm_decode_png(lm_ctx *ctx, const uint8_t *payload, int payload_on_device, const int64_t *offsets, int64_t n, uint8_t *frames);
/* FFV1-coded AVI frames (fourcc 'FFV1', version 3 as libavcodec writes it): extradata is the configuration record (the AVI
 * 'strf' bytes after the BITMAPINFOHEADER), payload / offsets / frames as for lm_decode_png.  The record must be version 3,
 * 8 bits, grey (colorspace 0 without chroma planes) or RGB (colorspace 1, with or without alpha), coder_type 0, 1 or 2;
 * frame 0 must be a keyframe.  The output is channel 0 of the frame cv::VideoCapture delivers (grey, or blue), bit-exact.
 * Each (GOP, slice) decodes serially on the device; slice CRCs are checked first.  LM_ERR_INVALID names the record problem
 * or the first bad frame and slice.  Needs lm_configure only.  lm_get_info("ms_decode") covers it. */
int lm_decode_ffv1(lm_ctx *ctx, const uint8_t *extradata, int64_t extradata_len, const uint8_t *payload, int payload_on_device,
                   const int64_t *offsets, int64_t n, uint8_t *frames);
int lm_device_alloc(lm_ctx *ctx, void **ptr, size_t bytes);   /* on the context's device, for callers without a CUDA runtime */
int lm_device_free(lm_ctx *ctx, void *ptr);
/* Copies `bytes` between two device buffers of the context's device on its stream and returns when the copy is done (a
 * driver that streams decoded video keeps the last frame of one window as the previous frame of the next). */
int lm_device_copy(lm_ctx *ctx, void *dst, const void *src, size_t bytes);

/* measurement / debugging ---------------------------------------------------------------- */
/* Device time (ms, CUDA events on the library's own stream) of the stages of the last
 * lm_detect_batch call, summed over its sub-batches:
 * ms[0]=min/max  ms[1]=preprocess+crop  ms[2]=correlation  ms[3]=tail  ms[4]=nms  ms[5]=pairing
 * ms[6]=whole call on the device (event before the first copy/kernel to event after the last D2H,
 * so host<->device copies and inter-sub-batch gaps are included).  launches = kernels launched. */
int lm_last_timing(const lm_ctx *ctx, float ms[7], int64_t *launches);

/* Copies an intermediate of the LAST sub-batch back to the host for parity debugging.
 * what: 0 = pre-processed bottom window (u8), 1 = side window (u8), 2 = bottom tail mask (u8 0/255,
 * bb_h_bottom x tail_w), 3 = per-frame min/max (2 x int32). frame is relative to the last call.
 * Returns the number of bytes written or a negative lm_status. */
int64_t lm_debug_fetch(lm_ctx *ctx, int what, int64_t frame, void *dst, int64_t dst_bytes,
                       int32_t dims[4]);

/* Runs the candidate-extraction kernels of the configured geometry on a caller-supplied score map (host, float32,
 * [bb_h of the view][bb_w]): view == LM_BOTTOM -> nmsMax (LocoMouse_class.cpp:1610-1747), view == LM_SIDE ->
 * peakClustering (1749-1905); the suppression box is the template size of (view, feat), feat in {LM_PAW, LM_SNOUT};
 * no tail mask.  out receives cand_cap records; returns the number of candidates or a negative lm_status.  Used to
 * check the kernels directly against the reference's own code (tests/test_gpu_nms_reference.py). */
int lm_debug_nms(lm_ctx *ctx, int view, int feat, const float *scores, lm_cand *out);

#ifdef __cplusplus
}
#endif
#endif /* LOCOMOUSE_B200_H */
