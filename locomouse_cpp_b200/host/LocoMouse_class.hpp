// LocoMouse_class.hpp — host-side C++ mirror of the reference's tracking-problem classes for the
// per-frame detection path (LocoMouse_Core/LocoMouse_class.hpp:170-350, LocoMouse_TM.hpp:45-47,
// LocoMouse_TM_DE.hpp:39-43).  Same class names, same public method names, same call sequence as
// the reference's main.cpp:43-91, same result members (CANDIDATES_*, CANDIDATES_MATCHED_VIEWS_*,
// TRACKS_TAIL, BB_*), same error convention (std::invalid_argument / std::runtime_error).
//
// What differs is WHERE the work happens: the per-frame methods do no pixel work.  The first
// readFrame() of a chunk sends the chunk's raw frames through lm_detect_batch (include/locomouse_b200.h)
// and the per-frame methods then move that frame's records from the batched result buffers into the
// reference's per-frame vectors, so a driver written against the reference's interface runs
// unmodified.  There is no CPU implementation behind these methods.
#pragma once
#include <cstdint>
#include <functional>
#include <future>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/locomouse_b200.h"
#include "Candidates.hpp"
#include "LocoMouse_ParseInputs.hpp"
#include "MyMat.hpp"
#include "lm_media.hpp"

// LocoMouse_Parameters (class.hpp:48-100): the subset that reaches the detection path, plus the
// inputs that replace the out-of-scope pass 1 (SURVEY §8f-1): per-frame box positions from a file.
// LocoMouse_LocationPrior (class.hpp:33-45, ctor class.cpp:3196-3202)
class LocoMouse_LocationPrior {
    double X = 0, Y = 0, MAX_DISTANCE = 1, MIN_X = 0, MAX_X = 1, MIN_Y = 0, MAX_Y = 1;

public:
    LocoMouse_LocationPrior() = default;
    LocoMouse_LocationPrior(double x, double y, double md, double minx, double maxx, double miny, double maxy);
    double max_distance() const { return MAX_DISTANCE; }
    lm_location_prior to_c() const { return lm_location_prior{X, Y, MAX_DISTANCE, MIN_X, MIN_Y, MAX_X - MIN_X, MAX_Y - MIN_Y}; }
};

// Page-locked host array (lm_host_alloc): frames upload at the full PCIe rate and result arrays receive their device ->
// host copies directly.  Falls back to nothing: lm_host_alloc failing is an error (std::runtime_error).
template <typename T>
class PinnedArray {
    T *p_ = nullptr;
    size_t n_ = 0, cap_ = 0;  // shrinking keeps the allocation (page-locking memory is slow)

public:
    PinnedArray() = default;
    PinnedArray(const PinnedArray &) = delete;
    PinnedArray &operator=(const PinnedArray &) = delete;
    ~PinnedArray() { lm_host_free(p_); }
    void resize(size_t n) {
        if (n <= cap_) {
            n_ = n;
            return;
        }
        lm_host_free(p_);
        p_ = nullptr;
        n_ = cap_ = 0;
        void *q = nullptr;
        if (lm_host_alloc(&q, n * sizeof(T)) != LM_OK) throw std::runtime_error("lm_host_alloc failed (page-locked host memory)");
        p_ = static_cast<T *>(q);
        n_ = cap_ = n;
    }
    T *data() { return p_; }
    const T *data() const { return p_; }
    size_t size() const { return n_; }
    size_t capacity() const { return cap_; }
    void swap(PinnedArray &o) {
        std::swap(p_, o.p_);
        std::swap(n_, o.n_);
        std::swap(cap_, o.cap_);
    }
    T &operator[](size_t i) { return p_[i]; }
    const T &operator[](size_t i) const { return p_[i]; }
    T *begin() { return p_; }
    T *end() { return p_ + n_; }
    const T *begin() const { return p_; }
    const T *end() const { return p_ + n_; }
};

// One video's index, background and the frames (or coded frame chunks) of one of its windows, as read from the files.  A
// video longer than one window (max_resident_bytes) is streamed: the window in `data` changes as pass 1 and the frame loop
// move through the video.  The page-locked buffer only grows, so a LocoMouse_Media reused across videos is a pool:
// locomouse_b200_batch reads each worker's next video (its index and first window) into one of two.
struct LocoMouse_Media {
    unsigned int n_frames = 0;
    int rows = 0, cols = 0;
    lmmedia::Codec codec = lmmedia::Codec::raw;
    lmmedia::Index index;               // where every frame lies in the file
    std::vector<int> windows;           // first frame of every window, then n_frames
    int window = 0;                     // the window in data / offsets
    PinnedArray<uint8_t> data;          // raw: channel 0 of the window's frames, [count][rows][cols]; coded: its frame chunks
    std::vector<int64_t> offsets;       // coded: frame first + i = data[offsets[i], offsets[i + 1])
    std::vector<uint8_t> extradata;     // FFV1: the configuration record; MPEG-4: the VOL
    std::vector<uint8_t> bkg;           // rows x cols
    // loadVideo + loadBackground (LocoMouse_class.cpp:367-417): the video's index and its first window (the whole video when
    // it fits in max_resident_bytes); throws std::runtime_error as the reference's constructor does
    void load(const std::string &video_file, const std::string &bkg_file, size_t max_resident_bytes, int batch_frames, bool decode_mjpeg = false,
              bool decode_mpeg4 = false);
    void read_window(int k, PinnedArray<uint8_t> &to, std::vector<int64_t> &to_offsets) const;
};

// Device memory that a compressed video is decoded into (grow-only, lm_device_alloc on the context that uses it).  Whoever
// owns it reuses it across videos: locomouse_b200_batch keeps one per worker.
struct LocoMouse_DeviceFrames {
    uint8_t *p = nullptr;
    size_t bytes = 0;
    bool reserve(lm_ctx *ctx, size_t need);  // false (lm_last_error(ctx) says why) when the device memory is not there
    void release(lm_ctx *ctx);
};

// What a video beyond LocoMouse_Media's window needs: the second window buffer that a reader thread fills while the device
// works on the first, the previous window's last frame (page-locked for raw video, device memory for decoded video) and the
// device memory a compressed window is decoded into.  Grow-only; locomouse_b200_batch keeps one per worker.
struct LocoMouse_WindowPool {
    PinnedArray<uint8_t> spare;
    std::vector<int64_t> spare_offsets;
    int spare_window = -1;
    PinnedArray<uint8_t> prev;
    LocoMouse_DeviceFrames decoded, prev_decoded;
    void release(lm_ctx *ctx) {
        decoded.release(ctx);
        prev_decoded.release(ctx);
    }
};

class LocoMouse_Parameters {
public:
    // host-tracker cost builders (class.hpp:59-68, 88; class.cpp:132-145): used by computeUnaryCostsBottom / computePairwiseCostsBottom
    int max_displacement_bottom = 15;
    int occlusion_grid_spacing_pixels_bottom = 20;
    double occlusion_grid_max_width = 0.75;
    double alpha_vel_bottom = 1E-1;
    double pairwise_occluded_cost = 1E-2;
    // side-view tracker (class.hpp:60-61, 67): bestSideViewMatch / pairwisePotential_SideView
    int max_displacement_side = 15;
    int occlusion_grid_spacing_pixels_side = 20;
    double alpha_vel_side = 100;
    int tracker_threads = 0;          // host threads for the independent match2nd problems (0: one per hardware thread;
                                      // locomouse_b200_batch: hardware threads / workers)
    int batch_workers_per_gpu = 2;    // locomouse_b200_batch: host threads (one lm_ctx each) per visible device
    std::vector<LocoMouse_LocationPrior> PRIOR_PAW, PRIOR_SNOUT;  // config key location_prior (5 x 7); empty: cost builders are skipped
    int conn_comp_connectivity = 8;
    int median_filter_size = 11;      // class.hpp:54-55: pass 1 of the base class
    int min_pixel_visible = 1;
    int pass1_integer_sums = 0;       // 0: firstLastOverT reads the CV_32S sums as floats, as the reference does; 1: as integers
    double side_bottom_min_overlap = 0.7;
    double tail_sub_bounding_box = 0.6;
    int use_provided_bb = 0;
    cv::Rect BB_USER_SIDE, BB_USER_BOTTOM;
    static constexpr unsigned int N_paws = 4, N_snout = 1, N_tail_points = 15;
    // TM / TM_DE (LocoMouse_TM.cpp:57-112)
    int bb_width = 400, bb_height_side = 150;
    // LocoMouse_TM_Parameters (LocoMouse_TM.cpp:44-113); -1: key absent from the configuration file
    int bw_threshold_bottom = -1, bw_threshold_side = -1, min_pixel_count = -1;
    int zero_col_pre = -1, zero_col_post = -1, zero_row_pre = -1, zero_row_post = -1;
    std::string disk_filter_file;   // default: diskfilter.yml beside the executable (LocoMouse_TM.cpp:6)
    int moving_average_window = 5;
    // B200 path
    std::string bounding_box_file;  // pass-1 output (BB_X_POS, BB_Y_SIDE_POS, BB_Y_BOTTOM_POS), see lm_files.hpp
    int device = 0;
    int batch_frames = 4096;        // frames per lm_detect_batch call
    // page-locked bytes of frames held at a time: a longer video is read, decoded and tracked in windows of this many bytes
    // (a multiple of batch_frames frames), each read on a reader thread while the device works on the one before
    int64_t max_resident_bytes = (int64_t)8 << 30;
    int decode_mjpeg = 0;  // 1: Motion-JPEG video is decoded (bit-exact with libavcodec's decoder, lm_decode_mjpeg), 0: refused
    int decode_mpeg4 = 0;  // 1: MPEG-4 Part 2 video is decoded (bit-exact with libavcodec's decoder, lm_decode_mpeg4), 0: refused
    int fma_mode = 1;
    int cand_cap = 64, det_cap = 8192, match_cap = 256;

    LocoMouse_Parameters() = default;
    explicit LocoMouse_Parameters(const std::string &config_file_name);  // throws std::invalid_argument
};

// LocoMouse_Feature / LocoMouse_Model (class.hpp:110-167): templates, biases, sizes, match boxes.
class LocoMouse_Feature {
    std::vector<float> W_B, W_S;
    cv::Size SIZE_B, SIZE_S;
    double RHO_B = 0, RHO_S = 0;
    cv::Rect MATCH_BOX_B, MATCH_BOX_S;

public:
    LocoMouse_Feature() = default;
    LocoMouse_Feature(std::vector<float> w_b, cv::Size size_b, double rho_b, std::vector<float> w_s, cv::Size size_s,
                      double rho_s);
    const std::vector<float> &w_b() const { return W_B; }
    const std::vector<float> &w_s() const { return W_S; }
    double rho_b() const { return RHO_B; }
    double rho_s() const { return RHO_S; }
    cv::Size size_bottom() const { return SIZE_B; }
    cv::Size size_side() const { return SIZE_S; }
    cv::Rect match_box_bottom() const { return MATCH_BOX_B; }  // class.cpp:2954-2969
    cv::Rect match_box_side() const { return MATCH_BOX_S; }
};

class LocoMouse_Model {
public:
    LocoMouse_Feature paw, snout, tail;
    LocoMouse_Model() = default;
    explicit LocoMouse_Model(const std::string &model_file_name);  // throws std::runtime_error
};

namespace cvyaml {
class Writer;
}
using cvyaml_writer = cvyaml::Writer;

class LocoMouse {
protected:
    LocoMouse_Parameters LM_PARAMS;
    std::string LM_CALL, CONFIG_FILE, VIDEO_FILE, BKG_FILE, MODEL_FILE, CALIBRATION_FILE, FLIP_CHAR, OUTPUT_PATH;
    std::string output_file;

    // The video and background (raw frames, or PNG- / FFV1-coded frame chunks decoded window by window into POOL->decoded,
    // device memory in the layout of raw frames), read by the constructor into OWN_MEDIA or handed in by the caller.  MEDIA
    // holds the current window; READER fills POOL->spare with the next one.
    std::unique_ptr<LocoMouse_Media> OWN_MEDIA;
    LocoMouse_Media *MEDIA = nullptr;
    std::unique_ptr<LocoMouse_WindowPool> OWN_POOL;
    LocoMouse_WindowPool *POOL = nullptr;
    std::future<void> READER;
    int DECODED_WINDOW = -1;           // the window in POOL->decoded
    int PREV_WINDOW = -1;              // the window whose last frame is in POOL->prev / prev_decoded
    int VID_ROWS = 0, VID_COLS = 0;
    std::vector<int32_t> CALIBRATION;  // ind_warp_mapping, N_ROWS x N_COLS
    bool IMAGE_FLIP = false;

    cv::Rect BB_SIDE_VIEW, BB_BOTTOM_VIEW;
    cv::Rect BB_BOTTOM_MOUSE, BB_SIDE_MOUSE;
    std::vector<unsigned int> BB_X_POS, BB_Y_SIDE_POS, BB_Y_BOTTOM_POS;

    unsigned int N_FRAMES = 0, N_ROWS = 0, N_COLS = 0;
    int CURRENT_FRAME = -1, METHOD = 0;

    LocoMouse_Model M;

    std::vector<std::vector<Candidate>> CANDIDATES_BOTTOM_PAW, CANDIDATES_BOTTOM_SNOUT;
    std::vector<std::vector<Candidate>> CANDIDATES_SIDE_PAW, CANDIDATES_SIDE_SNOUT;
    std::vector<std::vector<P22D>> CANDIDATES_MATCHED_VIEWS_PAW, CANDIDATES_MATCHED_VIEWS_SNOUT;
    std::vector<std::vector<int32_t>> TRACKS_TAIL;  // per frame 3 x N_tail_points (x, y, z), -1 = missing
    std::vector<MyMat> UNARY_BOTTOM_PAW, UNARY_BOTTOM_SNOUT;            // class.hpp: same names
    std::vector<MATSPARSE> PAIRWISE_BOTTOM_PAW, PAIRWISE_BOTTOM_SNOUT;
    std::string costs_file, tracks_file;
    // occlusion grids (class.hpp:238-246; filled by initializeFeatureLoop, class.cpp:726-759) and the tracker's results
    std::vector<cv::Point_<double>> ONG;
    cv::Size ONG_size;
    cv::Point_<double> ONG_BR_corner;
    std::vector<unsigned int> ONG_SIDE;
    unsigned int ONG_SIDE_LOWEST_POINT = 0;
    cv::Mat TRACK_INDEX_PAW_BOTTOM, TRACK_INDEX_SNOUT_BOTTOM, TRACK_INDEX_PAW_SIDE, TRACK_INDEX_SNOUT_SIDE;  // points x frames labels
    std::vector<cv::Mat> EXPORTED;    // the matrices exportResults wrote, in file order (tests)

    // ---- device side ------------------------------------------------------------------------------
    lm_ctx *CTX = nullptr;
    bool OWN_CTX = true;               // false: the caller's context, left alone by the destructor
    struct Batch;                      // result buffers of the chunk that contains CURRENT_FRAME
    std::unique_ptr<Batch> BATCH, SPARE;   // SPARE: the chunk before BATCH, whose page-locked arrays the next chunk reuses
    bool LOOP_READY = false;

    void initializePaths(const LocoMouse_ParseInputs &INPUT);
    void initializeInputs(LocoMouse_Media &media, LocoMouse_WindowPool *pool);  // calibration, model, side, sizes
    void loadCalibration();
    void loadFlip();
    void validateImageVideoSize();
    void check(int rc) const;          // lm_status -> exception
    void runChunk(unsigned int first_frame);
    void configureDevice();            // lm_configure + background + calibration for the current box sizes
    const uint8_t *frames(int &on_device) const;  // first frame of the current window: MEDIA's raw frames, or the decoded window
    // Makes window k current (read, and decoded for compressed video) and starts reading window `next` (-1: none) on READER
    void useWindow(int k, int next);
    // pass 1 window by window: run(first frame of the window, on device, its first frame index, its frame count)
    void pass1Windows(const std::function<void(const uint8_t *, int, unsigned int, unsigned int)> &run);
    int windowOf(unsigned int frame) const;
    const Batch &batchFor(int frame) const;
    virtual bool usesImadjust() const { return false; }  // LocoMouse_TM::readFrame applies imadjust(0, 0.6)
    // class.cpp:2221-2346, 2385-2482
    cv::Mat bestSideViewMatch(const cv::Mat &T, const std::vector<std::vector<P22D>> &candidates_bottom_side_matched,
                              const std::vector<unsigned int> &ONG_side, unsigned int lowest_point, unsigned int N_features);
    void exportPointTracks(cvyaml_writer &out, const cv::Mat &T_bottom, const cv::Mat &T_side,
                           const std::vector<std::vector<P22D>> &candidates_bottom_side_matched, const std::string &feature_name, unsigned int N_features);
    void exportTracks();
    void exportLineTracks(cvyaml_writer &out, const std::vector<std::vector<int32_t>> &Tracks, const std::string &track_name, int N_line_points);

public:
    explicit LocoMouse(LocoMouse_ParseInputs INPUTS);
    // For a driver of many videos (locomouse_b200_batch): the configuration already parsed (params), the video's index,
    // background and first window already read (media, which must outlive the object; its window changes as the video is
    // tracked), a context the object does not own (ctx, not destroyed with it) and the further window buffers (pool, kept by
    // the caller for the next video).  The paths in INPUTS name the calibration, model and output files as for the constructor
    // above; the results are the same.
    LocoMouse(LocoMouse_ParseInputs INPUTS, const LocoMouse_Parameters &params, LocoMouse_Media &media, lm_ctx *ctx,
              LocoMouse_WindowPool *pool);
    virtual ~LocoMouse();
    LocoMouse(const LocoMouse &) = delete;
    LocoMouse &operator=(const LocoMouse &) = delete;

    virtual void readFrame();
    virtual void getBoundingBox();
    virtual void computeBoundingBox();
    void initializeFeatureLoop();
    void cropBoundingBox();
    void detectTail();
    void detectBottomCandidates();
    void computeUnaryCostsBottom();
    void computePairwiseCostsBottom();
    void detectSideCandidates();
    void matchBottomSideCandidates();
    void storePreviousImage();
    void computeBottomTracks();
    void computeSideTracks();
    void exportResults();

    unsigned int N_frames() const { return N_FRAMES; }
    unsigned int windows() const { return (unsigned int)MEDIA->windows.size() - 1; }
    // page-locked bytes held for frames (both window buffers and the previous frame) plus device bytes of decoded frames
    size_t residentBytes() const;
    lm_ctx *context() const { return CTX; }

    // read access for the host stages that follow (cost builders, match2nd) and for tests
    const std::vector<std::vector<Candidate>> &candidatesBottomPaw() const { return CANDIDATES_BOTTOM_PAW; }
    const std::vector<std::vector<Candidate>> &candidatesBottomSnout() const { return CANDIDATES_BOTTOM_SNOUT; }
    const std::vector<std::vector<Candidate>> &candidatesSidePaw() const { return CANDIDATES_SIDE_PAW; }
    const std::vector<std::vector<Candidate>> &candidatesSideSnout() const { return CANDIDATES_SIDE_SNOUT; }
    const std::vector<std::vector<P22D>> &candidatesMatchedViewsPaw() const { return CANDIDATES_MATCHED_VIEWS_PAW; }
    const std::vector<std::vector<P22D>> &candidatesMatchedViewsSnout() const { return CANDIDATES_MATCHED_VIEWS_SNOUT; }
    const std::vector<std::vector<int32_t>> &tracksTail() const { return TRACKS_TAIL; }
    const std::vector<MyMat> &unaryBottomPaw() const { return UNARY_BOTTOM_PAW; }
    const std::vector<MyMat> &unaryBottomSnout() const { return UNARY_BOTTOM_SNOUT; }
    const std::vector<MATSPARSE> &pairwiseBottomPaw() const { return PAIRWISE_BOTTOM_PAW; }
    const std::vector<MATSPARSE> &pairwiseBottomSnout() const { return PAIRWISE_BOTTOM_SNOUT; }
    const cv::Mat &trackIndexPawBottom() const { return TRACK_INDEX_PAW_BOTTOM; }
    const cv::Mat &trackIndexSnoutBottom() const { return TRACK_INDEX_SNOUT_BOTTOM; }
    const cv::Mat &trackIndexPawSide() const { return TRACK_INDEX_PAW_SIDE; }
    const cv::Mat &trackIndexSnoutSide() const { return TRACK_INDEX_SNOUT_SIDE; }
    // LocoMouse_class.cpp:2073-2150 (see lm_track::side_view_transitions)
    static MATSPARSE pairwisePotential_SideView(const std::vector<unsigned int> &Zi, const std::vector<unsigned int> &Zip1, double grid_mapping,
                                                double grid_spacing, const std::vector<unsigned int> &ONGi, unsigned int Nong,
                                                double max_displacement_bottom, double alpha_vel_bottom, double pairwise_occluded_cost);
};

// LocoMouse_TM (LocoMouse_TM.hpp:45-47): imadjust in readFrame; box = bb_width x bb_height_side (side,
// anchored at row 164) and bb_width x bottom-view height (LocoMouse_TM.cpp:142-155).
class LocoMouse_TM : public LocoMouse {
protected:
    bool usesImadjust() const override { return true; }

public:
    explicit LocoMouse_TM(LocoMouse_ParseInputs INPUTS);
    LocoMouse_TM(LocoMouse_ParseInputs INPUTS, const LocoMouse_Parameters &params, LocoMouse_Media &media, lm_ctx *ctx,
                 LocoMouse_WindowPool *pool);
    void computeBoundingBox() override;

protected:
    std::vector<float> DISK_FILTER;   // diskfilter.yml "H" (LocoMouse_TM.cpp:4-14), row-major, DISK_SIZE x DISK_SIZE
    int DISK_SIZE = 0;
    std::string REF_PATH;
};

// LocoMouse_TM_DE (LocoMouse_TM_DE.hpp:39-43): same readFrame; 400-wide boxes over the full view heights
// (LocoMouse_TM_DE.cpp:38-51).
class LocoMouse_TM_DE : public LocoMouse_TM {
public:
    explicit LocoMouse_TM_DE(LocoMouse_ParseInputs INPUTS);
    LocoMouse_TM_DE(LocoMouse_ParseInputs INPUTS, const LocoMouse_Parameters &params, LocoMouse_Media &media, lm_ctx *ctx,
                    LocoMouse_WindowPool *pool);
    void computeBoundingBox() override;
};

// LocoMouse_Methods.cpp:3-26
std::unique_ptr<LocoMouse> LocoMouse_Initialize(LocoMouse_ParseInputs INPUT);
// the same choice of class for the constructor on loaded inputs and a caller's context (see LocoMouse above)
std::unique_ptr<LocoMouse> LocoMouse_Initialize(LocoMouse_ParseInputs INPUT, const LocoMouse_Parameters &params, LocoMouse_Media &media,
                                                lm_ctx *ctx, LocoMouse_WindowPool *pool);
