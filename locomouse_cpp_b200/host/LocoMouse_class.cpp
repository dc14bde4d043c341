// LocoMouse_class.cpp — host-side mirror of the reference's LocoMouse / LocoMouse_TM / LocoMouse_TM_DE
// for the per-frame detection path; see LocoMouse_class.hpp.  All pixel work happens behind the C ABI
// (include/locomouse_b200.h); nothing here computes scores, masks or candidates.
#include "LocoMouse_class.hpp"

#include <algorithm>
#include <cctype>
#include <cmath>
#include <fstream>
#include <iostream>
#include <sstream>
#include <stdexcept>

#include "cv_yaml.hpp"
#include "lm_files.hpp"
#include "lm_media.hpp"

// =====================================================================================================
// LocoMouse_ParseInputs (LocoMouse_ParseInputs.cpp:56-100)
// =====================================================================================================
LocoMouse_ParseInputs::LocoMouse_ParseInputs(int argc, char *argv[]) {
    if (argc != 9)
        // The reference falls back to sample files that are not shipped (LocoMouse_ParseInputs.cpp:62-84);
        // here a wrong argument list is an input error.
        throw std::invalid_argument(
            "Invalid input list. The input should be: LocoMouse method config.yml video background model_file "
            "calibration_file side_char output_folder.");
    LM_CALL = argv[0];
    METHOD = argv[1];
    CONFIG_FILE = argv[2];
    VIDEO_FILE = argv[3];
    BKG_FILE = argv[4];
    MODEL_FILE = argv[5];
    CALIBRATION_FILE = argv[6];
    FLIP_CHAR = argv[7];
    OUTPUT_PATH = argv[8];
    FILE_STEM = stripFileName(VIDEO_FILE);
    const size_t slash = LM_CALL.find_last_of("/\\");
    REF_PATH = slash == std::string::npos ? "./" : LM_CALL.substr(0, slash + 1);
}

std::string LocoMouse_ParseInputs::stripFileName(const std::string &s) {
    const size_t slash = s.find_last_of("/\\");
    std::string base = slash == std::string::npos ? s : s.substr(slash + 1);
    const size_t dot = base.find_last_of('.');
    return dot == std::string::npos ? base : base.substr(0, dot);
}

// =====================================================================================================
// LocoMouse_Parameters: "key: value" scalars and "[a, b, c, d]" boxes (the subset of config.yml that the
// detection path reads; range checks as LocoMouse_class.cpp:17-249 / LocoMouse_TM.cpp:57-112)
// =====================================================================================================
namespace {

std::string trim(const std::string &s) {
    size_t a = 0, b = s.size();
    while (a < b && std::isspace((unsigned char)s[a])) ++a;
    while (b > a && std::isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

std::vector<double> parse_list(const std::string &v, const std::string &key) {
    std::string t = trim(v);
    if (t.size() < 2 || t.front() != '[' || t.back() != ']') throw std::invalid_argument(key + " must be a [..] list.");
    std::stringstream ss(t.substr(1, t.size() - 2));
    std::vector<double> out;
    std::string item;
    while (std::getline(ss, item, ',')) out.push_back(std::stod(trim(item)));
    return out;
}

cv::Rect parse_rect(const std::string &v, const std::string &key) {
    std::vector<double> l = parse_list(v, key);
    if (l.size() != 4) throw std::invalid_argument(key + " must have 4 entries: [x, y, width, height].");
    return cv::Rect((int)l[0], (int)l[1], (int)l[2], (int)l[3]);
}

}  // namespace

LocoMouse_LocationPrior::LocoMouse_LocationPrior(double x, double y, double md, double minx, double maxx, double miny, double maxy)
    : X(x), Y(y), MAX_DISTANCE(md), MIN_X(minx), MAX_X(maxx), MIN_Y(miny), MAX_Y(maxy) {
    if (!(minx < maxx) || !(miny < maxy)) throw std::invalid_argument("location_prior: min must be below max.");  // CV_Assert, class.cpp:3197-3198
}

LocoMouse_Parameters::LocoMouse_Parameters(const std::string &config_file_name) {
    std::ifstream in(config_file_name);
    if (!in) throw std::invalid_argument("Could not open the configuration file: " + config_file_name);
    std::string line;
    while (std::getline(in, line)) {
        const size_t hash = line.find('#');
        if (hash != std::string::npos) line.erase(hash);
        if (line.rfind("%YAML", 0) == 0 || line.rfind("---", 0) == 0) continue;
        const size_t colon = line.find(':');
        if (colon == std::string::npos) continue;
        const std::string key = trim(line.substr(0, colon)), val = trim(line.substr(colon + 1));
        if (val.empty()) continue;
        try {
            if (key == "conn_comp_connectivity") conn_comp_connectivity = std::stoi(val);
            else if (key == "side_bottom_min_overlap") side_bottom_min_overlap = std::stod(val);
            else if (key == "median_filter_size") median_filter_size = std::stoi(val);
            else if (key == "min_pixel_visible") min_pixel_visible = std::stoi(val);
            else if (key == "pass1_integer_sums") pass1_integer_sums = std::stoi(val);
            else if (key == "tail_sub_bounding_box") tail_sub_bounding_box = std::stod(val);
            else if (key == "use_provided_bounding_box") use_provided_bb = std::stoi(val);
            else if (key == "bounding_box_side") BB_USER_SIDE = parse_rect(val, key);
            else if (key == "bounding_box_bottom") BB_USER_BOTTOM = parse_rect(val, key);
            else if (key == "bb_width") bb_width = std::stoi(val);
            else if (key == "bb_height_side") bb_height_side = std::stoi(val);
            else if (key == "moving_average_window") moving_average_window = std::stoi(val);
            else if (key == "bw_threshold_bottom") bw_threshold_bottom = std::stoi(val);
            else if (key == "bw_threshold_side") bw_threshold_side = std::stoi(val);
            else if (key == "min_pixel_count") min_pixel_count = std::stoi(val);
            else if (key == "zero_col_pre") zero_col_pre = std::stoi(val);
            else if (key == "zero_col_post") zero_col_post = std::stoi(val);
            else if (key == "zero_row_pre") zero_row_pre = std::stoi(val);
            else if (key == "zero_row_post") zero_row_post = std::stoi(val);
            else if (key == "disk_filter_file") disk_filter_file = val;
            else if (key == "bounding_box_file") bounding_box_file = val;
            else if (key == "device") device = std::stoi(val);
            else if (key == "batch_frames") batch_frames = std::stoi(val);
            else if (key == "max_resident_bytes") max_resident_bytes = std::stoll(val);
            else if (key == "fma_mode") fma_mode = std::stoi(val);
            else if (key == "cand_cap") cand_cap = std::stoi(val);
            else if (key == "det_cap") det_cap = std::stoi(val);
            else if (key == "match_cap") match_cap = std::stoi(val);
            else if (key == "max_displacement_bottom") max_displacement_bottom = std::stoi(val);
            else if (key == "occlusion_grid_spacing_pixels_bottom") occlusion_grid_spacing_pixels_bottom = std::stoi(val);
            else if (key == "occlusion_grid_max_width") occlusion_grid_max_width = std::stod(val);
            else if (key == "alpha_vel_bottom") alpha_vel_bottom = std::stod(val);
            else if (key == "pairwise_occluded_cost") pairwise_occluded_cost = std::stod(val);
            else if (key == "max_displacement_side") max_displacement_side = std::stoi(val);
            else if (key == "occlusion_grid_spacing_pixels_side") occlusion_grid_spacing_pixels_side = std::stoi(val);
            else if (key == "alpha_vel_side") alpha_vel_side = std::stod(val);
            else if (key == "tracker_threads") tracker_threads = std::stoi(val);
            else if (key == "batch_workers_per_gpu") batch_workers_per_gpu = std::stoi(val);
            else if (key == "location_prior" && val.rfind("!!", 0) != 0) {  // 5 x 7 as a row-major flow list; the OpenCV matrix node is read below
                const std::vector<double> W = parse_list(val, key);
                if (W.size() != 35) throw std::invalid_argument("location_prior must be a 5x7 matrix. Was " + std::to_string(W.size()) + " values.");
                for (unsigned int i = 0; i <= N_paws; ++i) {
                    const double *q = W.data() + 7 * i;
                    (i < N_paws ? PRIOR_PAW : PRIOR_SNOUT).push_back(LocoMouse_LocationPrior(q[0], q[1], q[2], q[3], q[4], q[5], q[6]));
                }
            }
            // every other reference key belongs to pass 1 or to the host tracker and is ignored here
        } catch (const std::invalid_argument &) {
            throw;
        } catch (const std::exception &) {
            throw std::invalid_argument("Could not parse the value of " + key + " in " + config_file_name);
        }
    }
    {   // location_prior written by OpenCV as a 5 x 7 matrix node (LocoMouse_class.cpp:132-145)
        cvyaml::File y(config_file_name);
        if (y.isOpened() && !y.mat("location_prior").empty() && PRIOR_PAW.empty()) {
            const cvyaml::Matrix &W = y.mat("location_prior");
            if (W.cols != 7 || W.rows != 5) throw std::invalid_argument("location_prior must be a 5x7 matrix. Was " + std::to_string(W.rows) + ".");
            for (unsigned int i = 0; i <= N_paws; ++i) {
                const double *q = W.data.data() + 7 * i;
                (i < N_paws ? PRIOR_PAW : PRIOR_SNOUT).push_back(LocoMouse_LocationPrior(q[0], q[1], q[2], q[3], q[4], q[5], q[6]));
            }
        }
    }
    if (conn_comp_connectivity != 4 && conn_comp_connectivity != 8)
        throw std::invalid_argument("conn_comp_connectivity must be either 4 or 8.");
    if (!(side_bottom_min_overlap >= 0 && side_bottom_min_overlap <= 1))
        throw std::invalid_argument("side_bottom_min_overlap must belong to [0, 1].");
    if (!(tail_sub_bounding_box >= 0 && tail_sub_bounding_box <= 1))
        throw std::invalid_argument("tail_sub_bounding_box must belong to [0, 1].");
    if (median_filter_size % 2 == 0) throw std::invalid_argument("median_filter_size must be odd. Was " + std::to_string(median_filter_size) + ".");
    if (min_pixel_visible < 0) throw std::invalid_argument("min_pixel_visible must be non-negative. Was " + std::to_string(min_pixel_visible) + ".");
    if (bb_width <= 0 || bb_height_side <= 0) throw std::invalid_argument("bb_width and bb_height_side must be positive.");
    if (batch_frames <= 0) throw std::invalid_argument("batch_frames must be positive.");
    if (max_resident_bytes <= 0) throw std::invalid_argument("max_resident_bytes must be positive.");
    if (batch_workers_per_gpu <= 0) throw std::invalid_argument("batch_workers_per_gpu must be positive.");
    if (max_displacement_side < 0) throw std::invalid_argument("max_displacement_side must be non-negative. Was " + std::to_string(max_displacement_side) + ".");
    if (occlusion_grid_spacing_pixels_side <= 0 || occlusion_grid_spacing_pixels_bottom <= 0)
        throw std::invalid_argument("occlusion_grid_spacing_pixels_side / _bottom must be positive.");
    if (alpha_vel_side < 0) throw std::invalid_argument("alpha_vel_side must be non-negative. Was " + std::to_string(alpha_vel_side) + ".");
    if (moving_average_window <= 0 || moving_average_window % 2 == 0)
        throw std::invalid_argument("moving_average_window must be a positive odd integer.");
}

// =====================================================================================================
// LocoMouse_Feature / LocoMouse_Model (LocoMouse_class.cpp:2941-2990, 3095-3162)
// =====================================================================================================
namespace {
// Rect(-(round(w/2)/2), -(round(h/2)/2), round(w/2), round(h/2)) — LocoMouse_class.cpp:2954-2969
cv::Rect half_box(cv::Size s) {
    const int w = (int)std::lround(s.width / 2.0), h = (int)std::lround(s.height / 2.0);
    return cv::Rect(-(w / 2), -(h / 2), w, h);
}
}  // namespace

LocoMouse_Feature::LocoMouse_Feature(std::vector<float> w_b, cv::Size size_b, double rho_b, std::vector<float> w_s,
                                     cv::Size size_s, double rho_s)
    : W_B(std::move(w_b)), W_S(std::move(w_s)), SIZE_B(size_b), SIZE_S(size_s), RHO_B(rho_b), RHO_S(rho_s),
      MATCH_BOX_B(half_box(size_b)), MATCH_BOX_S(half_box(size_s)) {}

LocoMouse_Model::LocoMouse_Model(const std::string &model_file_name) {
    {   // the reference's own format: OpenCV YAML with six matrices and six biases (LocoMouse_class.cpp:3095-3162)
        cvyaml::File y(model_file_name);
        if (y.isOpened()) {
            std::vector<float> w[6];
            cv::Size sz[6];
            double rho[6];
            const char *wn[6] = {"modelPaw_bottom", "modelSnout_bottom", "modelTail_bottom", "modelPaw_side", "modelSnout_side", "modelTail_side"};
            const char *bn[6] = {"biasPaw_bottom", "biasSnout_bottom", "biasTail_bottom", "biasPaw_side", "biasSnout_side", "biasTail_side"};
            for (int k = 0; k < 6; ++k) {
                const cvyaml::Matrix &m = y.mat(wn[k]);
                if (m.empty()) throw std::invalid_argument(std::string("Error: ") + wn[k] + " cannot be empty." + model_file_name);
                w[k].resize(m.data.size());
                for (size_t i = 0; i < m.data.size(); ++i) w[k][i] = (float)m.data[i];  // filter2D converts the kernel to CV_32F
                sz[k] = cv::Size(m.cols, m.rows);
                rho[k] = y.real(bn[k]);
            }
            paw = LocoMouse_Feature(w[0], sz[0], rho[0], w[3], sz[3], rho[3]);
            snout = LocoMouse_Feature(w[1], sz[1], rho[1], w[4], sz[4], rho[4]);
            tail = LocoMouse_Feature(w[2], sz[2], rho[2], w[5], sz[5], rho[5]);
            return;
        }
    }
    lmfile::Reader r(model_file_name, "LMM1");
    std::vector<float> w[6];
    cv::Size sz[6];
    double rho[6];
    for (int k = 0; k < 6; ++k) {
        const int rows = r.i32(), cols = r.i32();
        rho[k] = r.f64();
        if (rows <= 0 || cols <= 0 || rows > 4096 || cols > 4096) throw std::runtime_error("Model file holds an empty or oversized template.");
        w[k].resize((size_t)rows * cols);
        r.read(w[k].data(), w[k].size());
        sz[k] = cv::Size(cols, rows);
    }
    paw = LocoMouse_Feature(w[0], sz[0], rho[0], w[3], sz[3], rho[3]);
    snout = LocoMouse_Feature(w[1], sz[1], rho[1], w[4], sz[4], rho[4]);
    tail = LocoMouse_Feature(w[2], sz[2], rho[2], w[5], sz[5], rho[5]);
}

// =====================================================================================================
// LocoMouse
// =====================================================================================================
struct LocoMouse::Batch {
    unsigned int first = 0, count = 0;
    int cand_cap = 0, match_cap = 0, n_tail = 0;
    // page-locked: lm_detect_batch copies device -> here directly (include/locomouse_b200.h, lm_host_alloc)
    PinnedArray<int32_t> n_bottom, n_side, match_n, match_y, tail;
    PinnedArray<lm_cand> bottom, side;
    PinnedArray<double> match_s;
    PinnedArray<uint32_t> flags;
    // cost builders (per feature): unary [count][n_priors][cand_cap]; pairwise packed CSC over count + 1 frames (frame 0 =
    // last frame of the previous chunk, so that the first transition of this chunk is present)
    bool has_costs = false;
    int n_priors[2] = {0, 0}, nong = 0;
    std::vector<double> unary[2], pw_pr[2];
    std::vector<int64_t> pw_offs[2];
    std::vector<int32_t> pw_jc[2], pw_ir[2];
    lm_results view() {
        lm_results r{};
        r.n_frames = count;
        r.cand_cap = cand_cap;
        r.match_cap = match_cap;
        r.n_tail_points = n_tail;
        r.n_bottom = n_bottom.data();
        r.n_side = n_side.data();
        r.bottom = bottom.data();
        r.side = side.data();
        r.match_n = match_n.data();
        r.match_y = match_y.data();
        r.match_s = match_s.data();
        r.tail = tail.data();
        r.flags = flags.data();
        return r;
    }
};

void LocoMouse::check(int rc) const {
    if (rc == LM_OK) return;
    const std::string msg = lm_last_error(CTX);
    if (rc == LM_ERR_INVALID) throw std::invalid_argument(msg);
    throw std::runtime_error(msg);  // LM_ERR_RUNTIME, LM_ERR_ROI, LM_ERR_OVERFLOW, LM_ERR_STATE
}

void LocoMouse::initializePaths(const LocoMouse_ParseInputs &INPUT) {
    LM_CALL = INPUT.LM_CALL;
    CONFIG_FILE = INPUT.CONFIG_FILE;
    VIDEO_FILE = INPUT.VIDEO_FILE;
    BKG_FILE = INPUT.BKG_FILE;
    MODEL_FILE = INPUT.MODEL_FILE;
    CALIBRATION_FILE = INPUT.CALIBRATION_FILE;
    FLIP_CHAR = INPUT.FLIP_CHAR;
    OUTPUT_PATH = INPUT.OUTPUT_PATH;
    // output_<stem>.* next to the reference's output_<stem>.yml (LocoMouse_class.cpp:360)
    output_file = OUTPUT_PATH + "/output_" + INPUT.FILE_STEM + ".lmo";
    costs_file = OUTPUT_PATH + "/costs_" + INPUT.FILE_STEM + ".lmo";
    tracks_file = OUTPUT_PATH + "/output_" + INPUT.FILE_STEM + ".yml";  // the reference's own output file (class.cpp:360)
}

void LocoMouse_Media::load(const std::string &video_file, const std::string &bkg_file, size_t max_resident_bytes, int batch_frames) {
    // AVI, the reference's input (VideoCapture + extractChannel(0), class.cpp:367-400, 1282-1293), or the LMV1 container
    index = lmmedia::index_video(video_file);
    n_frames = (unsigned int)index.n;
    rows = index.rows;
    cols = index.cols;
    codec = index.codec;  // coded frames are decoded on the device once lm_configure has run (LocoMouse::useWindow)
    extradata = index.extradata;
    windows = lmmedia::plan_windows(index.n, lmmedia::window_frames(max_resident_bytes, (size_t)rows * cols, batch_frames), index.keyframe);
    window = 0;
    read_window(0, data, offsets);
    if (lmmedia::is_png(bkg_file)) {  // imread(BKG_FILE, CV_LOAD_IMAGE_GRAYSCALE) (class.cpp:402-417)
        lmmedia::Image I = lmmedia::read_png_gray(bkg_file);
        if (I.rows != rows || I.cols != cols) throw std::runtime_error("Background image and video frames must have the same size.");
        bkg = std::move(I.px);
        return;
    }
    lmfile::Reader r(bkg_file, "LMI1");
    const int brows = r.i32(), bcols = r.i32();
    if (brows <= 0 || bcols <= 0) throw std::runtime_error("Background image is empty: " + bkg_file);
    bkg.resize((size_t)brows * bcols);
    r.read(bkg.data(), bkg.size());
    if (brows != rows || bcols != cols) throw std::runtime_error("Background image and video frames must have the same size.");
}

// Frames (or coded chunks) of window k, read from the file straight into the page-locked buffer `to`
void LocoMouse_Media::read_window(int k, PinnedArray<uint8_t> &to, std::vector<int64_t> &to_offsets) const {
    lmmedia::Video V = lmmedia::read_frames(index, windows[(size_t)k], windows[(size_t)k + 1] - windows[(size_t)k], [&to](size_t b) {
        to.resize(b);
        return to.data();
    });
    to_offsets = std::move(V.offsets);
}

bool LocoMouse_DeviceFrames::reserve(lm_ctx *ctx, size_t need) {
    if (p && bytes >= need) return true;
    release(ctx);
    void *d = nullptr;
    if (lm_device_alloc(ctx, &d, need) != LM_OK) return false;
    p = static_cast<uint8_t *>(d);
    bytes = need;
    return true;
}

void LocoMouse_DeviceFrames::release(lm_ctx *ctx) {
    if (p) lm_device_free(ctx, p);
    p = nullptr;
    bytes = 0;
}

void LocoMouse::loadCalibration() {
    {   // the reference's own format: OpenCV YAML with ind_warp_mapping and view_boxes (LocoMouse_class.cpp:419-463)
        cvyaml::File y(CALIBRATION_FILE);
        if (y.isOpened()) {
            const cvyaml::Matrix &c = y.mat("ind_warp_mapping"), &vb = y.mat("view_boxes");
            if (c.empty()) throw std::invalid_argument("ind_warp_mapping is empty or undefined.");
            if (vb.empty()) throw std::invalid_argument("view_boxes is empty or undefined.");
            if (vb.rows != 2 || vb.cols != 4) throw std::invalid_argument("view_boxes sould be a 2x4 matrix.");
            if (vb.dt != 'i') throw std::invalid_argument("Bounding boxes must be defined with integer pixel positions!");
            if (!c.is_integer()) throw std::invalid_argument("ind_warp_mapping must hold integer pixel indices.");
            BB_SIDE_VIEW = cv::Rect((int)vb.data[0], (int)vb.data[1], (int)vb.data[2], (int)vb.data[3]);
            BB_BOTTOM_VIEW = cv::Rect((int)vb.data[4], (int)vb.data[5], (int)vb.data[6], (int)vb.data[7]);
            N_ROWS = (unsigned int)c.rows;
            N_COLS = (unsigned int)c.cols;
            CALIBRATION.resize(c.data.size());
            for (size_t i = 0; i < c.data.size(); ++i) CALIBRATION[i] = (int32_t)c.data[i];
            return;
        }
    }
    lmfile::Reader r(CALIBRATION_FILE, "LMC1");
    const int rows = r.i32(), cols = r.i32();
    if (rows <= 0 || cols <= 0) throw std::invalid_argument("ind_warp_mapping is empty or undefined.");
    int32_t vb[8];
    r.read(vb, 8);
    BB_SIDE_VIEW = cv::Rect(vb[0], vb[1], vb[2], vb[3]);
    BB_BOTTOM_VIEW = cv::Rect(vb[4], vb[5], vb[6], vb[7]);
    N_ROWS = (unsigned int)rows;
    N_COLS = (unsigned int)cols;
    CALIBRATION.resize((size_t)rows * cols);
    r.read(CALIBRATION.data(), CALIBRATION.size());
}

void LocoMouse::loadFlip() {
    if (FLIP_CHAR.length() != 1 || (FLIP_CHAR[0] != 'L' && FLIP_CHAR[0] != 'R'))
        throw std::invalid_argument("Mouse side option must be either \"L\" or \"R\".");
    IMAGE_FLIP = FLIP_CHAR[0] == 'L';
}

// LocoMouse_class.cpp:486-540: the calibration map must address pixels of the video frame and the view boxes
// must lie inside the calibrated image.
void LocoMouse::validateImageVideoSize() {
    const int64_t lim = (int64_t)VID_ROWS * VID_COLS;
    for (int32_t v : CALIBRATION)
        if (v < 0 || v >= lim) throw std::runtime_error("Calibration mapping indices do not match the video size.");
    auto inside = [&](const cv::Rect &b) {
        return b.x >= 0 && b.y >= 0 && b.width > 0 && b.height > 0 && b.x + b.width <= (int)N_COLS && b.y + b.height <= (int)N_ROWS;
    };
    if (!inside(BB_SIDE_VIEW) || !inside(BB_BOTTOM_VIEW)) throw std::runtime_error("view_boxes do not fit the calibrated image.");
}

LocoMouse::LocoMouse(LocoMouse_ParseInputs INPUTS) {
    initializePaths(INPUTS);
    LM_PARAMS = LocoMouse_Parameters(CONFIG_FILE);
    OWN_MEDIA.reset(new LocoMouse_Media());
    OWN_MEDIA->load(VIDEO_FILE, BKG_FILE, (size_t)LM_PARAMS.max_resident_bytes, LM_PARAMS.batch_frames);
    OWN_POOL.reset(new LocoMouse_WindowPool());
    initializeInputs(*OWN_MEDIA, OWN_POOL.get());
    const int rc = lm_create(&CTX, LM_PARAMS.device);
    if (rc != LM_OK) throw std::runtime_error(std::string("lm_create: ") + lm_last_error(nullptr));
}

LocoMouse::LocoMouse(LocoMouse_ParseInputs INPUTS, const LocoMouse_Parameters &params, LocoMouse_Media &media, lm_ctx *ctx,
                     LocoMouse_WindowPool *pool)
    : OWN_CTX(false) {
    initializePaths(INPUTS);
    LM_PARAMS = params;
    initializeInputs(media, pool);
    CTX = ctx;
}

void LocoMouse::initializeInputs(LocoMouse_Media &media, LocoMouse_WindowPool *pool) {
    MEDIA = &media;
    POOL = pool;
    POOL->spare_window = -1;
    N_FRAMES = media.n_frames;
    VID_ROWS = media.rows;
    VID_COLS = media.cols;
    loadCalibration();
    validateImageVideoSize();
    M = LocoMouse_Model(MODEL_FILE);
    loadFlip();
    // sized, not merely reserved (the reference indexes reserved vectors, SURVEY Q12)
    BB_X_POS.assign(N_FRAMES, 0);
    BB_Y_SIDE_POS.assign(N_FRAMES, 0);
    BB_Y_BOTTOM_POS.assign(N_FRAMES, 0);
}

LocoMouse::~LocoMouse() {
    if (READER.valid()) READER.wait();
    if (OWN_POOL) OWN_POOL->release(CTX);
    if (OWN_CTX) lm_destroy(CTX);
}

const uint8_t *LocoMouse::frames(int &on_device) const {
    on_device = MEDIA->codec != lmmedia::Codec::raw ? 1 : 0;
    return on_device ? POOL->decoded.p : MEDIA->data.data();
}

int LocoMouse::windowOf(unsigned int frame) const {
    return (int)(std::upper_bound(MEDIA->windows.begin(), MEDIA->windows.end(), (int)frame) - MEDIA->windows.begin()) - 1;
}

void LocoMouse::useWindow(int k, int next) {
    const size_t fsz = (size_t)VID_ROWS * VID_COLS;
    const bool coded = MEDIA->codec != lmmedia::Codec::raw;
    const std::vector<int> &W = MEDIA->windows;
    if (MEDIA->window != k) {
        const int cur = MEDIA->window;
        if (k == cur + 1 && (!coded || DECODED_WINDOW == cur)) {  // window k's first frame needs cur's last one (I_PREV_PAD)
            const size_t last = (size_t)(W[(size_t)k] - 1 - W[(size_t)cur]) * fsz;
            if (coded) {
                if (!POOL->prev_decoded.reserve(CTX, fsz)) throw std::runtime_error(std::string("Cannot keep the previous frame in device memory: ") + lm_last_error(CTX));
                check(lm_device_copy(CTX, POOL->prev_decoded.p, POOL->decoded.p + last, fsz));
            } else {
                POOL->prev.resize(fsz);
                std::copy_n(MEDIA->data.data() + last, fsz, POOL->prev.data());
            }
            PREV_WINDOW = cur;
        }
        if (READER.valid()) READER.get();  // rethrows what the reader met
        if (POOL->spare_window != k) {
            POOL->spare_window = -1;
            MEDIA->read_window(k, POOL->spare, POOL->spare_offsets);
        }
        MEDIA->data.swap(POOL->spare);
        MEDIA->offsets.swap(POOL->spare_offsets);
        POOL->spare_window = MEDIA->window;
        MEDIA->window = k;
    }
    if (coded && DECODED_WINDOW != k) {
        const int64_t n = W[(size_t)k + 1] - W[(size_t)k];
        const size_t bytes = (size_t)n * fsz;
        if (!POOL->decoded.reserve(CTX, bytes))
            throw std::runtime_error(std::string(W.size() > 2 ? "A decoded window of the video (" : "The decoded video (") + std::to_string(n) + " frames, " +
                                     std::to_string(bytes) + " bytes) does not fit in device memory: " + lm_last_error(CTX));
        DECODED_WINDOW = -1;
        if (MEDIA->codec == lmmedia::Codec::png)
            check(lm_decode_png(CTX, MEDIA->data.data(), 0, MEDIA->offsets.data(), n, POOL->decoded.p));
        else
            check(lm_decode_ffv1(CTX, MEDIA->extradata.data(), (int64_t)MEDIA->extradata.size(), MEDIA->data.data(), 0, MEDIA->offsets.data(), n,
                                 POOL->decoded.p));
        DECODED_WINDOW = k;
    }
    if (next >= 0 && next != k && POOL->spare_window != next && !READER.valid()) {
        POOL->spare_window = -1;
        READER = std::async(std::launch::async, [this, next] {
            MEDIA->read_window(next, POOL->spare, POOL->spare_offsets);
            POOL->spare_window = next;
        });
    }
}

void LocoMouse::pass1Windows(const std::function<void(const uint8_t *, int, unsigned int, unsigned int)> &run) {
    const int K = (int)windows();
    for (int k = 0; k < K; ++k) {
        useWindow(k, K > 1 ? (k + 1) % K : -1);  // after the last window the frame loop starts again at window 0
        int on_dev = 0;
        const uint8_t *video = frames(on_dev);
        run(video, on_dev, (unsigned int)MEDIA->windows[(size_t)k], (unsigned int)(MEDIA->windows[(size_t)k + 1] - MEDIA->windows[(size_t)k]));
    }
}

size_t LocoMouse::residentBytes() const {
    return MEDIA->data.capacity() + POOL->spare.capacity() + POOL->prev.capacity() + POOL->decoded.bytes + POOL->prev_decoded.bytes;
}

// ---- pass 1 (out of scope): positions come from the user box or from a pass-1 output file -------------
namespace {
void read_boxes(const std::string &file, unsigned int n_frames, std::vector<unsigned int> &x, std::vector<unsigned int> &ys,
                std::vector<unsigned int> &yb) {
    if (file.empty())
        throw std::invalid_argument(
            "The first pass (computeBoundingBox) is not part of this library: set use_provided_bounding_box or "
            "bounding_box_file in the configuration.");
    lmfile::Reader r(file, "LMB1");
    const int n = r.i32();
    if (n < 0 || (unsigned int)n != n_frames) throw std::runtime_error("bounding_box_file does not match the number of video frames.");
    x.resize(n_frames);
    ys.resize(n_frames);
    yb.resize(n_frames);
    r.read(x.data(), n_frames);
    r.read(ys.data(), n_frames);
    r.read(yb.data(), n_frames);
}
}  // namespace

void LocoMouse::getBoundingBox() {
    if (LM_PARAMS.use_provided_bb) {
        // LocoMouse_class.cpp:545-567: bottom-right corner = origin + size, boxes re-anchored at (0, 0)
        const unsigned int x = LM_PARAMS.BB_USER_BOTTOM.x + LM_PARAMS.BB_USER_BOTTOM.width;
        const unsigned int ys = LM_PARAMS.BB_USER_SIDE.y + LM_PARAMS.BB_USER_SIDE.height;
        const unsigned int yb = LM_PARAMS.BB_USER_BOTTOM.y + LM_PARAMS.BB_USER_BOTTOM.height;
        std::fill(BB_X_POS.begin(), BB_X_POS.end(), x);
        std::fill(BB_Y_SIDE_POS.begin(), BB_Y_SIDE_POS.end(), ys);
        std::fill(BB_Y_BOTTOM_POS.begin(), BB_Y_BOTTOM_POS.end(), yb);
        BB_BOTTOM_MOUSE = cv::Rect(0, 0, LM_PARAMS.BB_USER_BOTTOM.width, LM_PARAMS.BB_USER_BOTTOM.height);
        BB_SIDE_MOUSE = cv::Rect(0, 0, LM_PARAMS.BB_USER_SIDE.width, LM_PARAMS.BB_USER_SIDE.height);
    } else {
        computeBoundingBox();
    }
}

// LocoMouse::computeBoundingBox (LocoMouse_class.cpp:578-653).  Per frame computeMouseBox runs on the device
// (lm_bounding_box_base: median, threshold, largest component of each view, sums, first / last); computeMouseBoxSize and the
// three moving averages follow on the host as in the reference.  A pass-1 output file (bounding_box_file) replaces it.
void LocoMouse::computeBoundingBox() {
    if (!LM_PARAMS.bounding_box_file.empty()) {
        read_boxes(LM_PARAMS.bounding_box_file, N_FRAMES, BB_X_POS, BB_Y_SIDE_POS, BB_Y_BOTTOM_POS);
        if (LM_PARAMS.BB_USER_BOTTOM.width <= 0 || LM_PARAMS.BB_USER_SIDE.width <= 0)
            throw std::invalid_argument("bounding_box_side / bounding_box_bottom must give the box sizes when bounding_box_file is used.");
        BB_BOTTOM_MOUSE = cv::Rect(0, 0, LM_PARAMS.BB_USER_BOTTOM.width, LM_PARAMS.BB_USER_BOTTOM.height);
        BB_SIDE_MOUSE = cv::Rect(0, 0, LM_PARAMS.BB_USER_SIDE.width, LM_PARAMS.BB_USER_SIDE.height);
        return;
    }
    // lm_configure needs positive box sizes; pass 1 does not use them
    BB_BOTTOM_MOUSE = cv::Rect(0, 0, 1, 1);
    BB_SIDE_MOUSE = cv::Rect(0, 0, 1, 1);
    configureDevice();
    lm_bb_base_params p{};
    p.side_x = BB_SIDE_VIEW.x;
    p.side_y = BB_SIDE_VIEW.y;
    p.side_w = BB_SIDE_VIEW.width;
    p.side_h = BB_SIDE_VIEW.height;
    p.bottom_x = BB_BOTTOM_VIEW.x;
    p.bottom_y = BB_BOTTOM_VIEW.y;
    p.bottom_w = BB_BOTTOM_VIEW.width;
    p.bottom_h = BB_BOTTOM_VIEW.height;
    p.median_filter_size = LM_PARAMS.median_filter_size;
    p.min_pixel_visible = LM_PARAMS.min_pixel_visible;
    p.sums_as_float = LM_PARAMS.pass1_integer_sums ? 0 : 1;
    std::vector<double> box((size_t)N_FRAMES * 6);
    pass1Windows([&](const uint8_t *video, int on_dev, unsigned int first, unsigned int n) {
        check(lm_bounding_box_base(CTX, video, on_dev, n, &p, box.data() + (size_t)first * 6, nullptr));
    });
    std::vector<double> bb_x(N_FRAMES), bb_yb(N_FRAMES), bb_ys(N_FRAMES), w(N_FRAMES), hb(N_FRAMES), hs(N_FRAMES);
    for (unsigned int f = 0; f < N_FRAMES; ++f) {
        const double *o = &box[(size_t)f * 6];
        bb_x[f] = o[0];
        bb_yb[f] = o[1];
        bb_ys[f] = o[2];
        w[f] = o[3];
        hb[f] = o[4];
        hs[f] = o[5];
    }
    int32_t size[3];
    if (lm_mouse_box_size(w.data(), hb.data(), hs.data(), N_FRAMES, size) != LM_OK) throw std::runtime_error("computeMouseBoxSize failed.");
    BB_SIDE_MOUSE = cv::Rect(0, 0, size[0], size[2]);
    BB_BOTTOM_MOUSE = cv::Rect(0, 0, size[0], size[1]);
    BB_X_POS.assign(N_FRAMES, 0);
    BB_Y_BOTTOM_POS.assign(N_FRAMES, 0);
    BB_Y_SIDE_POS.assign(N_FRAMES, 0);
    const int win = LM_PARAMS.moving_average_window;
    if (lm_moving_average(bb_x.data(), N_FRAMES, win, BB_X_POS.data()) != LM_OK || lm_moving_average(bb_yb.data(), N_FRAMES, win, BB_Y_BOTTOM_POS.data()) != LM_OK ||
        lm_moving_average(bb_ys.data(), N_FRAMES, win, BB_Y_SIDE_POS.data()) != LM_OK)
        throw std::invalid_argument("moving_average_window is invalid.");
    if (size[0] <= 0 || size[1] <= 0 || size[2] <= 0)
        // With the reference's own settings this is what its pass 1 yields: firstLastOverT reads the integer sums as floats
        // (LocoMouse_class.hpp:417), every limit is -1 and the box collapses; the reference then fails inside OpenCV.
        throw std::runtime_error("computeBoundingBox(): the mouse box is empty (width " + std::to_string(size[0]) + ", heights " + std::to_string(size[1]) + " / " +
                                 std::to_string(size[2]) + "); set pass1_integer_sums: 1, use_provided_bounding_box or bounding_box_file.");
}

LocoMouse_TM::LocoMouse_TM(LocoMouse_ParseInputs INPUTS) : LocoMouse(INPUTS) {
    METHOD = 1;
    REF_PATH = INPUTS.REF_PATH;
}

LocoMouse_TM::LocoMouse_TM(LocoMouse_ParseInputs INPUTS, const LocoMouse_Parameters &params, LocoMouse_Media &media, lm_ctx *ctx,
                           LocoMouse_WindowPool *pool)
    : LocoMouse(INPUTS, params, media, ctx, pool) {
    METHOD = 1;
    REF_PATH = INPUTS.REF_PATH;
}

// LocoMouse_TM::computeBoundingBox (LocoMouse_TM.cpp:115-157): x from computeMouseBox_DD per frame (on the device:
// lm_bounding_box_tm) smoothed by the moving average, bottom anchor = last image row, side anchor = row 164.  A pass-1 output
// file (bounding_box_file) replaces the per-frame part.  The reference reads its parameters and diskfilter.yml in the
// constructor (LocoMouse_TM.cpp:3-42) and fails there when they are missing; here they are only required when pass 1 runs.
void LocoMouse_TM::computeBoundingBox() {
    if (!LM_PARAMS.bounding_box_file.empty()) {
        std::vector<unsigned int> ys, yb;
        read_boxes(LM_PARAMS.bounding_box_file, N_FRAMES, BB_X_POS, ys, yb);
    } else {
        const std::string dfile = LM_PARAMS.disk_filter_file.empty() ? REF_PATH + "diskfilter.yml" : LM_PARAMS.disk_filter_file;
        cvyaml::File y(dfile);
        if (!y.isOpened() || !y.has("H")) throw std::invalid_argument("Failed to read config file: diskfilter.yml");  // LocoMouse_TM.cpp:9
        const cvyaml::Matrix &Hm = y.mat("H");
        if (Hm.empty() || Hm.rows != Hm.cols) throw std::invalid_argument("diskfilter.yml: H must be a square matrix.");
        DISK_SIZE = Hm.rows;
        DISK_FILTER.assign(Hm.data.begin(), Hm.data.end());
        // LocoMouse_TM_Parameters' range checks (LocoMouse_TM.cpp:58-111), same messages
        const std::string em = "Invalid configuration parameter: ";
        if (LM_PARAMS.bw_threshold_bottom < 0 || LM_PARAMS.bw_threshold_bottom > 255) throw std::invalid_argument(em + "bw_threshold_bottom must belong to [0, 1].");
        if (LM_PARAMS.bw_threshold_side < 0 || LM_PARAMS.bw_threshold_side > 255) throw std::invalid_argument(em + "bw_threshold_side must belong to [0, 255].");
        if (LM_PARAMS.min_pixel_count < 1) throw std::invalid_argument(em + "Min pixel count must be at least 1.");
        if (LM_PARAMS.zero_col_post < 0 || LM_PARAMS.zero_col_pre < 0 || LM_PARAMS.zero_row_post < 0 || LM_PARAMS.zero_row_pre < 0)
            throw std::invalid_argument(em + "zero_*_* parameters range from 0 to the relevant size of the image.");
        if (LM_PARAMS.bb_width < 1) throw std::invalid_argument(em + "bb_width must be at least 1 pixel.");
        if (LM_PARAMS.bb_height_side < 1) throw std::invalid_argument(em + "bb_height_side must be at least 1 pixel.");
        // LocoMouse_TM.cpp:20-36
        if (BB_SIDE_VIEW.width < LM_PARAMS.zero_col_pre || BB_SIDE_VIEW.width < LM_PARAMS.zero_col_post)
            throw std::invalid_argument("Side View image size is not compatible with the zero_col parameters for the bounding box computations. See the definition of the LocoMouse_TM class.");
        if (BB_SIDE_VIEW.height < LM_PARAMS.zero_row_pre || BB_SIDE_VIEW.height < LM_PARAMS.zero_row_post)
            throw std::invalid_argument("Side View image size is not compatible with the zero_row parameters for the bounding box computations. See the definition of the LocoMouse_TM class.");
        // lm_configure needs positive box sizes; pass 1 does not use them
        BB_SIDE_MOUSE = cv::Rect(0, 0, LM_PARAMS.bb_width, LM_PARAMS.bb_height_side);
        BB_BOTTOM_MOUSE = cv::Rect(0, 0, LM_PARAMS.bb_width, BB_BOTTOM_VIEW.height);
        configureDevice();
        lm_bb_tm_params p{};
        p.side_x = BB_SIDE_VIEW.x;
        p.side_y = BB_SIDE_VIEW.y;
        p.side_w = BB_SIDE_VIEW.width;
        p.side_h = BB_SIDE_VIEW.height;
        p.side_threshold = LM_PARAMS.bw_threshold_side;
        p.min_pixel_count = LM_PARAMS.min_pixel_count;
        p.min_pixel_visible = LM_PARAMS.min_pixel_visible;
        p.zero_col_pre = LM_PARAMS.zero_col_pre;
        p.zero_col_post = LM_PARAMS.zero_col_post;
        p.zero_row_pre = LM_PARAMS.zero_row_pre;
        p.zero_row_post = LM_PARAMS.zero_row_post;
        p.sums_as_float = LM_PARAMS.pass1_integer_sums ? 0 : 1;
        p.disk_size = DISK_SIZE;
        p.disk = DISK_FILTER.data();
        std::vector<double> bb_x(N_FRAMES);
        pass1Windows([&](const uint8_t *video, int on_dev, unsigned int first, unsigned int n) {
            check(lm_bounding_box_tm(CTX, video, on_dev, n, &p, bb_x.data() + first, nullptr));
        });
        BB_X_POS.assign(N_FRAMES, 0);
        if (lm_moving_average(bb_x.data(), N_FRAMES, LM_PARAMS.moving_average_window, BB_X_POS.data()) != LM_OK)
            throw std::invalid_argument("moving_average_window is invalid.");
    }
    std::fill(BB_Y_BOTTOM_POS.begin(), BB_Y_BOTTOM_POS.end(), N_ROWS - 1);
    std::fill(BB_Y_SIDE_POS.begin(), BB_Y_SIDE_POS.end(), 165u - 1u);
    BB_SIDE_MOUSE = cv::Rect(0, 0, LM_PARAMS.bb_width, LM_PARAMS.bb_height_side);
    BB_BOTTOM_MOUSE = cv::Rect(0, 0, LM_PARAMS.bb_width, BB_BOTTOM_VIEW.height);
}

LocoMouse_TM_DE::LocoMouse_TM_DE(LocoMouse_ParseInputs INPUTS) : LocoMouse_TM(INPUTS) { METHOD = 2; }

LocoMouse_TM_DE::LocoMouse_TM_DE(LocoMouse_ParseInputs INPUTS, const LocoMouse_Parameters &params, LocoMouse_Media &media, lm_ctx *ctx,
                                 LocoMouse_WindowPool *pool)
    : LocoMouse_TM(INPUTS, params, media, ctx, pool) {
    METHOD = 2;
}

// LocoMouse_TM_DE.cpp:8-53: side anchor = last row of the side view, 400-wide boxes over the full view heights.  The
// per-frame mouse position (computeMouseBox_DE, LocoMouse_TM_DE.cpp:56-113) runs on the device unless a pass-1 output
// file is supplied; the moving average over the video follows on the host as in the reference.
void LocoMouse_TM_DE::computeBoundingBox() {
    BB_SIDE_MOUSE = cv::Rect(0, 0, 400, BB_SIDE_VIEW.height);
    BB_BOTTOM_MOUSE = cv::Rect(0, 0, 400, BB_BOTTOM_VIEW.height);
    if (!LM_PARAMS.bounding_box_file.empty()) {
        std::vector<unsigned int> ys, yb;
        read_boxes(LM_PARAMS.bounding_box_file, N_FRAMES, BB_X_POS, ys, yb);
    } else {
        configureDevice();
        lm_bb_de_params p{};
        p.side_x = BB_SIDE_VIEW.x;
        p.side_y = BB_SIDE_VIEW.y;
        p.side_w = BB_SIDE_VIEW.width;
        p.side_h = BB_SIDE_VIEW.height;
        p.zero_col_pre = 46;            // LocoMouse_TM_DE.cpp:68-71 ("hand-set like this for the TM")
        p.zero_col_post = 760;
        p.zero_row_pre = 100;
        p.zero_row_post = 149;
        p.threshold = 255 * 0.05;       // LocoMouse_TM_DE.hpp:27-29
        p.min_count = 10;
        p.width_margin = 1.1;
        std::vector<double> bb_x(N_FRAMES);
        pass1Windows([&](const uint8_t *video, int on_dev, unsigned int first, unsigned int n) {
            check(lm_bounding_box_tm_de(CTX, video, on_dev, n, &p, bb_x.data() + first, nullptr));
        });
        BB_X_POS.assign(N_FRAMES, 0);
        if (lm_moving_average(bb_x.data(), N_FRAMES, LM_PARAMS.moving_average_window, BB_X_POS.data()) != LM_OK)
            throw std::invalid_argument("moving_average_window is invalid.");
    }
    std::fill(BB_Y_BOTTOM_POS.begin(), BB_Y_BOTTOM_POS.end(), N_ROWS - 1);
    std::fill(BB_Y_SIDE_POS.begin(), BB_Y_SIDE_POS.end(), (unsigned int)BB_SIDE_VIEW.height - 1u);
}

void LocoMouse::configureDevice() {
    lm_config c{};
    c.vid_rows = VID_ROWS;
    c.vid_cols = VID_COLS;
    c.n_rows = (int)N_ROWS;
    c.n_cols = (int)N_COLS;
    c.bb_w = BB_BOTTOM_MOUSE.width;
    c.bb_h_bottom = BB_BOTTOM_MOUSE.height;
    c.bb_h_side = BB_SIDE_MOUSE.height;
    c.tail_w = (int)(unsigned int)((int)(double)(BB_BOTTOM_MOUSE.width) * LM_PARAMS.tail_sub_bounding_box);  // class.cpp:711
    c.flip = IMAGE_FLIP ? 1 : 0;
    c.imadjust = usesImadjust() ? 1 : 0;
    c.conn = LM_PARAMS.conn_comp_connectivity;
    c.n_tail_points = (int)LM_PARAMS.N_tail_points;
    c.min_overlap = LM_PARAMS.side_bottom_min_overlap;
    c.fma_mode = LM_PARAMS.fma_mode;
    c.cand_cap = LM_PARAMS.cand_cap;
    c.det_cap = LM_PARAMS.det_cap;
    c.match_cap = LM_PARAMS.match_cap;
    check(lm_configure(CTX, &c));
    check(lm_set_background(CTX, MEDIA->bkg.data()));
    check(lm_set_calibration(CTX, CALIBRATION.data()));
    if (windows() == 1) useWindow(0, -1);  // a compressed video in one window is decoded once; pass 1 and the frame loop read it in place
}

// ---- initializeFeatureLoop (LocoMouse_class.cpp:655-769): hand the per-video state to the device -------
void LocoMouse::initializeFeatureLoop() {
    if (BB_BOTTOM_MOUSE.width <= 0 || BB_BOTTOM_MOUSE.width != BB_SIDE_MOUSE.width)
        throw std::invalid_argument("getBoundingBox() must run first and both views must share the box width.");
    configureDevice();
    const LocoMouse_Feature *F[3] = {&M.paw, &M.snout, &M.tail};
    lm_template t[2][3];
    for (int k = 0; k < 3; ++k) {
        t[LM_BOTTOM][k] = lm_template{F[k]->w_b().data(), F[k]->size_bottom().height, F[k]->size_bottom().width, F[k]->rho_b()};
        t[LM_SIDE][k] = lm_template{F[k]->w_s().data(), F[k]->size_side().height, F[k]->size_side().width, F[k]->rho_s()};
    }
    check(lm_set_model(CTX, t));

    CANDIDATES_BOTTOM_PAW.clear();
    CANDIDATES_BOTTOM_SNOUT.clear();
    CANDIDATES_SIDE_PAW.clear();
    CANDIDATES_SIDE_SNOUT.clear();
    CANDIDATES_MATCHED_VIEWS_PAW.clear();
    CANDIDATES_MATCHED_VIEWS_SNOUT.clear();
    TRACKS_TAIL.clear();
    CANDIDATES_BOTTOM_PAW.reserve(N_FRAMES);
    CANDIDATES_BOTTOM_SNOUT.reserve(N_FRAMES);
    CANDIDATES_SIDE_PAW.reserve(N_FRAMES);
    CANDIDATES_SIDE_SNOUT.reserve(N_FRAMES);
    CANDIDATES_MATCHED_VIEWS_PAW.reserve(N_FRAMES);
    CANDIDATES_MATCHED_VIEWS_SNOUT.reserve(N_FRAMES);
    TRACKS_TAIL.reserve(N_FRAMES);
    {   // occlusion grids (class.cpp:726-759); integer / double arithmetic as written there
        const int sp = LM_PARAMS.occlusion_grid_spacing_pixels_bottom, sps = LM_PARAMS.occlusion_grid_spacing_pixels_side;
        const unsigned int ngrid_y = (unsigned int)(((BB_BOTTOM_MOUSE.height - sp) / sp) + 1);
        const unsigned int ngrid_x = (unsigned int)(((LM_PARAMS.occlusion_grid_max_width * BB_BOTTOM_MOUSE.width) - sp) / sp + 1);
        ONG_size = cv::Size((int)ngrid_x, (int)ngrid_y);
        ONG_BR_corner = cv::Point_<double>(BB_BOTTOM_MOUSE.width - 1 - sp / 2, BB_BOTTOM_MOUSE.height - 1 - sp / 2);
        ONG.assign((size_t)ngrid_x * ngrid_y, cv::Point_<double>(0, 0));
        for (unsigned int j = 0; j < ngrid_y; ++j)
            for (unsigned int i = 0; i < ngrid_x; ++i)
                ONG[(size_t)j * ngrid_x + i] = cv::Point_<double>(ONG_BR_corner.x - (double)(i * (unsigned int)sp), ONG_BR_corner.y - (double)(j * (unsigned int)sp));
        const unsigned int nong_side = (unsigned int)(((BB_SIDE_MOUSE.height - sps) / sps) + 1);
        ONG_SIDE_LOWEST_POINT = (unsigned int)(BB_SIDE_MOUSE.height - 1 - sps / 2);
        ONG_SIDE.clear();
        for (unsigned int i = 0; i < nong_side; ++i) ONG_SIDE.push_back(ONG_SIDE_LOWEST_POINT - i * (unsigned int)sps);
    }
    UNARY_BOTTOM_PAW.clear();
    UNARY_BOTTOM_SNOUT.clear();
    PAIRWISE_BOTTOM_PAW.clear();
    PAIRWISE_BOTTOM_SNOUT.clear();
    CURRENT_FRAME = -1;  // the reference rewinds the video here (class.cpp:762)
    BATCH.reset();
    SPARE.reset();
    LOOP_READY = true;
}

// One lm_detect_batch call for frames [first, first + batch_frames): this is the whole hot loop of
// main.cpp:54-82 for those frames.
void LocoMouse::runChunk(unsigned int first) {
    // a chunk ends with its window; the window after it is read while this one is tracked
    const int k = windowOf(first), K = (int)windows();
    useWindow(k, k + 1 < K ? k + 1 : -1);
    const unsigned int w0 = (unsigned int)MEDIA->windows[(size_t)k];
    const unsigned int n = std::min<unsigned int>((unsigned int)LM_PARAMS.batch_frames, (unsigned int)MEDIA->windows[(size_t)k + 1] - first);
    std::unique_ptr<Batch> b = std::move(SPARE);
    if (!b) b.reset(new Batch());
    b->has_costs = false;
    b->first = first;
    b->count = n;
    b->cand_cap = LM_PARAMS.cand_cap;
    b->match_cap = LM_PARAMS.match_cap;
    b->n_tail = (int)LM_PARAMS.N_tail_points;
    b->n_bottom.resize((size_t)n * 2);
    b->n_side.resize((size_t)n * 2);
    b->bottom.resize((size_t)n * 2 * b->cand_cap);
    b->side.resize((size_t)n * 2 * b->cand_cap);
    b->match_n.resize((size_t)n * 2 * b->cand_cap);
    b->match_y.resize((size_t)n * 2 * b->match_cap);
    b->match_s.resize((size_t)n * 2 * b->match_cap);
    b->tail.resize((size_t)n * 3 * b->n_tail);
    b->flags.resize(n);
    lm_results r = b->view();
    const size_t fsz = (size_t)VID_ROWS * VID_COLS;
    int on_dev = 0;
    const uint8_t *video = frames(on_dev);
    const uint8_t *prev = nullptr;
    if (first > w0) prev = video + (size_t)(first - 1 - w0) * fsz;
    else if (first > 0) {  // the previous window's last frame, kept by useWindow
        if (PREV_WINDOW != k - 1) throw std::runtime_error("readFrame(): the frame before frame " + std::to_string(first) + " was not kept.");
        prev = on_dev ? POOL->prev_decoded.p : POOL->prev.data();
    }
    check(lm_detect_batch(CTX, video + (size_t)(first - w0) * fsz, on_dev, prev, n, first, BB_X_POS.data() + first,
                          BB_Y_SIDE_POS.data() + first, BB_Y_BOTTOM_POS.data() + first, &r));
    if (!LM_PARAMS.PRIOR_PAW.empty() && !LM_PARAMS.PRIOR_SNOUT.empty()) {
        // ---- cost builders for the whole chunk (class.cpp:873-919) --------------------------------------------------
        // bottom candidates of [previous chunk's last frame | this chunk]: the halo gives the first pairwise transition
        const size_t per = (size_t)2 * b->cand_cap;
        std::vector<lm_cand> hb((size_t)(n + 1) * per);
        std::vector<int32_t> hn((size_t)(n + 1) * 2, 0);
        if (BATCH && first > 0) {
            const size_t last = BATCH->count - 1;
            std::copy(BATCH->bottom.begin() + last * per, BATCH->bottom.begin() + (last + 1) * per, hb.begin());
            hn[0] = BATCH->n_bottom[last * 2];
            hn[1] = BATCH->n_bottom[last * 2 + 1];
        }
        std::copy(b->bottom.begin(), b->bottom.end(), hb.begin() + per);
        std::copy(b->n_bottom.begin(), b->n_bottom.end(), hn.begin() + 2);
        lm_results h = r;
        h.n_frames = n + 1;
        h.bottom = hb.data();
        h.n_bottom = hn.data();
        lm_pairwise_params P{};
        const int sp = LM_PARAMS.occlusion_grid_spacing_pixels_bottom;
        P.ong_h = (int32_t)(unsigned int)(((BB_BOTTOM_MOUSE.height - sp) / sp) + 1);                                  // class.cpp:726
        P.ong_w = (int32_t)(unsigned int)(((LM_PARAMS.occlusion_grid_max_width * BB_BOTTOM_MOUSE.width) - sp) / sp + 1);  // 727
        P.grid_x = (double)(BB_BOTTOM_MOUSE.width - 1 - sp / 2);                                                        // 733
        P.grid_y = (double)(BB_BOTTOM_MOUSE.height - 1 - sp / 2);
        P.grid_spacing = (double)sp;
        P.max_displacement = (double)LM_PARAMS.max_displacement_bottom;
        P.alpha_vel = LM_PARAMS.alpha_vel_bottom;
        P.occluded_cost = LM_PARAMS.pairwise_occluded_cost;
        b->nong = P.ong_w * P.ong_h;
        for (int feat = 0; feat < 2; ++feat) {
            const std::vector<LocoMouse_LocationPrior> &pri = feat == LM_PAW ? LM_PARAMS.PRIOR_PAW : LM_PARAMS.PRIOR_SNOUT;
            std::vector<lm_location_prior> pc;
            for (const LocoMouse_LocationPrior &q : pri) pc.push_back(q.to_c());
            b->n_priors[feat] = (int)pc.size();
            b->unary[feat].assign((size_t)n * pc.size() * b->cand_cap, 0.0);
            check(lm_unary_costs(CTX, &r, n, feat, BB_BOTTOM_MOUSE.width, BB_BOTTOM_MOUSE.height, pc.data(), (int32_t)pc.size(), b->unary[feat].data()));
            b->pw_offs[feat].assign((size_t)n + 2, 0);
            b->pw_jc[feat].assign((size_t)(n + 1) * (b->cand_cap + b->nong + 1), 0);
            int64_t cap = (int64_t)(n + 1) * (2 * b->nong + 64), total = 0;
            for (int attempt = 0; attempt < 2; ++attempt) {
                b->pw_ir[feat].assign((size_t)cap, 0);
                b->pw_pr[feat].assign((size_t)cap, 0.0);
                const int rc = lm_pairwise_costs(CTX, &h, n + 1, feat, &P, b->pw_offs[feat].data(), b->pw_jc[feat].data(), b->pw_ir[feat].data(),
                                                 b->pw_pr[feat].data(), cap, &total);
                if (rc == LM_ERR_OVERFLOW && total > cap && attempt == 0) {
                    cap = total;
                    continue;
                }
                check(rc);
                break;
            }
        }
        b->has_costs = true;
    }
    SPARE = std::move(BATCH);
    BATCH = std::move(b);
}

const LocoMouse::Batch &LocoMouse::batchFor(int frame) const {
    if (!BATCH || frame < (int)BATCH->first || frame >= (int)(BATCH->first + BATCH->count))
        throw std::runtime_error("readFrame() must be called before the per-frame detection methods.");
    return *BATCH;
}

// ---- the per-frame methods (same names and order as main.cpp:57-80) ---------------------------------
void LocoMouse::readFrame() {
    if (!LOOP_READY) throw std::runtime_error("initializeFeatureLoop() must be called before readFrame().");
    if (CURRENT_FRAME + 1 >= (int)N_FRAMES) throw std::runtime_error("readFrame(): no more frames.");
    ++CURRENT_FRAME;
    if (!BATCH || CURRENT_FRAME >= (int)(BATCH->first + BATCH->count)) runChunk((unsigned int)CURRENT_FRAME);
}

void LocoMouse::cropBoundingBox() { batchFor(CURRENT_FRAME); }  // rect validity was checked by lm_detect_batch (LM_ERR_ROI)

void LocoMouse::detectTail() {
    const Batch &b = batchFor(CURRENT_FRAME);
    const size_t i = (size_t)CURRENT_FRAME - b.first, len = (size_t)3 * b.n_tail;
    TRACKS_TAIL.emplace_back(b.tail.begin() + i * len, b.tail.begin() + (i + 1) * len);
}

namespace {
std::vector<Candidate> to_candidates(const lm_cand *c, int n) {
    std::vector<Candidate> v;
    v.reserve(n);
    for (int i = 0; i < n; ++i) v.emplace_back(c[i].x, c[i].y, c[i].s);
    return v;
}
}  // namespace

void LocoMouse::detectBottomCandidates() {
    const Batch &b = batchFor(CURRENT_FRAME);
    const size_t i = (size_t)CURRENT_FRAME - b.first;
    CANDIDATES_BOTTOM_PAW.push_back(to_candidates(&b.bottom[(i * 2 + LM_PAW) * b.cand_cap], b.n_bottom[i * 2 + LM_PAW]));
    CANDIDATES_BOTTOM_SNOUT.push_back(to_candidates(&b.bottom[(i * 2 + LM_SNOUT) * b.cand_cap], b.n_bottom[i * 2 + LM_SNOUT]));
}

// computeUnaryCostsBottom / computePairwiseCostsBottom (LocoMouse_class.cpp:873-919): the MyMat / MATSPARSE inputs of the
// host tracker, built on the device for the whole chunk (lm_unary_costs / lm_pairwise_costs) and handed out per frame.
// Without a location_prior in the configuration they are skipped (the reference refuses to start without one).
void LocoMouse::computeUnaryCostsBottom() {
    const Batch &b = batchFor(CURRENT_FRAME);
    if (!b.has_costs) return;
    const size_t i = (size_t)CURRENT_FRAME - b.first;
    for (int feat = 0; feat < 2; ++feat) {
        const int nc = b.n_bottom[i * 2 + feat], np = b.n_priors[feat];
        MyMat M((unsigned int)nc, (unsigned int)np);
        for (int j = 0; j < np; ++j)
            std::copy_n(&b.unary[feat][(i * np + j) * b.cand_cap], nc, M.getValues() + (size_t)j * nc);
        (feat == LM_PAW ? UNARY_BOTTOM_PAW : UNARY_BOTTOM_SNOUT).push_back(std::move(M));
    }
}

void LocoMouse::computePairwiseCostsBottom() {
    const Batch &b = batchFor(CURRENT_FRAME);
    if (!b.has_costs || CURRENT_FRAME <= 0) return;  // class.cpp:901
    const size_t i = (size_t)CURRENT_FRAME - b.first + 1;  // index in the halo-extended chunk
    for (int feat = 0; feat < 2; ++feat) {
        const std::vector<std::vector<Candidate>> &C = feat == LM_PAW ? CANDIDATES_BOTTOM_PAW : CANDIDATES_BOTTOM_SNOUT;
        const int ni = (int)C.end()[-2].size(), nip1 = (int)C.end()[-1].size();
        const int32_t *jc = &b.pw_jc[feat][i * (b.cand_cap + b.nong + 1)];
        const int64_t o = b.pw_offs[feat][i];
        (feat == LM_PAW ? PAIRWISE_BOTTOM_PAW : PAIRWISE_BOTTOM_SNOUT)
            .push_back(MATSPARSE(nip1 + b.nong, ni + b.nong, jc, &b.pw_ir[feat][o], &b.pw_pr[feat][o]));
    }
}

void LocoMouse::detectSideCandidates() {
    const Batch &b = batchFor(CURRENT_FRAME);
    const size_t i = (size_t)CURRENT_FRAME - b.first;
    CANDIDATES_SIDE_PAW.push_back(to_candidates(&b.side[(i * 2 + LM_PAW) * b.cand_cap], b.n_side[i * 2 + LM_PAW]));
    CANDIDATES_SIDE_SNOUT.push_back(to_candidates(&b.side[(i * 2 + LM_SNOUT) * b.cand_cap], b.n_side[i * 2 + LM_SNOUT]));
}

// P22D records exactly as matchViews builds them (LocoMouse_class.cpp:1154-1251): P22D(Cb, Candidate(-1,-1,-1)) when a
// bottom candidate has no accepted side match, else P22D(Cb, first) followed by add_side_candidate for the rest.
void LocoMouse::matchBottomSideCandidates() {
    const Batch &b = batchFor(CURRENT_FRAME);
    const size_t i = (size_t)CURRENT_FRAME - b.first;
    for (int feat = 0; feat < 2; ++feat) {
        const std::vector<Candidate> &Cb = feat == LM_PAW ? CANDIDATES_BOTTOM_PAW.back() : CANDIDATES_BOTTOM_SNOUT.back();
        const int32_t *mn = &b.match_n[(i * 2 + feat) * b.cand_cap];
        const int32_t *my = &b.match_y[(i * 2 + feat) * b.match_cap];
        const double *ms = &b.match_s[(i * 2 + feat) * b.match_cap];
        std::vector<P22D> C;
        C.reserve(Cb.size());
        size_t o = 0;
        for (size_t k = 0; k < Cb.size(); ++k) {
            if (mn[k] == 0) {
                C.push_back(P22D(Cb[k], Candidate(-1, -1, -1)));
                continue;
            }
            C.push_back(P22D(Cb[k], Candidate(Cb[k].point().x, my[o], ms[o])));
            for (int q = 1; q < mn[k]; ++q) C.back().add_side_candidate(my[o + q], ms[o + q]);
            o += (size_t)mn[k];
        }
        (feat == LM_PAW ? CANDIDATES_MATCHED_VIEWS_PAW : CANDIDATES_MATCHED_VIEWS_SNOUT).push_back(std::move(C));
    }
}

void LocoMouse::storePreviousImage() {}  // the device keeps the previous raw frame (halo) itself

// computeBottomTracks / computeSideTracks / exportPointTracks / exportLineTracks: LocoMouse_tracks.cpp

// "LMO1": i32 n_frames, n_tail_points; per frame: 3*n_tail i32 tail track; then for paw, snout:
//   i32 n_bottom, n_bottom x {i32 x, y; f64 s};  i32 n_side, n_side x {i32 x, y; f64 s};
//   n_bottom x { i32 n_match, n_match x {i32 y; f64 s} }     (n_match = P22D::number_of_candidates())
void LocoMouse::exportResults() {
    exportTracks();  // output_<stem>.yml, the reference's output (LocoMouse_tracks.cpp); skipped when the tracker did not run
    lmfile::Writer w(output_file, "LMO1");
    const size_t n = CANDIDATES_MATCHED_VIEWS_PAW.size();
    w.i32((int32_t)n);
    w.i32((int32_t)LM_PARAMS.N_tail_points);
    auto put = [&](const std::vector<Candidate> &v) {
        w.i32((int32_t)v.size());
        for (const Candidate &c : v) {
            w.i32(c.p.x);
            w.i32(c.p.y);
            w.f64(c.s);
        }
    };
    for (size_t f = 0; f < n; ++f) {
        w.write(TRACKS_TAIL[f].data(), TRACKS_TAIL[f].size());
        for (int feat = 0; feat < 2; ++feat) {
            put(feat == 0 ? CANDIDATES_BOTTOM_PAW[f] : CANDIDATES_BOTTOM_SNOUT[f]);
            put(feat == 0 ? CANDIDATES_SIDE_PAW[f] : CANDIDATES_SIDE_SNOUT[f]);
            const std::vector<P22D> &P = feat == 0 ? CANDIDATES_MATCHED_VIEWS_PAW[f] : CANDIDATES_MATCHED_VIEWS_SNOUT[f];
            for (const P22D &p : P) {
                const int m = p.number_of_candidates();
                w.i32(m);
                for (int q = 0; q < m; ++q) {
                    w.i32(p.y_side_coord((uint)q));
                    w.f64(p.score_side((uint)q));
                }
            }
        }
    }
    if (!UNARY_BOTTOM_PAW.empty()) {  // the tracker's inputs, for tests and for a host match2nd: costs_<stem>.lmo
        lmfile::Writer c(costs_file, "LMC1");
        c.i32((int32_t)UNARY_BOTTOM_PAW.size());
        for (size_t f = 0; f < UNARY_BOTTOM_PAW.size(); ++f)
            for (int feat = 0; feat < 2; ++feat) {
                const MyMat &U = feat == 0 ? UNARY_BOTTOM_PAW[f] : UNARY_BOTTOM_SNOUT[f];
                c.i32(U.Nrows());
                c.i32(U.Ncols());
                c.write(U.getValues(), (size_t)U.Numel());
                if (f == 0) continue;
                const MATSPARSE &S = feat == 0 ? PAIRWISE_BOTTOM_PAW[f - 1] : PAIRWISE_BOTTOM_SNOUT[f - 1];
                c.i32(S.Nrows());
                c.i32(S.Ncols());
                c.i32(S.nz());
                c.write(S.getJc(), (size_t)S.Ncols() + 1);
                c.write(S.getIr(), (size_t)S.nz());
                c.write(S.getPr(), (size_t)S.nz());
            }
    }
}

// =====================================================================================================
// LocoMouse_Initialize (LocoMouse_Methods.cpp:3-26)
// =====================================================================================================
namespace {
template <class... A>
std::unique_ptr<LocoMouse> initialize(const LocoMouse_ParseInputs &INPUT, A &&...more) {
    std::unique_ptr<LocoMouse> L;
    int mode = 0;
    try {
        mode = std::stoi(INPUT.METHOD);
    } catch (const std::exception &) {
        throw std::invalid_argument("method must be an integer: 0 (default), 1 (TM) or 2 (TM_DE).");
    }
    switch (mode) {
        case 0: L.reset(new LocoMouse(INPUT, more...)); break;
        case 1: L.reset(new LocoMouse_TM(INPUT, more...)); break;
        case 2: L.reset(new LocoMouse_TM_DE(INPUT, more...)); break;
        default:
            std::cout << "Unknown method option. Attempting to track with the default method." << std::endl;
            L.reset(new LocoMouse(INPUT, more...));
    }
    return L;
}
}  // namespace

std::unique_ptr<LocoMouse> LocoMouse_Initialize(LocoMouse_ParseInputs INPUT) { return initialize(INPUT); }

std::unique_ptr<LocoMouse> LocoMouse_Initialize(LocoMouse_ParseInputs INPUT, const LocoMouse_Parameters &params, LocoMouse_Media &media,
                                                lm_ctx *ctx, LocoMouse_WindowPool *pool) {
    return initialize(INPUT, params, media, ctx, pool);
}
