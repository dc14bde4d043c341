// match2nd_c.cpp — plain-C entry points of the host tracker (match2nd.hpp) for the Python tests: the trellis is passed as
// packed arrays, exactly what lm_unary_costs / lm_pairwise_costs return and what the reference-compiled checker
// (oracle/ref_glue.cpp: ref_match2nd) takes, so both are driven with identical inputs.
#include <cstdint>
#include <memory>
#include <vector>

#include "cv_yaml.hpp"
#include "lm_media.hpp"
#include "match2nd.hpp"

namespace {
void build(int frames, int points, const int32_t *n_loc, const double *unary, const int64_t *unary_off, int nong, const int32_t *jc,
           const int64_t *jc_off, const int32_t *ir, const double *pr, const int64_t *nz_off, std::vector<MyMat> &U, std::vector<MATSPARSE> &P) {
    U.reserve((size_t)frames);
    for (int f = 0; f < frames; ++f) {
        MyMat M((unsigned int)n_loc[f], (unsigned int)points);
        for (int64_t i = 0; i < (int64_t)n_loc[f] * points; ++i) M.getValues()[i] = unary[unary_off[f] + i];
        U.push_back(std::move(M));
    }
    for (int f = 0; f + 1 < frames; ++f)
        P.push_back(MATSPARSE(n_loc[f + 1] + nong, n_loc[f] + nong, jc + jc_off[f], ir + nz_off[f], pr + nz_off[f]));
}
}  // namespace

extern "C" {
// unary: frame f's n_loc[f] x points column-major block at unary_off[f]; transition f: jc at jc_off[f] (n_loc[f] + nong + 1
// entries, starting at 0), ir / pr at nz_off[f].  labels: points x frames, row-major.
int lmh_match2nd(int frames, int points, const int32_t *n_loc, const double *unary, const int64_t *unary_off, int nong, const int32_t *jc,
                 const int64_t *jc_off, const int32_t *ir, const double *pr, const int64_t *nz_off, double occ_cost, double bam,
                 const int32_t *permutation, int32_t *labels) {
    std::vector<MyMat> U;
    std::vector<MATSPARSE> P;
    build(frames, points, n_loc, unary, unary_off, nong, jc, jc_off, ir, pr, nz_off, U, P);
    const cv::Mat T = match2nd(U, P, nong, occ_cost, bam, (unsigned int)frames, (unsigned int)points, permutation);
    for (int p = 0; p < points; ++p)
        for (int f = 0; f < frames; ++f) labels[(size_t)p * frames + f] = T.at<int>(p, f);
    return 0;
}
double lmh_cost_track(int frames, int points, const int32_t *n_loc, const double *unary, const int64_t *unary_off, const int32_t *permutation,
                      const int32_t *labels) {
    std::vector<MyMat> U;
    std::vector<MATSPARSE> P;
    for (int f = 0; f < frames; ++f) {
        MyMat M((unsigned int)n_loc[f], (unsigned int)points);
        for (int64_t i = 0; i < (int64_t)n_loc[f] * points; ++i) M.getValues()[i] = unary[unary_off[f] + i];
        U.push_back(std::move(M));
    }
    cv::Mat T(points, frames, CV_32SC1);
    for (int p = 0; p < points; ++p)
        for (int f = 0; f < frames; ++f) T.at<int>(p, f) = labels[(size_t)p * frames + f];
    return computeCostTrack(T, U, P, permutation);
}
// lm_track::side_view_transitions -> jc[ni + nong + 1], ir / pr [nnz]; dims = {rows, cols, nnz}
int lmh_pairwise_potential_side(const uint32_t *zi, int ni, const uint32_t *zip1, int nip1, double grid_mapping, double spacing, int nong,
                                double max_disp, double alpha_vel, double occluded_cost, int32_t *jc, int32_t *ir, double *pr, int cap, int32_t *dims) {
    const std::vector<unsigned int> A(zi, zi + ni), B(zip1, zip1 + nip1);
    const MATSPARSE S = lm_track::side_view_transitions(A, B, grid_mapping, spacing, (unsigned int)nong, max_disp, alpha_vel, occluded_cost);
    dims[0] = S.Nrows();
    dims[1] = S.Ncols();
    dims[2] = S.nz();
    if (S.nz() > cap) return 1;
    for (int c = 0; c <= S.Ncols(); ++c) jc[c] = S.getJc()[c];
    for (int k = 0; k < S.nz(); ++k) {
        ir[k] = S.getIr()[k];
        pr[k] = S.getPr()[k];
    }
    return 0;
}
// cvyaml::Writer: `n` int32 matrices (names separated by '\n', rows / cols per matrix, data back to back) into `path`
int lmh_yaml_write(const char *path, const char *names, int n, const int32_t *rows, const int32_t *cols, const int32_t *data) {
    try {
        cvyaml::Writer w(path);
        std::string all(names);
        size_t pos = 0;
        for (int i = 0; i < n; ++i) {
            const size_t e = all.find('\n', pos);
            const std::string name = all.substr(pos, e == std::string::npos ? std::string::npos : e - pos);
            pos = e == std::string::npos ? all.size() : e + 1;
            w.write(name, rows[i], cols[i], data);
            data += (size_t)rows[i] * cols[i];
        }
        return w.good() ? 0 : 1;
    } catch (const std::exception &) {
        return 2;
    }
}
// lm_media.hpp readers: dims = {n, rows, cols}; with out == NULL only the dimensions are returned.  0 ok, 1 error (msg filled)
int lmh_read_avi(const char *path, int32_t *dims, uint8_t *out, char *msg, int msg_cap) {
    try {
        const lmmedia::Video V = lmmedia::read_avi(path);
        if (V.codec == lmmedia::Codec::png) throw std::runtime_error(std::string("Video file ") + path + ": PNG-coded stream (lmh_read_avi_png)");
        if (V.codec == lmmedia::Codec::ffv1) throw std::runtime_error(std::string("Video file ") + path + ": FFV1-coded stream (lmh_read_avi_ffv1)");
        dims[0] = V.n;
        dims[1] = V.rows;
        dims[2] = V.cols;
        if (out) std::memcpy(out, V.frames.data(), V.frames.size());
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// PNG-coded video (any container index_video reads): dims = {n, rows, cols, payload bytes}; with payload / offsets NULL only the dimensions are returned,
// otherwise payload receives the frame chunks and offsets[n + 1] their bounds.  0 ok, 1 error (msg filled)
int lmh_read_avi_png(const char *path, int64_t *dims, uint8_t *payload, int64_t *offsets, char *msg, int msg_cap) {
    try {
        const lmmedia::Index ix = lmmedia::index_video(path);
        const lmmedia::Video V = lmmedia::read_frames(ix, 0, ix.n);
        if (V.codec != lmmedia::Codec::png) throw std::runtime_error(std::string("Video file ") + path + ": not a PNG-coded stream");
        dims[0] = V.n;
        dims[1] = V.rows;
        dims[2] = V.cols;
        dims[3] = V.offsets.back();
        if (payload) std::memcpy(payload, V.payload.get(), (size_t)V.offsets.back());
        if (offsets) std::memcpy(offsets, V.offsets.data(), V.offsets.size() * sizeof(int64_t));
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// FFV1-coded video (any container index_video reads): dims = {n, rows, cols, payload bytes, extradata bytes}; with payload / offsets / extradata NULL only the
// dimensions are returned.  0 ok, 1 error (msg filled)
int lmh_read_avi_ffv1(const char *path, int64_t *dims, uint8_t *payload, int64_t *offsets, uint8_t *extradata, char *msg, int msg_cap) {
    try {
        const lmmedia::Index ix = lmmedia::index_video(path);
        const lmmedia::Video V = lmmedia::read_frames(ix, 0, ix.n);
        if (V.codec != lmmedia::Codec::ffv1) throw std::runtime_error(std::string("Video file ") + path + ": not an FFV1-coded stream");
        dims[0] = V.n;
        dims[1] = V.rows;
        dims[2] = V.cols;
        dims[3] = V.offsets.back();
        dims[4] = (int64_t)V.extradata.size();
        if (payload) std::memcpy(payload, V.payload.get(), (size_t)V.offsets.back());
        if (offsets) std::memcpy(offsets, V.offsets.data(), V.offsets.size() * sizeof(int64_t));
        if (extradata) std::memcpy(extradata, V.extradata.data(), V.extradata.size());
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// Frames [first, first + count) of a video (AVI, Matroska, QuickTime / MP4, LMV1) through lmmedia::index_video + read_frames: dims = {n (whole video),
// rows, cols, codec (0 raw, 1 PNG, 2 FFV1), bytes of the range}.  out receives the pixels (raw) or the frame chunks (coded, with
// offsets[count + 1] relative to the first); with out NULL only dims are returned.  0 ok, 1 error (msg filled)
int lmh_read_avi_range(const char *path, int64_t first, int64_t count, int64_t *dims, uint8_t *out, int64_t *offsets, char *msg, int msg_cap) {
    try {
        const lmmedia::Index ix = lmmedia::index_video(path);
        dims[0] = ix.n;
        dims[1] = ix.rows;
        dims[2] = ix.cols;
        dims[3] = (int64_t)ix.codec;
        dims[4] = 0;
        if (count <= 0) return 0;
        const lmmedia::Video V = lmmedia::read_frames(ix, (int)first, (int)count);
        dims[4] = V.codec == lmmedia::Codec::raw ? (int64_t)V.frames.size() : V.offsets.back();
        if (out) std::memcpy(out, V.codec == lmmedia::Codec::raw ? V.frames.data() : V.payload.get(), (size_t)dims[4]);
        if (offsets && V.codec != lmmedia::Codec::raw) std::memcpy(offsets, V.offsets.data(), V.offsets.size() * sizeof(int64_t));
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// The windows LocoMouse streams a video through for a budget of max_bytes frame bytes and batch_frames: starts[] receives
// the first frame of each window, then the number of frames.  Returns the number of windows, or -1 (msg filled).
int lmh_plan_windows(const char *path, int64_t max_bytes, int batch_frames, int32_t *starts, int cap, char *msg, int msg_cap) {
    try {
        const lmmedia::Index ix = lmmedia::index_video(path);
        const int W = lmmedia::window_frames((size_t)max_bytes, (size_t)ix.rows * ix.cols, batch_frames);
        const std::vector<int> s = lmmedia::plan_windows(ix.n, W, ix.keyframe);
        for (size_t i = 0; i < s.size() && (int)i < cap; ++i) starts[i] = s[i];
        return (int)s.size() - 1;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return -1;
    }
}
// ffv1_format.h run serially on the CPU: the record parse and the chain decode that k_ffv1.cu runs per thread, for the CPU
// tests.  out: [n][rows][cols].  0 ok, 1 error (msg names the record problem, or the first bad frame and slice)
int lmh_decode_ffv1(const uint8_t *extradata, int64_t extradata_len, const uint8_t *payload, const int64_t *offsets, int64_t n, int rows,
                    int cols, uint8_t *out, char *msg, int msg_cap) {
    auto *rec = new ffv1::Record;
    std::unique_ptr<ffv1::Record> hold(rec);
    char why[200];
    int64_t ib = 0;
    if (ffv1::parse_record(extradata, extradata_len, rows, cols, *rec, nullptr, &ib, why, sizeof why)) {
        std::snprintf(msg, (size_t)msg_cap, "%s", why);
        return 1;
    }
    std::vector<uint8_t> initial((size_t)ib);
    ffv1::parse_record(extradata, extradata_len, rows, cols, *rec, initial.data(), &ib, why, sizeof why);
    const int S = rec->slices();
    std::vector<int64_t> soff((size_t)(n * S));
    std::vector<int32_t> slen((size_t)(n * S)), status((size_t)(n * S), -1);
    uint32_t ct[256];
    ffv1::crc_table(ct);
    for (int64_t f = 0; f < n; ++f) {
        const uint8_t *fr = payload + offsets[f];
        if (ffv1::locate_slices(fr, offsets[f + 1] - offsets[f], S, rec->ec, &soff[f * S], &slen[f * S])) {
            for (int s = 0; s < S; ++s) status[f * S + s] = ffv1::LM_FFV1_FOOTER;
            continue;
        }
        for (int s = 0; s < S; ++s) {
            soff[f * S + s] += offsets[f];
            uint32_t crc = 0;
            for (int32_t i = 0; rec->ec && i < slen[f * S + s]; ++i) crc = ffv1::crc_update(ct, crc, payload[soff[f * S + s] + i]);
            if (crc) status[f * S + s] = ffv1::LM_FFV1_CRC;
        }
    }
    std::vector<uint64_t> work((size_t)(ffv1::work_bytes(*rec, cols) + 7) / 8);
    for (int64_t f0 = 0; f0 < n;) {
        int64_t f1 = f0 + 1;
        while (f1 < n && !ffv1::keyframe_bit(payload + offsets[f1], offsets[f1 + 1] - offsets[f1])) ++f1;
        if (f0 == 0 && !ffv1::keyframe_bit(payload, offsets[1] - offsets[0])) {
            std::snprintf(msg, (size_t)msg_cap, "frame 0 is not a keyframe");
            return 1;
        }
        for (int s = 0; s < S; ++s) {
            if (rec->ac)
                ffv1::decode_chain<true>(*rec, rec->t, initial.data(), payload, soff.data(), slen.data(), status.data(), out, rows, cols, f0,
                                         (int)(f1 - f0), s, reinterpret_cast<uint8_t *>(work.data()));
            else
                ffv1::decode_chain<false>(*rec, rec->t, initial.data(), payload, soff.data(), slen.data(), status.data(), out, rows, cols, f0,
                                          (int)(f1 - f0), s, reinterpret_cast<uint8_t *>(work.data()));
        }
        f0 = f1;
    }
    for (int64_t i = 0; i < n * S; ++i)
        if (status[i]) {
            std::snprintf(msg, (size_t)msg_cap, "frame %lld, slice %d: %s", (long long)(i / S), (int)(i % S), ffv1::status_text(status[i]));
            return 1;
        }
    return 0;
}
// Motion-JPEG video (any container index_video reads) with decode_mjpeg on: dims = {n, rows, cols, payload bytes}; with
// payload / offsets NULL only the dimensions are returned.  0 ok, 1 error (msg filled)
int lmh_read_video_mjpeg(const char *path, int64_t *dims, uint8_t *payload, int64_t *offsets, char *msg, int msg_cap) {
    try {
        lmmedia::Options opt;
        opt.decode_mjpeg = true;
        const lmmedia::Index ix = lmmedia::index_video(path, opt);
        const lmmedia::Video V = lmmedia::read_frames(ix, 0, ix.n);
        if (V.codec != lmmedia::Codec::mjpeg) throw std::runtime_error(std::string("Video file ") + path + ": not a Motion-JPEG stream");
        dims[0] = V.n;
        dims[1] = V.rows;
        dims[2] = V.cols;
        dims[3] = V.offsets.back();
        if (payload) std::memcpy(payload, V.payload.get(), (size_t)V.offsets.back());
        if (offsets) std::memcpy(offsets, V.offsets.data(), V.offsets.size() * sizeof(int64_t));
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// lmh_read_avi_range with decode_mjpeg on (codec 3 = Motion-JPEG)
int lmh_read_avi_range_mjpeg(const char *path, int64_t first, int64_t count, int64_t *dims, uint8_t *out, int64_t *offsets, char *msg,
                             int msg_cap) {
    try {
        lmmedia::Options opt;
        opt.decode_mjpeg = true;
        const lmmedia::Index ix = lmmedia::index_video(path, opt);
        dims[0] = ix.n;
        dims[1] = ix.rows;
        dims[2] = ix.cols;
        dims[3] = (int64_t)ix.codec;
        dims[4] = 0;
        if (count <= 0) return 0;
        const lmmedia::Video V = lmmedia::read_frames(ix, (int)first, (int)count);
        dims[4] = V.codec == lmmedia::Codec::raw ? (int64_t)V.frames.size() : V.offsets.back();
        if (out) std::memcpy(out, V.codec == lmmedia::Codec::raw ? V.frames.data() : V.payload.get(), (size_t)dims[4]);
        if (offsets && V.codec != lmmedia::Codec::raw) std::memcpy(offsets, V.offsets.data(), V.offsets.size() * sizeof(int64_t));
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// mjpeg_format.h run serially on the CPU: the header parse, entropy decode and IDCT that k_mjpeg.cu runs on the device, for
// the CPU tests.  out: [n][rows][cols].  0 ok, 1 error (msg names the first bad frame and why)
int lmh_decode_mjpeg(const uint8_t *payload, const int64_t *offsets, int64_t n, int rows, int cols, uint8_t *out, char *msg, int msg_cap) {
    std::unique_ptr<mjpeg::Header> hold(new mjpeg::Header);
    mjpeg::Header &h = *hold;
    std::vector<uint16_t> fast((size_t)4 << mjpeg::FAST_BITS);
    std::vector<int16_t> coef;
    int dht0 = -1;  // the tables frame 0's DHT defines: every frame must define the same (libavcodec carries them over)
    for (int64_t f = 0; f < n; ++f) {
        const uint8_t *fr = payload + offsets[f];
        const int64_t len = offsets[f + 1] - offsets[f];
        int st = mjpeg::parse(fr, len, rows, cols, h);
        for (int t = 0; t < 4 && st == mjpeg::LM_MJPEG_OK; ++t)
            if (!mjpeg::build_fast(h.tab[t], fast.data() + ((size_t)t << mjpeg::FAST_BITS))) st = mjpeg::LM_MJPEG_TABLE;
        if (st == mjpeg::LM_MJPEG_OK && f == 0) dht0 = h.dht_mask;
        if (st == mjpeg::LM_MJPEG_OK && h.dht_mask != dht0) st = mjpeg::LM_MJPEG_DHT_CHANGE;
        if (st == mjpeg::LM_MJPEG_OK) {
            coef.assign((size_t)h.blocks() * 64, 0);
            st = mjpeg::decode_scan(h, fr + h.ecs, fr + len, fast.data(),
                                    [&](int64_t b, const int16_t *blk) { std::memcpy(&coef[(size_t)b * 64], blk, 64 * sizeof(int16_t)); });
        }
        if (st != mjpeg::LM_MJPEG_OK) {
            std::snprintf(msg, (size_t)msg_cap, "frame %lld: %s", (long long)f, mjpeg::status_text(st));
            return 1;
        }
        for (int by = 0; by < h.y_blocks_y(); ++by)
            for (int bx = 0; bx < h.y_blocks_x(); ++bx) mjpeg::put_y_block(h, coef.data(), by, bx, out + f * (int64_t)rows * cols);
    }
    return 0;
}
// MPEG-4 Part 2 video (any container index_video reads) with decode_mpeg4 on: dims = {n, rows, cols, payload bytes,
// extradata bytes}; with payload / offsets / extradata NULL only the dimensions are returned; ivop (optional, n bytes):
// each frame's I-VOP bit.  0 ok, 1 error (msg filled)
int lmh_read_video_mpeg4(const char *path, int64_t *dims, uint8_t *payload, int64_t *offsets, uint8_t *extradata, uint8_t *ivop, char *msg,
                         int msg_cap) {
    try {
        lmmedia::Options opt;
        opt.decode_mpeg4 = true;
        const lmmedia::Index ix = lmmedia::index_video(path, opt);
        const lmmedia::Video V = lmmedia::read_frames(ix, 0, ix.n);
        if (V.codec != lmmedia::Codec::mpeg4) throw std::runtime_error(std::string("Video file ") + path + ": not an MPEG-4 Part 2 stream");
        dims[0] = V.n;
        dims[1] = V.rows;
        dims[2] = V.cols;
        dims[3] = V.offsets.back();
        dims[4] = (int64_t)ix.extradata.size();
        if (payload) std::memcpy(payload, V.payload.get(), (size_t)V.offsets.back());
        if (offsets) std::memcpy(offsets, V.offsets.data(), V.offsets.size() * sizeof(int64_t));
        if (extradata && !ix.extradata.empty()) std::memcpy(extradata, ix.extradata.data(), ix.extradata.size());
        if (ivop) std::memcpy(ivop, ix.keyframe.data(), ix.keyframe.size());
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// mpeg4_format.h run serially on the CPU: the header parse, macroblock decode and reconstruction that k_mpeg4.cu runs on the
// device, for the CPU tests.  out: [n][rows][cols].  0 ok, 1 error (msg names the first bad frame and why)
int lmh_decode_mpeg4(const uint8_t *extradata, int64_t extradata_len, const uint8_t *payload, const int64_t *offsets, int64_t n, int rows,
                     int cols, uint8_t *out, char *msg, int msg_cap) {
    static const std::unique_ptr<mpeg4::Tables> tables = [] {
        std::unique_ptr<mpeg4::Tables> t(new mpeg4::Tables);
        mpeg4::build_tables(*t, 0, 0, 1);
        mpeg4::build_tables(*t, 1, 0, 1);
        return t;
    }();
    const int mbw = (cols + 15) / 16, mbh = (rows + 15) / 16;
    auto fail = [&](int64_t f, int st) {
        std::snprintf(msg, (size_t)msg_cap, "frame %lld: %s", (long long)f, mpeg4::status_text(st));
        return 1;
    };
    mpeg4::Vol vol{};
    mpeg4::Vop vop{};
    if (extradata_len > 0)
        if (int st = mpeg4::parse(extradata, extradata_len, rows, cols, false, vol, vop)) {
            std::snprintf(msg, (size_t)msg_cap, "extradata: %s", mpeg4::status_text(st));
            return 1;
        }
    std::vector<uint8_t> ref((size_t)mbw * mbh * 320), cur(ref.size()), lines((size_t)mpeg4::lines_bytes(mbw));
    std::vector<mpeg4::MbInfo> info((size_t)mbw * mbh);
    std::vector<int16_t> coef((size_t)mbw * mbh * mpeg4::BLOCKS_PER_MB * 64);
    for (int64_t f = 0; f < n; ++f) {
        const uint8_t *fr = payload + offsets[f];
        const int64_t len = offsets[f + 1] - offsets[f];
        int st = mpeg4::parse(fr, len, rows, cols, true, vol, vop);
        if (st == mpeg4::LM_MPEG4_OK && vop.type == mpeg4::VOP_N) st = mpeg4::LM_MPEG4_NOT_CODED;
        if (st == mpeg4::LM_MPEG4_OK && f == 0 && vop.type != mpeg4::VOP_I) st = mpeg4::LM_MPEG4_FIRST_NOT_I;
        if (st == mpeg4::LM_MPEG4_OK)
            st = mpeg4::decode_vop(
                *tables, vop, mbw, mbh, fr, len, mpeg4::lines_at(lines.data(), mbw), [&](int mb, const mpeg4::MbInfo &mi) { info[(size_t)mb] = mi; },
                [&](int mb, int b, const int16_t *blk) { std::memcpy(&coef[((size_t)mb * mpeg4::BLOCKS_PER_MB + b) * 64], blk, 64 * sizeof(int16_t)); });
        if (st != mpeg4::LM_MPEG4_OK) return fail(f, st);
        uint8_t *cy = cur.data(), *cc = cy + (size_t)mbw * mbh * 256;
        for (int my = 0; my < mbh; ++my)
            for (int mx = 0; mx < mbw; ++mx)
                mpeg4::build_mb(mbw, mbh, mx, my, info[(size_t)(my * mbw + mx)], &coef[(size_t)(my * mbw + mx) * mpeg4::BLOCKS_PER_MB * 64],
                                vop.rounding, ref.data(), ref.data() + (size_t)mbw * mbh * 256, cy, cc);
        for (int my = 0; my < mbh; ++my)
            for (int mx = 0; mx < mbw; ++mx) mpeg4::put_mb(mbw, mx, my, cy, cc, rows, cols, out + f * (int64_t)rows * cols);
        std::swap(ref, cur);
    }
    return 0;
}
// lmh_plan_windows with decode_mpeg4 on: MPEG-4 windows end before an I-VOP
int lmh_plan_windows_mpeg4(const char *path, int64_t max_bytes, int batch_frames, int32_t *starts, int cap, char *msg, int msg_cap) {
    try {
        lmmedia::Options opt;
        opt.decode_mpeg4 = true;
        const lmmedia::Index ix = lmmedia::index_video(path, opt);
        const int W = lmmedia::window_frames((size_t)max_bytes, (size_t)ix.rows * ix.cols, batch_frames);
        const std::vector<int> s = lmmedia::plan_windows(ix.n, W, ix.keyframe);
        for (size_t i = 0; i < s.size() && (int)i < cap; ++i) starts[i] = s[i];
        return (int)s.size() - 1;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return -1;
    }
}
// mpeg4::blue for every (Y, Cb): table[Y * 256 + Cb]
void lmh_mpeg4_blue(uint8_t *table) {
    for (int y = 0; y < 256; ++y)
        for (int c = 0; c < 256; ++c) table[y * 256 + c] = mpeg4::blue(y, c);
}
// (last, run, level) of TCOEF symbol s (< 102) of the intra (intra = 1) or inter table, for the tests' encoder
void lmh_mpeg4_tcoef_event(int intra, int s, int32_t *lrl) {
    int last, run, level;
    mpeg4::tcoef_event(intra, s, last, run, level);
    lrl[0] = last, lrl[1] = run, lrl[2] = level;
}
// {code, length} of every symbol of VLC table t of mpeg4_format.h (codes, lens: mpeg4::count(t) entries); returns the count
int lmh_mpeg4_vlc(int t, int32_t *codes, int32_t *lens) {
    if (t < 0 || t >= mpeg4::T_COUNT) return 0;
    for (int s = 0; s < mpeg4::count(t); ++s) {
        int c, l;
        mpeg4::code(t, s, c, l);
        codes[s] = c;
        lens[s] = l;
    }
    return mpeg4::count(t);
}
int lmh_read_png(const char *path, int32_t *dims, uint8_t *out, char *msg, int msg_cap) {
    try {
        const lmmedia::Image I = lmmedia::read_png_gray(path);
        dims[0] = 1;
        dims[1] = I.rows;
        dims[2] = I.cols;
        if (out) std::memcpy(out, I.px.data(), I.px.size());
        return 0;
    } catch (const std::exception &e) {
        if (msg && msg_cap > 0) std::snprintf(msg, (size_t)msg_cap, "%s", e.what());
        return 1;
    }
}
// the same job `copies` times on `threads` host threads; returns 1 when every result equals the serial one
int lmh_match2nd_concurrent_check(int frames, int points, const int32_t *n_loc, const double *unary, const int64_t *unary_off, int nong,
                                  const int32_t *jc, const int64_t *jc_off, const int32_t *ir, const double *pr, const int64_t *nz_off, double occ_cost,
                                  double bam, const int32_t *permutation, int copies, int threads) {
    std::vector<MyMat> U;
    std::vector<MATSPARSE> P;
    build(frames, points, n_loc, unary, unary_off, nong, jc, jc_off, ir, pr, nz_off, U, P);
    const cv::Mat T = match2nd(U, P, nong, occ_cost, bam, (unsigned int)frames, (unsigned int)points, permutation);
    std::vector<lm_track::Job> jobs((size_t)copies);
    for (lm_track::Job &j : jobs) {
        j.unary = &U;
        j.pairwise = &P;
        j.Nong = nong;
        j.occlusion_point_cost = occ_cost;
        j.bam_tie = bam;
        j.frames = (unsigned int)frames;
        j.points = (unsigned int)points;
        j.permutation = permutation;
    }
    lm_track::match2nd_concurrent(jobs, (unsigned int)threads);
    for (const lm_track::Job &j : jobs)
        for (int p = 0; p < points; ++p)
            for (int f = 0; f < frames; ++f)
                if (j.result.at<int>(p, f) != T.at<int>(p, f)) return 0;
    return 1;
}
}
