// lm_media.hpp — the reference's own input media, read without OpenCV (SURVEY §8f-3):
//   video       cv::VideoCapture + extractChannel(F, F, 0)   (LocoMouse_class.cpp:367-400, 1282-1293)
//   background  cv::imread(file, CV_LOAD_IMAGE_GRAYSCALE)    (LocoMouse_class.cpp:402-417)
// Video: AVI (RIFF, also OpenDML 'AVIX' extensions) whose stream 0 holds UNCOMPRESSED frames -- 8-bit grey ('Y800' /
// 'GREY' / 'Y8  ', what cv2.VideoWriter(fourcc = 0, isColor = False) writes), BI_RGB 8-bit with a palette, BI_RGB 24- / 32-bit
// (channel 0 = blue, as extractChannel takes it).  PNG-coded streams ('MPNG' / 'png ', lossless, what cv2.VideoWriter writes
// with those fourccs) are not decoded here: their frame chunks -- each a complete PNG file -- are returned as one payload with
// offsets, for lm_decode_png to decode on the device.  Motion-JPEG streams are returned the same way for lm_decode_mjpeg when
// the caller opts in (Options::decode_mjpeg), and MPEG-4 Part 2 streams for lm_decode_mpeg4 with their VOL as extradata
// (Options::decode_mpeg4; every frame's VOP header is checked and its I-VOP bit recorded); otherwise they are refused like
// every other lossy codec.  FFV1-coded streams ('FFV1', lossless, version 3 as libavcodec writes
// it) are returned the same way, with the configuration record from 'strf' as extradata, for lm_decode_ffv1; the record is
// checked here (ffv1_format.h) and so is every frame's keyframe bit.  Other compressed or YUV-planar streams need a decoder
// that is outside this library: they are refused with a message that says so.  The same frames in Matroska and QuickTime / MP4
// files are indexed by lm_containers.hpp into the same Index; index_video picks the container by signature (AVI, Matroska,
// ISO BMFF, LMV1).  Background: PNG, 8 bits per channel, non-interlaced; colour images are
// reduced to grey as libpng does for OpenCV (png_set_rgb_to_gray with 0.299 / 0.587).  Both are checked against what the
// real OpenCV reads from the same files (tests/test_host_media.py).  A video is read in two steps, so that a long one can be
// streamed: index_avi (index_mkv, index_mov) walks the file's structure once, read_frames reads any range of frames
// (tests/test_avi_ranges.py, tests/test_containers.py).
#pragma once
#include <zlib.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../csrc/ffv1_format.h"
#include "../csrc/mjpeg_format.h"
#include "../csrc/mpeg4_format.h"

namespace lmmedia {

inline std::vector<uint8_t> slurp(const std::string &name, size_t limit = 0) {
    FILE *f = std::fopen(name.c_str(), "rb");
    if (!f) throw std::runtime_error("Cannot open file: " + name);
    std::vector<uint8_t> d;
    uint8_t buf[1 << 16];
    size_t n;
    while ((n = std::fread(buf, 1, sizeof buf, f)) > 0) {
        d.insert(d.end(), buf, buf + n);
        if (limit && d.size() >= limit) break;
    }
    std::fclose(f);
    return d;
}
inline uint32_t le32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline uint32_t be32(const uint8_t *p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3]; }
inline bool is_avi(const std::string &name) {
    const std::vector<uint8_t> h = slurp(name, 12);
    return h.size() >= 12 && !std::memcmp(h.data(), "RIFF", 4) && !std::memcmp(h.data() + 8, "AVI ", 4);
}
inline bool is_png(const std::string &name) {
    const std::vector<uint8_t> h = slurp(name, 8);
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    return h.size() >= 8 && !std::memcmp(h.data(), sig, 8);
}

// Where read_avi puts the pixels of an uncompressed stream or the frame chunks of a coded one: a buffer of the requested size
// that the caller owns (the class mirror passes pooled page-locked memory, so that the frames are read from the file straight
// into memory the upload runs from at the PCIe rate).  Without one they go to Video::frames / a malloc'ed Video::payload.
using Dest = std::function<uint8_t *(size_t bytes)>;

enum class Codec { raw, png, ffv1, mjpeg, mpeg4 };

// What the index functions accept beyond the lossless codecs.  Motion-JPEG is decoded bit-exactly with the libavcodec
// decoder OpenCV calls (mjpeg_format.h), so a caller whose reference reads it through another decoder turns it on knowingly.
struct Options {
    bool decode_mjpeg = false;  // Motion-JPEG (AVI 'MJPG', Matroska V_MJPEG, QuickTime 'jpeg', MP4 object type 0x6C) instead of a refusal
    // MPEG-4 Part 2 (AVI 'XVID' / 'DIVX' / 'DX50' / 'FMP4' / 'MP4V', Matroska V_MPEG4/ISO/SP and ASP, MP4 'mp4v' object type
    // 0x20) decoded bit-exactly with libavcodec's mpeg4 decoder (mpeg4_format.h), instead of a refusal
    bool decode_mpeg4 = false;
};

// AVI / VfW fourccs of MPEG-4 Part 2 video
inline bool mpeg4_fourcc(uint32_t fourcc) {
    for (const char *s : {"XVID", "xvid", "DIVX", "DX50", "FMP4", "MP4V", "mp4v"})
        if (fourcc == le32(reinterpret_cast<const uint8_t *>(s))) return true;
    return false;
}

// What a refusal of MPEG-4 Part 2 video without decode_mpeg4 adds
inline const char *mpeg4_opt_in() {
    return " MPEG-4 Part 2 video is decoded with the configuration key decode_mpeg4: 1 (bit-exact with libavcodec's decoder).";
}

struct Video {
    int n = 0, rows = 0, cols = 0;
    std::vector<uint8_t> frames;  // channel 0 of every frame, [n][rows][cols] (uncompressed streams read without a Dest)
    // Compressed streams: frame i = payload[offsets[i], offsets[i + 1]), one frame chunk (a complete PNG file, or one FFV1
    // frame whose configuration record is `extradata`); `frames` stays empty
    Codec codec = Codec::raw;
    std::shared_ptr<uint8_t> payload;
    std::vector<int64_t> offsets;
    std::vector<uint8_t> extradata;
};

// Signature and IHDR of one PNG frame: 8-bit grey / RGB / RGBA, not interlaced (what lm_decode_png decodes)
inline void check_png_frame(const uint8_t *d, size_t len, int &rows, int &cols, const std::string &where) {
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    auto fail = [&](const std::string &why) { throw std::runtime_error(where + ": " + why); };
    if (len < 45 || std::memcmp(d, sig, 8) || be32(d + 8) != 13 || std::memcmp(d + 12, "IHDR", 4)) fail("not a PNG image");
    const int w = (int)be32(d + 16), h = (int)be32(d + 20), depth = d[24], ct = d[25];
    if (depth != 8 || (ct != 0 && ct != 2 && ct != 6))
        fail("bit depth " + std::to_string(depth) + ", colour type " + std::to_string(ct) +
             ": only 8-bit grey, RGB and RGBA PNG frames are decoded (no 16-bit or palette frames)");
    if (d[26] || d[27]) fail("unknown PNG compression or filter method");
    if (d[28]) fail("interlaced PNG frames are not decoded");
    if (w <= 0 || h <= 0) fail("empty image");
    if (rows == 0) rows = h, cols = w;
    else if (h != rows || w != cols)
        fail(std::to_string(w) + " x " + std::to_string(h) + " pixels, frame 0 has " + std::to_string(cols) + " x " + std::to_string(rows));
}

// Header segments of one Motion-JPEG frame up to its SOS: what lm_decode_mjpeg decodes.  Its SOF size must be the video's
// rows x cols (rows = 0: any, and it becomes the video's), and its DHT must define the tables the video's first frame
// defines (dht < 0: any, and its set becomes the video's), because libavcodec carries tables from one frame to the next.
inline void check_mjpeg_frame(const uint8_t *d, size_t len, int &rows, int &cols, int &dht, const std::string &where) {
    std::unique_ptr<mjpeg::Header> h(new mjpeg::Header);
    const int st = mjpeg::parse(d, (int64_t)len, 0, 0, *h);
    if (st != mjpeg::LM_MJPEG_OK) throw std::runtime_error(where + ": " + mjpeg::status_text(st));
    if (rows && (h->rows != rows || h->cols != cols))
        throw std::runtime_error(where + ": " + mjpeg::status_text(mjpeg::LM_MJPEG_SIZE) + ": the frame is " + std::to_string(h->cols) + " x " +
                                 std::to_string(h->rows) + " pixels (SOF), the video " + std::to_string(cols) + " x " + std::to_string(rows));
    if (dht >= 0 && h->dht_mask != dht) throw std::runtime_error(where + ": " + mjpeg::status_text(mjpeg::LM_MJPEG_DHT_CHANGE));
    rows = h->rows;
    cols = h->cols;
    dht = h->dht_mask;
}

// Where every frame of a video lies in its file: the result of one walk over the chunk headers (index_avi, or index_lmv for
// the LMV1 container of lm_files.hpp), from which read_frames reads any range of frames.  Every chunk is checked against the
// file size here, so a truncated chunk is refused before any frame is used, wherever it lies.
struct Index {
    std::string name;
    int n = 0, rows = 0, cols = 0;
    Codec codec = Codec::raw;
    // uncompressed frames: chunk position, size and row stride; channel-0 extraction as extractChannel(F, F, 0) takes it
    struct RawChunk {
        int64_t at;
        uint32_t size;
        size_t stride;
    };
    std::vector<RawChunk> raw;
    int bpp = 1, channel0 = 0;  // bytes per pixel; byte of channel 0 in a pixel (2 where a container stores RGB, not BGR)
    bool grey = true, bottom_up = false;
    uint8_t palette_b[256] = {};
    // coded frames: file offset and size of every frame chunk; FFV1: every frame's keyframe bit and the configuration record
    std::vector<std::pair<int64_t, uint32_t>> coded;
    std::vector<uint8_t> keyframe, extradata;
    int mjpeg_dht = -1;  // Motion-JPEG: the tables frame 0's DHT defines (mjpeg::Header::dht_mask), which every frame must match
    // MPEG-4 Part 2: the container's fourcc (AVI / VfW, 0 elsewhere); keyframe holds every frame's I-VOP bit and extradata
    // the VOL (the container's, or the headers in front of frame 0's VOP)
    uint32_t fourcc = 0;
};

namespace detail {
struct File {
    FILE *f;
    explicit File(const std::string &name) : f(std::fopen(name.c_str(), "rb")) {
        if (!f) throw std::runtime_error("Cannot open file: " + name);
    }
    ~File() { std::fclose(f); }
    bool read(void *dst, size_t n) { return std::fread(dst, 1, n, f) == n; }
    bool seek(int64_t at) { return fseeko(f, (off_t)at, SEEK_SET) == 0; }
    int64_t size() { return fseeko(f, 0, SEEK_END) == 0 ? (int64_t)ftello(f) : -1; }
};
}  // namespace detail

// Every MPEG-4 frame's headers up to its VOP header: the VOL (the container's extradata, else the frame's) is the one
// mpeg4_format.h decodes, of the container's size, the same in every frame; the VOP is I or P, frame 0 an I-VOP.  A
// not-coded VOP is left out, as a zero-size AVI chunk is: libavcodec returns no frame for it, so VideoCapture reads one frame
// less.  Records the I-VOP bits (windows end before one) and, where the container has no extradata, the headers in front of
// frame 0's VOP as extradata, so that every window's decode has the VOL.  libavcodec decodes an 'XVID' or 'DIVX' stream without
// libavcodec's user data with XviD's IDCT and bug workarounds, so such streams are refused.
inline void index_mpeg4(Index &V, detail::File &file) {
    auto fail = [&](const std::string &why) -> void { throw std::runtime_error("Video file " + V.name + ": " + why); };
    if (V.rows <= 0 || V.cols <= 0) fail("the video track has no frame size");
    mpeg4::Vol vol{};
    mpeg4::Vop vop{};
    if (!V.extradata.empty())
        if (int st = mpeg4::parse(V.extradata.data(), (int64_t)V.extradata.size(), V.rows, V.cols, false, vol, vop))
            fail(std::string("MPEG-4 extradata: ") + mpeg4::status_text(st));
    auto lavc = [](const uint8_t *d, size_t n) {
        for (size_t i = 0; i + 8 <= n; ++i)
            if (d[i] == 0 && d[i + 1] == 0 && d[i + 2] == 1 && d[i + 3] == 0xB2 && !std::memcmp(d + i + 4, "Lavc", 4)) return true;
        return false;
    };
    bool lavc_seen = lavc(V.extradata.data(), V.extradata.size());
    V.keyframe.clear();
    std::vector<std::pair<int64_t, uint32_t>> kept;
    std::vector<uint8_t> d;
    for (size_t i = 0; i < V.coded.size(); ++i) {
        // the headers in front of the VOP's macroblocks: a prefix of the frame, or all of it when the prefix ends too soon
        const std::string where = "Video file " + V.name + ", frame " + std::to_string(i);
        size_t len = std::min<size_t>(V.coded[i].second, 512);
        for (int pass = 0; pass < 2; ++pass) {
            d.resize(len);
            if (!file.seek(V.coded[i].first) || !file.read(d.data(), len)) fail("truncated frame");
            const int st = mpeg4::parse(d.data(), (int64_t)len, V.rows, V.cols, true, vol, vop);
            if (st == mpeg4::LM_MPEG4_OK && (vop.data_bit >> 3) + 8 <= (int64_t)len) break;
            if (len == V.coded[i].second) {
                if (st) throw std::runtime_error(where + ": " + mpeg4::status_text(st));
                break;
            }
            len = V.coded[i].second;
        }
        if (vop.type == mpeg4::VOP_N) continue;
        V.keyframe.push_back(vop.type == mpeg4::VOP_I);
        kept.push_back(V.coded[i]);
        if (kept.size() == 1) {
            if (vop.type != mpeg4::VOP_I) throw std::runtime_error(where + ": " + mpeg4::status_text(mpeg4::LM_MPEG4_FIRST_NOT_I));
            lavc_seen = lavc_seen || lavc(d.data(), d.size());
            if (V.extradata.empty()) {  // everything in front of the VOP start code
                const int64_t vop_at = (vop.data_bit >> 3);
                int64_t e = 0;
                for (int64_t p = 0; p + 3 < vop_at; ++p)
                    if (d[p] == 0 && d[p + 1] == 0 && d[p + 2] == 1 && d[p + 3] == 0xB6) e = p;
                V.extradata.assign(d.begin(), d.begin() + e);
            }
        }
    }
    V.coded.swap(kept);
    V.n = (int)V.coded.size();
    auto cc = [](const char *s) { return le32(reinterpret_cast<const uint8_t *>(s)); };
    uint32_t upper = V.fourcc;  // libavcodec compares the codec tag upper-cased (ff_toupper4)
    for (int k = 0; k < 4; ++k) {
        const uint32_t c = (upper >> (8 * k)) & 255;
        if (c >= 'a' && c <= 'z') upper -= (uint32_t)('a' - 'A') << (8 * k);
    }
    if ((upper == cc("XVID") || upper == cc("DIVX")) && !lavc_seen)
        fail("'" + std::string(reinterpret_cast<const char *>(&V.fourcc), 4) +
             "' MPEG-4 video without libavcodec's user data: libavcodec decodes it with XviD's IDCT and bug workarounds, which "
             "are not restated here");
}

// The checks every container's index ends with (index_avi, index_mkv, index_mov), once V.n, the codec, the chunks and the
// record are set: every chunk lies inside the file, also the bytes behind the image area that are not read; an FFV1 stream's
// record parses and every frame's keyframe bit is recorded, frame 0's set; a PNG stream's size is frame 0's IHDR.
inline void finish_index(Index &V, detail::File &file) {
    auto fail = [&](const std::string &why) -> void { throw std::runtime_error("Video file " + V.name + ": " + why); };
    const int64_t file_bytes = file.size();
    if (file_bytes < 0) fail("truncated frame");
    for (const Index::RawChunk &c : V.raw)
        if (c.at + (int64_t)c.size > file_bytes) fail("truncated frame");
    for (const auto &c : V.coded)
        if (c.first + (int64_t)c.second > file_bytes) fail("truncated frame");
    if (V.codec == Codec::ffv1) {
        ffv1::Record rec;
        char why[200];
        if (ffv1::parse_record(V.extradata.data(), (int64_t)V.extradata.size(), V.rows, V.cols, rec, nullptr, nullptr, why, sizeof why))
            fail(std::string("FFV1 configuration record: ") + why);
        V.keyframe.resize(V.coded.size());
        for (size_t i = 0; i < V.coded.size(); ++i) {  // the first two bytes of each chunk hold its keyframe bit
            uint8_t d[2] = {0, 0};
            const uint32_t len = std::min<uint32_t>(V.coded[i].second, 2);
            if (!file.seek(V.coded[i].first) || !file.read(d, len)) fail("truncated frame");
            V.keyframe[i] = (uint8_t)ffv1::keyframe_bit(d, len);
        }
        if (!V.keyframe.empty() && !V.keyframe[0])
            throw std::runtime_error("Video file " + V.name + ", frame 0: the first FFV1 frame is not a keyframe");
    } else if (V.codec == Codec::mpeg4) {
        index_mpeg4(V, file);
    } else {
        V.extradata.clear();
    }
    if (V.codec == Codec::png && !V.coded.empty()) {  // the size is frame 0's (IHDR); read_frames checks every other frame against it
        uint8_t d[45];
        const uint32_t len = std::min<uint32_t>(V.coded[0].second, sizeof d);
        V.rows = V.cols = 0;
        if (!file.seek(V.coded[0].first) || !file.read(d, len)) fail("truncated frame");
        check_png_frame(d, V.coded[0].second < sizeof d ? V.coded[0].second : sizeof d, V.rows, V.cols, "Video file " + V.name + ", frame 0");
    }
    if (V.codec == Codec::mjpeg && !V.coded.empty()) {
        // Frame 0's SOF must give the container's frame size (where the container states one): libavcodec weaves a frame
        // whose SOF height is below 3/4 of the container's as an interlaced field pair, and this decoder does not.  read_frames
        // checks every other frame against the size and frame 0's DHT tables.
        std::vector<uint8_t> d(V.coded[0].second);
        if (V.rows <= 0 || V.cols <= 0) V.rows = V.cols = 0;
        if (!file.seek(V.coded[0].first) || !file.read(d.data(), d.size())) fail("truncated frame");
        check_mjpeg_frame(d.data(), d.size(), V.rows, V.cols, V.mjpeg_dht, "Video file " + V.name + ", frame 0");
    }
    if (V.n == 0) fail("no video frames found");
}

// What a refusal of a stream this library does not decode ends with.
inline const char *outside_this_library() {
    return "Decoding compressed or YUV-planar video is outside this library (convert the video first).";
}

// The walk over stream 0's frame chunks ('00db' / '00dc') in file order, with the format and record checks.
inline Index index_avi(const std::string &name, const Options &opt = {}) {
    detail::File file(name);
    FILE *f = file.f;
    auto fail = [&](const std::string &why) -> void { throw std::runtime_error("Video file " + name + ": " + why); };
    auto rd = [&](void *dst, size_t n) { return file.read(dst, n); };
    auto skip = [&](uint64_t n) { return fseeko(f, (off_t)n, SEEK_CUR) == 0; };
    uint8_t h[12];
    if (!rd(h, 12) || std::memcmp(h, "RIFF", 4) || std::memcmp(h + 8, "AVI ", 4)) fail("not an AVI file");
    Index V;
    V.name = name;
    int bits = 0, height_signed = 0;
    uint32_t fourcc = 0;
    for (int i = 0; i < 256; ++i) V.palette_b[i] = (uint8_t)i;
    bool have_format = false, stream0_is_video = false, raw_rgb = false;
    int stream_index = -1;
    std::vector<uint8_t> chunk;
    // A flat walk: LIST / RIFF headers are entered (only their 4-byte type is consumed), every other chunk is read or skipped.
    for (;;) {
        uint8_t ch[8];
        if (!rd(ch, 8)) break;
        const uint32_t size = le32(ch + 4);
        if (!std::memcmp(ch, "LIST", 4) || !std::memcmp(ch, "RIFF", 4)) {
            uint8_t type[4];
            if (!rd(type, 4)) break;
            if (!std::memcmp(type, "strl", 4)) ++stream_index;
            if (!std::memcmp(ch, "LIST", 4) && std::memcmp(type, "hdrl", 4) && std::memcmp(type, "strl", 4) && std::memcmp(type, "movi", 4)) {
                if (!skip((uint64_t)size - 4 + (size & 1))) break;  // INFO, odml ... : not needed
            }
            continue;
        }
        if (!std::memcmp(ch, "strh", 4) && stream_index == 0) {
            chunk.resize(size);
            if (!rd(chunk.data(), size)) fail("truncated stream header");
            stream0_is_video = size >= 4 && !std::memcmp(chunk.data(), "vids", 4);
            if (size & 1) skip(1);
            continue;
        }
        if (!std::memcmp(ch, "strf", 4) && stream_index == 0) {
            chunk.resize(size);
            if (!rd(chunk.data(), size) || size < 40) fail("truncated stream format");
            if (size & 1) skip(1);
            V.cols = (int)le32(chunk.data() + 4);
            height_signed = (int)le32(chunk.data() + 8);
            V.rows = height_signed < 0 ? -height_signed : height_signed;
            bits = chunk[14] | (chunk[15] << 8);
            fourcc = le32(chunk.data() + 16);
            const uint32_t used = le32(chunk.data() + 32);
            V.extradata.assign(chunk.begin() + 40, chunk.end());
            const size_t ncol = used ? used : (bits <= 8 ? (size_t)1 << bits : 0);
            for (size_t i = 0; i < ncol && 40 + 4 * i + 3 < size && i < 256; ++i) V.palette_b[i] = chunk[40 + 4 * i];  // RGBQUAD: blue first
            have_format = true;
            continue;
        }
        const bool frame_chunk = ch[0] == '0' && ch[1] == '0' && ch[2] == 'd' && (ch[3] == 'b' || ch[3] == 'c');
        if (!frame_chunk) {
            if (!skip((uint64_t)size + (size & 1))) break;
            continue;
        }
        if (!have_format || !stream0_is_video || V.rows <= 0 || V.cols <= 0) fail("frame data before a usable video stream format");
        auto cc = [](const char *s) { return le32(reinterpret_cast<const uint8_t *>(s)); };
        const bool grey = fourcc == cc("Y800") || fourcc == cc("GREY") || fourcc == cc("Y8  ") || fourcc == cc("Y8\0\0");
        const bool rgb = fourcc == 0 || fourcc == cc("DIB ") || fourcc == cc("RGB ") || fourcc == cc("RAW ");
        const bool png = fourcc == cc("MPNG") || fourcc == cc("png ");
        const bool mjpg = opt.decode_mjpeg && (fourcc == cc("MJPG") || fourcc == cc("mjpg"));
        const bool mp4v = opt.decode_mpeg4 && mpeg4_fourcc(fourcc);
        if (png || mjpg || mp4v || fourcc == cc("FFV1")) {
            if (size == 0) continue;
            V.codec = png ? Codec::png : mjpg ? Codec::mjpeg : mp4v ? Codec::mpeg4 : Codec::ffv1;
            V.fourcc = fourcc;
            const off_t at = ftello(f);
            V.coded.emplace_back((int64_t)at, size);
            if (!skip((uint64_t)size + (size & 1))) fail("truncated frame");
            continue;
        }
        if (!(grey && bits == 8) && !(rgb && (bits == 8 || bits == 24 || bits == 32))) {
            char fc[5] = {(char)(fourcc & 255), (char)((fourcc >> 8) & 255), (char)((fourcc >> 16) & 255), (char)((fourcc >> 24) & 255), 0};
            fail(std::string("stream 0 is '") + fc + "' with " + std::to_string(bits) +
                 " bits per pixel; only uncompressed 8-bit grey (Y800) and BI_RGB 8 / 24 / 32-bit frames are read here. " + outside_this_library() +
                 (mpeg4_fourcc(fourcc) ? mpeg4_opt_in() : ""));
        }
        if (size == 0) continue;  // dropped frame: VideoCapture repeats nothing, it simply has one frame less
        const size_t tight = (size_t)V.cols * (bits / 8), padded = (tight + 3) & ~(size_t)3;
        size_t stride;
        if (size >= padded * V.rows) stride = padded;
        else if (size >= tight * V.rows) stride = tight;
        else { fail("frame chunk smaller than one image"); return V; }
        V.grey = grey;
        raw_rgb = rgb;
        V.raw.push_back(Index::RawChunk{(int64_t)ftello(f), size, stride});
        if (!skip((uint64_t)size + (size & 1))) fail("truncated frame");
    }
    V.bpp = bits / 8;
    V.bottom_up = raw_rgb && height_signed > 0;  // BI_RGB DIBs are stored bottom-up unless the height is negative
    if (!V.raw.empty()) {
        V.codec = Codec::raw;
        V.coded.clear();
        V.n = (int)V.raw.size();
    } else {
        V.n = (int)V.coded.size();
    }
    finish_index(V, file);
    return V;
}

// The LMV1 container (lm_files.hpp): a header, then every frame's rows x cols bytes back to back.
inline Index index_lmv(const std::string &name) {
    detail::File file(name);
    uint8_t h[16];
    if (!file.read(h, 4) || std::memcmp(h, "LMV1", 4)) throw std::runtime_error("Unexpected file format (LMV1 expected): " + name);
    if (!file.read(h + 4, 12)) throw std::runtime_error("File is truncated: " + name);
    Index V;
    V.name = name;
    V.n = (int)le32(h + 4);
    V.rows = (int)le32(h + 8);
    V.cols = (int)le32(h + 12);
    if (V.n <= 0 || V.rows <= 0 || V.cols <= 0) throw std::runtime_error("Video file is empty: " + name);
    const size_t fsz = (size_t)V.rows * V.cols;
    if (file.size() < 16 + (int64_t)(fsz * V.n)) throw std::runtime_error("File is truncated: " + name);
    V.raw.reserve((size_t)V.n);
    for (int i = 0; i < V.n; ++i) V.raw.push_back(Index::RawChunk{16 + (int64_t)(fsz * i), (uint32_t)fsz, (size_t)V.cols});
    return V;
}

// Matroska and QuickTime / MP4 (lm_containers.hpp)
inline bool is_mkv(const std::string &name);
inline bool is_mov(const std::string &name);
inline Index index_mkv(const std::string &name, const Options &opt = {});
inline Index index_mov(const std::string &name, const Options &opt = {});

// The container is chosen by the file's signature, not its extension: AVI, Matroska, QuickTime / MP4, LMV1.
inline Index index_video(const std::string &name, const Options &opt = {}) {
    if (is_avi(name)) return index_avi(name, opt);
    if (is_mkv(name)) return index_mkv(name, opt);
    if (is_mov(name)) return index_mov(name, opt);
    const std::vector<uint8_t> h = slurp(name, 4);
    if (h.size() < 4 || std::memcmp(h.data(), "LMV1", 4))
        throw std::runtime_error("Video file " + name +
                                 ": unrecognised container; the videos read here are AVI, Matroska (.mkv), QuickTime / MP4 (.mov, .mp4) and LMV1");
    return index_lmv(name);
}

// Frames [first, first + n) of an indexed video.  Uncompressed: channel 0 of each frame, [n][rows][cols]; coded: the frame
// chunks back to back, with offsets relative to the first of them (PNG frames are checked here against frame 0's size).
inline Video read_frames(const Index &ix, int first, int n, const Dest &dest = nullptr) {
    if (first < 0 || n <= 0 || first + n > ix.n) throw std::runtime_error("Video file " + ix.name + ": frame range outside the video");
    detail::File file(ix.name);
    auto fail = [&](const std::string &why) -> void { throw std::runtime_error("Video file " + ix.name + ": " + why); };
    Video V;
    V.rows = ix.rows;
    V.cols = ix.cols;
    V.codec = ix.codec;
    if (ix.codec == Codec::raw) {
        const size_t fsz = (size_t)V.rows * V.cols;
        uint8_t *out = nullptr;
        if (dest) {
            out = dest((size_t)n * fsz);
            if (!out) fail("cannot allocate " + std::to_string((size_t)n * fsz) + " bytes for the frames");
        } else {
            V.frames.resize((size_t)n * fsz);
            out = V.frames.data();
        }
        std::vector<uint8_t> chunk;
        for (int i = 0; i < n; ++i) {
            const Index::RawChunk &c = ix.raw[(size_t)(first + i)];
            const size_t stride = c.stride;
            const bool direct = ix.grey && ix.bpp == 1 && stride == (size_t)V.cols;  // the chunk is the frame: read it in place
            uint8_t *frame = out + (size_t)i * fsz;
            chunk.resize(stride * V.rows);
            if (!file.seek(c.at) || !file.read(direct ? frame : chunk.data(), direct ? fsz : chunk.size())) fail("truncated frame");
            if (!direct)
                for (int r = 0; r < V.rows; ++r) {
                    const uint8_t *src = chunk.data() + (size_t)(ix.bottom_up ? V.rows - 1 - r : r) * stride;
                    uint8_t *dst = frame + (size_t)r * V.cols;
                    if (ix.bpp == 1) {
                        if (ix.grey) std::memcpy(dst, src, (size_t)V.cols);
                        else for (int x = 0; x < V.cols; ++x) dst[x] = ix.palette_b[src[x]];
                    } else {
                        for (int x = 0; x < V.cols; ++x) dst[x] = src[(size_t)x * ix.bpp + ix.channel0];  // B of BGR(A): channel 0
                    }
                }
        }
        V.n = n;
        return V;
    }
    uint64_t total = 0;
    for (int i = 0; i < n; ++i) total += ix.coded[(size_t)(first + i)].second;
    uint8_t *buf = dest ? dest((size_t)total) : static_cast<uint8_t *>(std::malloc(total ? (size_t)total : 1));
    if (!buf) fail("cannot allocate " + std::to_string(total) + " bytes for the compressed frames");
    if (dest) V.payload = std::shared_ptr<uint8_t>(buf, [](uint8_t *) {});  // owned by the caller
    else V.payload = std::shared_ptr<uint8_t>(buf, [](uint8_t *q) { std::free(q); });
    V.offsets.push_back(0);
    int dht = ix.mjpeg_dht;
    for (int i = 0; i < n; ++i) {
        const auto &c = ix.coded[(size_t)(first + i)];
        uint8_t *d = buf + V.offsets.back();
        if (!file.seek(c.first) || !file.read(d, c.second)) fail("truncated frame");
        if (ix.codec == Codec::png) check_png_frame(d, c.second, V.rows, V.cols, "Video file " + ix.name + ", frame " + std::to_string(first + i));
        if (ix.codec == Codec::mjpeg) check_mjpeg_frame(d, c.second, V.rows, V.cols, dht, "Video file " + ix.name + ", frame " + std::to_string(first + i));
        V.offsets.push_back(V.offsets.back() + c.second);
    }
    V.n = n;
    V.extradata = ix.extradata;
    return V;
}

// The whole video: its index, then every frame in one read.
inline Video read_avi(const std::string &name, const Dest &dest = nullptr) {
    const Index ix = index_avi(name);
    return read_frames(ix, 0, ix.n, dest);
}

// Window length for a budget of `max_bytes` of frames: whole multiples of batch_frames, at least one.
inline int window_frames(size_t max_bytes, size_t frame_bytes, int batch_frames) {
    const size_t w = max_bytes / frame_bytes / (size_t)batch_frames * (size_t)batch_frames;
    return (int)std::min<size_t>(std::max<size_t>(w, (size_t)batch_frames), (size_t)1 << 30);
}

// The first frame of every window of at most W frames, then n.  A video of n <= W frames is one window.  FFV1 (keyframe
// given): a window ends just before a keyframe, so that each window decodes on its own; a GOP longer than W is one window.
inline std::vector<int> plan_windows(int n, int W, const std::vector<uint8_t> &keyframe) {
    std::vector<int> s{0};
    while (n - s.back() > W) {
        const int a = s.back();
        int b = a + W;
        if (!keyframe.empty()) {
            while (b > a && !keyframe[(size_t)b]) --b;                       // the last keyframe in (a, a + W]
            if (b == a)
                for (b = a + W + 1; b < n && !keyframe[(size_t)b]; ++b) {}  // none: the window runs to the next keyframe
        }
        s.push_back(b);
    }
    if (s.back() != n) s.push_back(n);
    return s;
}

struct Image {
    int rows = 0, cols = 0;
    std::vector<uint8_t> px;
};

inline Image read_png_gray(const std::string &name) {
    const std::vector<uint8_t> d = slurp(name);
    auto fail = [&](const std::string &why) -> void { throw std::runtime_error("Image file " + name + ": " + why); };
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    if (d.size() < 8 || std::memcmp(d.data(), sig, 8)) fail("not a PNG file");
    Image I;
    int depth = 0, ctype = 0, interlace = 0;
    std::vector<uint8_t> idat, plte;
    for (size_t pos = 8; pos + 12 <= d.size();) {
        const uint32_t len = be32(&d[pos]);
        const uint8_t *type = &d[pos + 4], *data = &d[pos + 8];
        if (pos + 12 + (size_t)len > d.size()) fail("truncated chunk");
        if (!std::memcmp(type, "IHDR", 4) && len >= 13) {
            I.cols = (int)be32(data);
            I.rows = (int)be32(data + 4);
            depth = data[8];
            ctype = data[9];
            interlace = data[12];
        } else if (!std::memcmp(type, "PLTE", 4)) {
            plte.assign(data, data + len);
        } else if (!std::memcmp(type, "IDAT", 4)) {
            idat.insert(idat.end(), data, data + len);
        } else if (!std::memcmp(type, "IEND", 4)) {
            break;
        }
        pos += 12 + (size_t)len;
    }
    if (I.rows <= 0 || I.cols <= 0) fail("missing header");
    if (depth != 8 || interlace != 0) fail("only 8 bits per channel, non-interlaced PNG images are read here");
    int ch = 0;
    switch (ctype) {
        case 0: ch = 1; break;
        case 2: ch = 3; break;
        case 3: ch = 1; break;
        case 4: ch = 2; break;
        case 6: ch = 4; break;
        default: fail("unknown colour type");
    }
    const size_t stride = (size_t)I.cols * ch;
    std::vector<uint8_t> raw((stride + 1) * (size_t)I.rows);
    uLongf out_len = (uLongf)raw.size();
    if (uncompress(raw.data(), &out_len, idat.data(), (uLong)idat.size()) != Z_OK || out_len != raw.size()) fail("corrupt image data");
    std::vector<uint8_t> cur(stride), prev(stride, 0);
    I.px.resize((size_t)I.rows * I.cols);
    for (int r = 0; r < I.rows; ++r) {
        const uint8_t *src = &raw[(stride + 1) * (size_t)r];
        const int ft = src[0];
        ++src;
        for (size_t i = 0; i < stride; ++i) {
            const int a = i >= (size_t)ch ? cur[i - ch] : 0, b = prev[i], c = i >= (size_t)ch ? prev[i - ch] : 0;
            int pred = 0;
            switch (ft) {
                case 0: pred = 0; break;
                case 1: pred = a; break;
                case 2: pred = b; break;
                case 3: pred = (a + b) >> 1; break;
                case 4: {
                    const int p = a + b - c, pa = p > a ? p - a : a - p, pb = p > b ? p - b : b - p, pc = p > c ? p - c : c - p;
                    pred = (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
                    break;
                }
                default: fail("unknown row filter");
            }
            cur[i] = (uint8_t)(src[i] + pred);
        }
        uint8_t *dst = &I.px[(size_t)r * I.cols];
        for (int x = 0; x < I.cols; ++x) {
            const uint8_t *p = &cur[(size_t)x * ch];
            int R, G, B;
            if (ctype == 0 || ctype == 4) {
                dst[x] = p[0];
                continue;
            }
            if (ctype == 3) {
                if ((size_t)p[0] * 3 + 2 >= plte.size()) fail("palette index out of range");
                R = plte[p[0] * 3];
                G = plte[p[0] * 3 + 1];
                B = plte[p[0] * 3 + 2];
            } else {
                R = p[0];
                G = p[1];
                B = p[2];
            }
            // libpng's png_set_rgb_to_gray(1, 0.299, 0.587) as OpenCV's PNG reader requests it: 15-bit fixed point (9797 / 19234 and
            // the remainder 3737 for blue), truncated -- verified against cv2.imread(IMREAD_GRAYSCALE) of OpenCV 4.13; equal
            // channels pass through unchanged
            dst[x] = (R == G && G == B) ? (uint8_t)R : (uint8_t)((R * 9797 + G * 19234 + B * 3737) >> 15);
        }
        std::swap(cur, prev);
    }
    return I;
}

}  // namespace lmmedia

#include "lm_containers.hpp"
