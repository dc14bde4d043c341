// mjpeg_format.h — baseline JPEG frames of Motion-JPEG video as libavcodec's 'mjpeg' decoder reads them, reduced to channel 0
// of the BGR frame cv::VideoCapture delivers.
//
// Shared by the host (the video index checks frame 0's SOF and every frame of a window against it; lmh_decode_mjpeg runs
// the whole decode on the CPU for the tests) and by k_mjpeg.cu (k_mjpeg_locate runs parse() per frame, k_mjpeg_entropy runs
// decode_scan() per frame, k_mjpeg_idct runs idct_block() per block).  Every function that touches stream bytes is bounded by
// the frame it reads: bytes past the end read as zero and are counted, every loop consumes input or produces output, and
// malformed data ends the frame with an LM_MJPEG_* status.
//
// The rules (verified against cv2.VideoCapture of OpenCV 4.13 with its FFmpeg build, see DESIGN §8):
//   - DC predictor starts at 1024 (4 << 8: the +128 level shift folded in) and resets at every restart marker;
//     dc = diff * q[0] + pred, block[0] = clip_int16(dc); AC block[zigzag[k]] = (int16) (level * q[k]).
//   - IDCT: libavcodec's simple_idct for 8 bits (idct_row / idct_col below), outputs clipped to 0..255.
//   - 1 component: channel 0 = Y.  3 components (Y at 2x2 or 2x1, Cb / Cr at 1x1, even frame height):
//     channel 0 = clip((Y * 8192 + (Cb - 128) * 14516) >> 13) with Cb replicated over its Y samples.  Cr is entropy-decoded
//     (the bit stream runs through it) but never stored.
//   - Refused: progressive, lossless and arithmetic-coded frames, 12-bit samples, 16-bit quantisation tables, 2 or 4
//     components, RGB-coded 3-component frames (Adobe transform 0 or component ids 'R', 'G', 'B'), 4:4:4 and other layouts,
//     odd heights with chroma, non-interleaved scans, and a frame whose size is not the stream's.  libavcodec keeps DQT and
//     DHT tables from frame to frame; here each frame is decoded alone, so a frame must define its quantisation tables, and
//     every frame of a video must define the same Huffman tables by DHT as the first (dht_mask), or none (Annex K tables).
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define MJPEG_HD __host__ __device__ __forceinline__
#else
#define MJPEG_HD inline
#endif

namespace mjpeg {

// Per-frame status codes (k_mjpeg_locate / k_mjpeg_entropy write one per frame; -1 = not decoded)
enum {
    LM_MJPEG_OK = 0, LM_MJPEG_MARKER, LM_MJPEG_HEADER, LM_MJPEG_PROGRESSIVE, LM_MJPEG_LOSSLESS, LM_MJPEG_ARITHMETIC, LM_MJPEG_PRECISION,
    LM_MJPEG_DQT16, LM_MJPEG_COMPONENTS, LM_MJPEG_RGB, LM_MJPEG_SAMPLING, LM_MJPEG_SIZE, LM_MJPEG_TABLE, LM_MJPEG_SCAN, LM_MJPEG_CODE,
    LM_MJPEG_CATEGORY, LM_MJPEG_RUN, LM_MJPEG_TRUNCATED, LM_MJPEG_RESTART, LM_MJPEG_NO_DQT, LM_MJPEG_DHT_CHANGE
};

inline const char *status_text(int st) {
    switch (st) {
        case LM_MJPEG_OK: return "ok";
        case LM_MJPEG_MARKER: return "not a JPEG image, or a marker is missing where one must be";
        case LM_MJPEG_HEADER: return "truncated or malformed JPEG header segment";
        case LM_MJPEG_PROGRESSIVE: return "progressive JPEG (SOF2) is not decoded";
        case LM_MJPEG_LOSSLESS: return "lossless or hierarchical JPEG (SOF3, SOF5..7) is not decoded";
        case LM_MJPEG_ARITHMETIC: return "arithmetic-coded JPEG (SOF9 and up) is not decoded";
        case LM_MJPEG_PRECISION: return "only 8-bit JPEG samples are decoded (12-bit frame)";
        case LM_MJPEG_DQT16: return "16-bit quantisation tables are not decoded";
        case LM_MJPEG_COMPONENTS: return "only 1-component (grey) and 3-component (YCbCr) JPEG frames are decoded";
        case LM_MJPEG_RGB: return "RGB-coded JPEG (Adobe transform 0, or components 'R', 'G', 'B') is not decoded";
        case LM_MJPEG_SAMPLING:
            return "chroma layout not decoded: only Y at 2x2 (4:2:0) or 2x1 (4:2:2) with Cb and Cr at 1x1 and an even frame height "
                   "match VideoCapture's colour conversion by a rule this library restates";
        case LM_MJPEG_SIZE: return "the frame's SOF size differs from the video's (interlaced field pairs are not woven)";
        case LM_MJPEG_TABLE: return "malformed or missing quantisation / Huffman table";
        case LM_MJPEG_SCAN: return "malformed scan header (only one interleaved baseline scan of all components is decoded)";
        case LM_MJPEG_CODE: return "invalid Huffman code in the entropy-coded data";
        case LM_MJPEG_CATEGORY: return "coefficient category out of range in the entropy-coded data";
        case LM_MJPEG_RUN: return "AC run past coefficient 63";
        case LM_MJPEG_TRUNCATED: return "the entropy-coded data ends before the last block";
        case LM_MJPEG_RESTART: return "restart marker missing where the restart interval puts one";
        case LM_MJPEG_NO_DQT:
            return "a component's quantisation table is not defined in the frame (libavcodec would reuse an earlier frame's DQT, "
                   "which is not decoded)";
        case LM_MJPEG_DHT_CHANGE:
            return "the frame defines other Huffman tables (DHT) than the video's first frame (libavcodec carries tables from frame "
                   "to frame, which is not decoded)";
        case -1: return "not decoded";
        default: return "unknown error";
    }
}

constexpr int FAST_BITS = 9;  // lookahead of the Huffman tables

MJPEG_HD int zigzag(int k) {
    constexpr uint8_t z[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                               41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                               30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return z[k];
}

struct Huff {
    uint8_t bits[17];   // bits[l]: codes of length l (1..16)
    uint8_t vals[256];
    uint8_t defined;
    uint8_t pad_[2];
};

// What parse() finds in one frame: enough to entropy-decode and transform it.
struct Header {
    int32_t rows, cols, ncomp, hy, vy, dri;
    int32_t td[3], ta[3];      // DC / AC table of each component
    int64_t ecs;               // entropy-coded data starts at this byte of the frame
    uint16_t q[2][64];         // quantisation of Y and Cb, in zigzag order
    uint8_t qcr_ok;
    uint8_t dht_mask;          // bit s: the frame's DHT defines tab[s]; every frame of a video must define the same set
    uint8_t pad_[6];
    Huff tab[4];               // DC 0, DC 1, AC 0, AC 1
    MJPEG_HD int mcu_w() const { return 8 * hy; }
    MJPEG_HD int mcu_h() const { return 8 * vy; }
    MJPEG_HD int mcus_x() const { return (cols + mcu_w() - 1) / mcu_w(); }
    MJPEG_HD int mcus_y() const { return (rows + mcu_h() - 1) / mcu_h(); }
    MJPEG_HD int y_blocks_x() const { return mcus_x() * hy; }
    MJPEG_HD int y_blocks_y() const { return mcus_y() * vy; }
    // coefficient blocks of a frame: Y blocks [y_blocks_y][y_blocks_x], then (3 components) Cb blocks [mcus_y][mcus_x]
    MJPEG_HD int64_t blocks() const { return (int64_t)y_blocks_x() * y_blocks_y() + (ncomp == 3 ? (int64_t)mcus_x() * mcus_y() : 0); }
};

// Coefficient blocks of a frame of the given size in the layout that has the most (grey, 4:2:0 or 4:2:2): the scratch
// bound per frame
MJPEG_HD int64_t max_blocks(int rows, int cols) {
    const int64_t x8 = (cols + 7) / 8, y8 = (rows + 7) / 8, x16 = (cols + 15) / 16, y16 = (rows + 15) / 16;
    const int64_t grey = x8 * y8, c420 = x16 * y16 * 5, c422 = x16 * y8 * 3;
    return grey > c420 ? (grey > c422 ? grey : c422) : (c420 > c422 ? c420 : c422);
}

// JPEG Annex K.3 tables, which libavcodec uses where a frame has no DHT
MJPEG_HD void default_table(int slot, Huff &h) {
    constexpr uint8_t dc_bits[2][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0}, {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}};
    constexpr uint8_t ac_bits[2][16] = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d}, {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
    constexpr uint8_t ac_vals[2][162] = {
        {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81,
         0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18,
         0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
         0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75,
         0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99,
         0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
         0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5,
         0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
        {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08,
         0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25,
         0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47,
         0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74,
         0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97,
         0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
         0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4,
         0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};
    const int ac = slot >> 1, id = slot & 1;
    h.bits[0] = 0;
    for (int l = 0; l < 16; ++l) h.bits[l + 1] = ac ? ac_bits[id][l] : dc_bits[id][l];
    for (int i = 0; i < 256; ++i) h.vals[i] = ac ? (i < 162 ? ac_vals[id][i] : 0) : (uint8_t)(i < 12 ? i : 0);
    h.defined = 1;
}

MJPEG_HD int be16(const uint8_t *p) { return (p[0] << 8) | p[1]; }

// The header segments of one frame up to its SOS.  rows / cols: the video's size (0: take the frame's).  Returns a status.
MJPEG_HD int parse(const uint8_t *f, int64_t len, int rows, int cols, Header &h) {
    uint8_t qt[4][64];
    bool qdef[4] = {false, false, false, false}, adobe_rgb = false, sof = false;
    int cid[3] = {0, 0, 0}, ctq[3] = {0, 0, 0}, chs[3] = {0, 0, 0}, cvs[3] = {0, 0, 0};
    for (int s = 0; s < 4; ++s) default_table(s, h.tab[s]);
    h.dri = 0;
    h.dht_mask = 0;
    if (len < 4 || f[0] != 0xFF || f[1] != 0xD8) return LM_MJPEG_MARKER;
    int64_t p = 2;
    for (;;) {
        if (p >= len || f[p] != 0xFF) return LM_MJPEG_MARKER;
        while (p < len && f[p] == 0xFF) ++p;  // fill bytes
        if (p + 2 >= len) return LM_MJPEG_HEADER;
        const int m = f[p];
        if (m == 0xD8 || m == 0xD9 || m == 0x01 || (m >= 0xD0 && m <= 0xD7) || m == 0) return LM_MJPEG_MARKER;
        const int L = be16(f + p + 1);
        const int64_t s = p + 3, e = p + 1 + L;  // segment payload [s, e)
        if (L < 2 || e > len) return LM_MJPEG_HEADER;
        const uint8_t *d = f + s;
        const int n = (int)(e - s);
        if (m == 0xC2 || m == 0xC6 || m == 0xCA || m == 0xCE) return LM_MJPEG_PROGRESSIVE;
        if (m == 0xC3 || m == 0xC5 || m == 0xC7) return LM_MJPEG_LOSSLESS;
        if (m >= 0xC9 && m <= 0xCF) return LM_MJPEG_ARITHMETIC;
        if (m == 0xDB) {  // DQT
            for (int i = 0; i < n;) {
                const int pq = d[i] >> 4, tq = d[i] & 15;
                if (pq) return LM_MJPEG_DQT16;
                if (tq > 3 || i + 65 > n) return LM_MJPEG_TABLE;
                for (int k = 0; k < 64; ++k) qt[tq][k] = d[i + 1 + k];
                qdef[tq] = true;
                i += 65;
            }
        } else if (m == 0xC4) {  // DHT
            for (int i = 0; i < n;) {
                if (i + 17 > n) return LM_MJPEG_TABLE;
                const int tc = d[i] >> 4, th = d[i] & 15;
                if (tc > 1 || th > 1) return LM_MJPEG_TABLE;
                Huff &t = h.tab[tc * 2 + th];
                h.dht_mask |= (uint8_t)(1 << (tc * 2 + th));
                int cnt = 0;
                t.bits[0] = 0;
                for (int l = 1; l <= 16; ++l) cnt += (t.bits[l] = d[i + l]);
                if (cnt > 256 || i + 17 + cnt > n) return LM_MJPEG_TABLE;
                for (int k = 0; k < 256; ++k) t.vals[k] = k < cnt ? d[i + 17 + k] : 0;
                i += 17 + cnt;
            }
        } else if (m == 0xC0 || m == 0xC1) {  // SOF0 / SOF1
            if (n < 6) return LM_MJPEG_HEADER;
            if (d[0] != 8) return LM_MJPEG_PRECISION;
            h.rows = be16(d + 1);
            h.cols = be16(d + 3);
            h.ncomp = d[5];
            if (h.ncomp != 1 && h.ncomp != 3) return LM_MJPEG_COMPONENTS;
            if (n < 6 + 3 * h.ncomp) return LM_MJPEG_HEADER;
            for (int c = 0; c < h.ncomp; ++c) {
                cid[c] = d[6 + 3 * c];
                chs[c] = d[7 + 3 * c] >> 4;
                cvs[c] = d[7 + 3 * c] & 15;
                ctq[c] = d[8 + 3 * c];
                if (ctq[c] > 3) return LM_MJPEG_TABLE;
            }
            sof = true;
        } else if (m == 0xDD) {  // DRI
            if (n < 2) return LM_MJPEG_HEADER;
            h.dri = be16(d);
        } else if (m == 0xEE) {  // APP14: "Adobe", transform byte last
            if (n >= 12 && d[0] == 'A' && d[1] == 'd' && d[2] == 'o' && d[3] == 'b' && d[4] == 'e' && d[11] == 0) adobe_rgb = true;
        } else if (m == 0xDA) {  // SOS
            if (!sof) return LM_MJPEG_MARKER;
            if (h.rows <= 0 || h.cols <= 0) return LM_MJPEG_SIZE;
            if ((rows || cols) && (h.rows != rows || h.cols != cols)) return LM_MJPEG_SIZE;
            if (h.ncomp == 1) {
                h.hy = h.vy = 1;  // a single component is never interleaved: 8 x 8 blocks whatever its factors say
            } else {
                if (adobe_rgb || (cid[0] == 'R' && cid[1] == 'G' && cid[2] == 'B')) return LM_MJPEG_RGB;
                h.hy = chs[0];
                h.vy = cvs[0];
                if (!(h.hy == 2 && (h.vy == 2 || h.vy == 1)) || chs[1] != 1 || cvs[1] != 1 || chs[2] != 1 || cvs[2] != 1 || (h.rows & 1))
                    return LM_MJPEG_SAMPLING;
            }
            const int ns = n >= 1 ? d[0] : 0;
            if (ns != h.ncomp || n < 4 + 2 * ns) return LM_MJPEG_SCAN;
            for (int c = 0; c < ns; ++c) {
                if (d[1 + 2 * c] != cid[c]) return LM_MJPEG_SCAN;
                h.td[c] = d[2 + 2 * c] >> 4;
                h.ta[c] = d[2 + 2 * c] & 15;
                if (h.td[c] > 1 || h.ta[c] > 1) return LM_MJPEG_TABLE;
            }
            if (d[1 + 2 * ns] != 0 || d[2 + 2 * ns] != 63 || d[3 + 2 * ns] != 0) return LM_MJPEG_SCAN;
            for (int c = 0; c < h.ncomp && c < 2; ++c) {
                if (!qdef[ctq[c]]) return LM_MJPEG_NO_DQT;
                for (int k = 0; k < 64; ++k) h.q[c][k] = qt[ctq[c]][k];
            }
            h.qcr_ok = h.ncomp == 1 || qdef[ctq[2]];
            if (!h.qcr_ok) return LM_MJPEG_NO_DQT;
            h.ecs = e;
            return LM_MJPEG_OK;
        }
        // APPn, COM and every other segment: skipped
        p = e;
    }
}

// Lookahead table of one Huffman table: entry = length << 8 | symbol for codes of up to FAST_BITS bits, 0 otherwise.
// Returns false when the counts describe more codes than fit (an over-subscribed table).
MJPEG_HD bool build_fast(const Huff &t, uint16_t *fast) {
    for (int i = 0; i < (1 << FAST_BITS); ++i) fast[i] = 0;
    int code = 0, k = 0;
    for (int l = 1; l <= 16; ++l) {
        for (int i = 0; i < t.bits[l]; ++i, ++k, ++code) {
            if (code >= (1 << l)) return false;
            if (l <= FAST_BITS) {
                const int lo = code << (FAST_BITS - l), hi = (code + 1) << (FAST_BITS - l);
                for (int j = lo; j < hi; ++j) fast[j] = (uint16_t)((l << 8) | t.vals[k]);
            }
        }
        code <<= 1;
    }
    return true;
}

// The entropy-coded bytes as libavcodec's unescaping reads them: FF 00 is a data byte FF (also after fill bytes FF FF ..),
// FF D0..D7 is a restart marker, any other marker ends the data; past the end the reader feeds zero bits and counts them.
struct BitReader {
    const uint8_t *begin, *p, *end;
    uint64_t acc;  // bits MSB-first: the next bit is bit 63
    int nbits;
    int pad;       // zero bits fed past the data, at the bottom of acc
    bool at_marker;
    MJPEG_HD void init(const uint8_t *b, const uint8_t *e) {
        begin = p = b;
        end = e;
        acc = 0;
        nbits = 0;
        pad = 0;
        at_marker = false;
    }
    MJPEG_HD uint32_t load4(const uint8_t *q) const {  // 4 stream bytes, big-endian, q + 4 <= end
#ifdef __CUDA_ARCH__
        const uintptr_t a = (uintptr_t)q;
        const uint8_t *w0 = reinterpret_cast<const uint8_t *>(a & ~(uintptr_t)3);
        if ((a & 3) == 0) return __byte_perm(*reinterpret_cast<const uint32_t *>(q), 0, 0x0123);
        if (w0 >= begin && w0 + 8 <= end) {  // two aligned words, both inside the data
            const uint32_t lo = __ldg(reinterpret_cast<const uint32_t *>(w0)), hi = __ldg(reinterpret_cast<const uint32_t *>(w0) + 1);
            return __byte_perm(__funnelshift_r(lo, hi, (unsigned)(a & 3) * 8), 0, 0x0123);
        }
#endif
        return ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
    }
    MJPEG_HD void feed(uint32_t b) {
        acc |= (uint64_t)b << (56 - nbits);
        nbits += 8;
    }
    // at least 32 bits in acc
    MJPEG_HD void refill() {
        while (nbits <= 56) {
            if (nbits <= 32 && !at_marker && p + 4 <= end) {  // four bytes at once when none of them is FF
                const uint32_t w = load4(p), nw = ~w;
                if (((nw - 0x01010101u) & w & 0x80808080u) == 0) {
                    acc |= (uint64_t)w << (32 - nbits);
                    nbits += 32;
                    p += 4;
                    continue;
                }
            }
            if (at_marker || p >= end) {
                feed(0);
                pad += 8;
                continue;
            }
            const uint8_t b = *p;
            if (b != 0xFF) {
                feed(b);
                ++p;
                continue;
            }
            const uint8_t *q = p + 1;
            while (q < end && *q == 0xFF) ++q;
            if (q < end && *q == 0) {
                feed(0xFF);
                p = q + 1;
            } else {
                p = q - 1;  // the marker's last FF
                at_marker = true;
            }
        }
    }
    MJPEG_HD uint32_t peek(int n) const { return (uint32_t)(acc >> (64 - n)); }
    MJPEG_HD void skip(int n) {
        acc <<= n;
        nbits -= n;
    }
    MJPEG_HD bool overrun() const { return nbits < pad; }
};

// One Huffman symbol (refill() done by the caller): symbol, or -1 for a code no table entry has.
MJPEG_HD int huff_decode(BitReader &br, const uint16_t *fast, const Huff &t) {
    const uint16_t e = fast[br.peek(FAST_BITS)];
    if (e) {
        br.skip(e >> 8);
        return e & 255;
    }
    const uint32_t c16 = br.peek(16);
    int code = 0, first = 0, index = 0;
    for (int l = 1; l <= 16; ++l) {
        code |= (c16 >> (16 - l)) & 1;
        const int cnt = t.bits[l];
        if (code - first < cnt) {
            br.skip(l);
            return t.vals[index + code - first];
        }
        index += cnt;
        first = (first + cnt) << 1;
        code <<= 1;
    }
    return -1;
}

MJPEG_HD int extend(uint32_t v, int s) { return (int)v < (1 << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v; }

// The blocks of one frame, in file order, dequantised into `coef` (layout of Header::blocks(); Y and Cb only, Cr is read and
// dropped).  fast[4][1 << FAST_BITS]: build_fast() of h.tab[0..3].  Returns a status.
template <class Sink>
MJPEG_HD int decode_scan(const Header &h, const uint8_t *data, const uint8_t *end, const uint16_t *fast, Sink &&sink) {
    BitReader br;
    br.init(data, end);
    const int mx = h.mcus_x(), my = h.mcus_y(), nmcu = mx * my;
    const int ybx = h.y_blocks_x();
    const int64_t ny = (int64_t)ybx * h.y_blocks_y();
    int pred[3] = {1024, 1024, 1024};
    int left = h.dri;
    for (int m = 0; m < nmcu; ++m) {
        if (h.dri && left == 0) {  // restart: byte-align, expect RSTn
            br.skip(br.nbits & 7);
            if (br.nbits > br.pad) return LM_MJPEG_RESTART;  // data left in the interval
            br.refill();                                     // up to the marker
            if (!br.at_marker || br.nbits > br.pad) return LM_MJPEG_RESTART;
            const uint8_t *q = br.p;
            if (q + 1 >= end || (q[1] & 0xF8) != 0xD0) return LM_MJPEG_RESTART;
            br.init(q + 2, end);
            pred[0] = pred[1] = pred[2] = 1024;
            left = h.dri;
        }
        --left;
        const int mcu_y = m / mx, mcu_x = m - mcu_y * mx;
        for (int c = 0; c < h.ncomp; ++c) {
            const int nb = c == 0 ? h.hy * h.vy : 1;
            const uint16_t *fdc = fast + h.td[c] * (1 << FAST_BITS), *fac = fast + (2 + h.ta[c]) * (1 << FAST_BITS);
            const Huff &tdc = h.tab[h.td[c]], &tac = h.tab[2 + h.ta[c]];
            const uint16_t *q = h.q[c < 2 ? c : 1];
            for (int b = 0; b < nb; ++b) {
                alignas(16) int16_t blk[64];
                const bool keep = c < 2;
                if (keep)
                    for (int k = 0; k < 64; ++k) blk[k] = 0;
                br.refill();
                const int s = huff_decode(br, fdc, tdc);
                if (s < 0) return LM_MJPEG_CODE;
                if (s > 11) return LM_MJPEG_CATEGORY;
                const int diff = s ? extend(br.peek(s), s) : 0;
                br.skip(s);
                const int dc = (int)((unsigned)diff * q[0] + (unsigned)pred[c]);  // wrapping, as libavcodec
                pred[c] = dc;
                if (keep) blk[0] = (int16_t)(dc < -32768 ? -32768 : dc > 32767 ? 32767 : dc);
                for (int k = 1; k < 64;) {
                    br.refill();
                    const int rs = huff_decode(br, fac, tac);
                    if (rs < 0) return LM_MJPEG_CODE;
                    const int r = rs >> 4, sz = rs & 15;
                    if (sz == 0) {
                        if (r == 15) {
                            k += 16;
                            if (k > 64) return LM_MJPEG_RUN;
                            continue;
                        }
                        break;  // EOB
                    }
                    if (sz > 10) return LM_MJPEG_CATEGORY;
                    k += r;
                    if (k > 63) return LM_MJPEG_RUN;
                    const int level = extend(br.peek(sz), sz);
                    br.skip(sz);
                    if (keep) blk[zigzag(k)] = (int16_t)(level * (int)q[k]);
                    ++k;
                }
                if (br.overrun()) return LM_MJPEG_TRUNCATED;
                if (keep) {
                    int64_t idx;
                    if (c == 0) {
                        const int by = mcu_y * h.vy + b / h.hy, bx = mcu_x * h.hy + b % h.hy;
                        idx = (int64_t)by * ybx + bx;
                    } else {
                        idx = ny + m;
                    }
                    sink(idx, blk);
                }
            }
        }
    }
    return LM_MJPEG_OK;
}

// libavcodec simple_idct, 8 bits: ROW_SHIFT 11, COL_SHIFT 20, unsigned (wrapping) sums.
constexpr int W1 = 22725, W2 = 21407, W3 = 19266, W4 = 16383, W5 = 12873, W6 = 8867, W7 = 4520;

MJPEG_HD void idct_row(int16_t *r) {
    if (!(r[1] | r[2] | r[3] | r[4] | r[5] | r[6] | r[7])) {
        const int16_t t = (int16_t)(uint16_t)(((uint32_t)(int32_t)r[0] * 8u) & 0xffffu);
        for (int i = 0; i < 8; ++i) r[i] = t;
        return;
    }
    const int32_t x0 = r[0], x1 = r[1], x2 = r[2], x3 = r[3], x4 = r[4], x5 = r[5], x6 = r[6], x7 = r[7];
    uint32_t a0 = (uint32_t)(W4 * x0) + (1u << 10), a1 = a0, a2 = a0, a3 = a0;
    a0 += (uint32_t)(W2 * x2); a1 += (uint32_t)(W6 * x2); a2 -= (uint32_t)(W6 * x2); a3 -= (uint32_t)(W2 * x2);
    uint32_t b0 = (uint32_t)(W1 * x1) + (uint32_t)(W3 * x3), b1 = (uint32_t)(W3 * x1) - (uint32_t)(W7 * x3);
    uint32_t b2 = (uint32_t)(W5 * x1) - (uint32_t)(W1 * x3), b3 = (uint32_t)(W7 * x1) - (uint32_t)(W5 * x3);
    a0 += (uint32_t)(W4 * x4) + (uint32_t)(W6 * x6); a1 += (uint32_t)(-W4 * x4) - (uint32_t)(W2 * x6);
    a2 += (uint32_t)(-W4 * x4) + (uint32_t)(W2 * x6); a3 += (uint32_t)(W4 * x4) - (uint32_t)(W6 * x6);
    b0 += (uint32_t)(W5 * x5) + (uint32_t)(W7 * x7); b1 += (uint32_t)(-W1 * x5) - (uint32_t)(W5 * x7);
    b2 += (uint32_t)(W7 * x5) + (uint32_t)(W3 * x7); b3 += (uint32_t)(W3 * x5) - (uint32_t)(W1 * x7);
    r[0] = (int16_t)((int32_t)(a0 + b0) >> 11); r[7] = (int16_t)((int32_t)(a0 - b0) >> 11);
    r[1] = (int16_t)((int32_t)(a1 + b1) >> 11); r[6] = (int16_t)((int32_t)(a1 - b1) >> 11);
    r[2] = (int16_t)((int32_t)(a2 + b2) >> 11); r[5] = (int16_t)((int32_t)(a2 - b2) >> 11);
    r[3] = (int16_t)((int32_t)(a3 + b3) >> 11); r[4] = (int16_t)((int32_t)(a3 - b3) >> 11);
}

MJPEG_HD uint8_t clip_u8(int32_t v) { return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v); }

// column x of the row-transformed block -> 8 pixels at out[0], out[stride], ...
MJPEG_HD void idct_col(const int16_t *c, uint8_t *out, int stride) {
    const int32_t x0 = c[0], x1 = c[8], x2 = c[16], x3 = c[24], x4 = c[32], x5 = c[40], x6 = c[48], x7 = c[56];
    uint32_t a0 = (uint32_t)(W4 * (x0 + ((1 << 19) / W4))), a1 = a0, a2 = a0, a3 = a0;
    a0 += (uint32_t)(W2 * x2); a1 += (uint32_t)(W6 * x2); a2 += (uint32_t)(-W6 * x2); a3 += (uint32_t)(-W2 * x2);
    uint32_t b0 = (uint32_t)(W1 * x1), b1 = (uint32_t)(W3 * x1), b2 = (uint32_t)(W5 * x1), b3 = (uint32_t)(W7 * x1);
    b0 += (uint32_t)(W3 * x3); b1 += (uint32_t)(-W7 * x3); b2 += (uint32_t)(-W1 * x3); b3 += (uint32_t)(-W5 * x3);
    if (x4) { a0 += (uint32_t)(W4 * x4); a1 += (uint32_t)(-W4 * x4); a2 += (uint32_t)(-W4 * x4); a3 += (uint32_t)(W4 * x4); }
    if (x5) { b0 += (uint32_t)(W5 * x5); b1 += (uint32_t)(-W1 * x5); b2 += (uint32_t)(W7 * x5); b3 += (uint32_t)(W3 * x5); }
    if (x6) { a0 += (uint32_t)(W6 * x6); a1 += (uint32_t)(-W2 * x6); a2 += (uint32_t)(W2 * x6); a3 += (uint32_t)(-W6 * x6); }
    if (x7) { b0 += (uint32_t)(W7 * x7); b1 += (uint32_t)(-W5 * x7); b2 += (uint32_t)(W3 * x7); b3 += (uint32_t)(-W1 * x7); }
    out[0] = clip_u8((int32_t)(a0 + b0) >> 20); out[7 * stride] = clip_u8((int32_t)(a0 - b0) >> 20);
    out[1 * stride] = clip_u8((int32_t)(a1 + b1) >> 20); out[6 * stride] = clip_u8((int32_t)(a1 - b1) >> 20);
    out[2 * stride] = clip_u8((int32_t)(a2 + b2) >> 20); out[5 * stride] = clip_u8((int32_t)(a2 - b2) >> 20);
    out[3 * stride] = clip_u8((int32_t)(a3 + b3) >> 20); out[4 * stride] = clip_u8((int32_t)(a3 - b3) >> 20);
}

// 8 x 8 pixels of one coefficient block (natural order, 64 int16; transformed in place)
MJPEG_HD void idct_block(int16_t *blk, uint8_t px[64]) {
    for (int r = 0; r < 8; ++r) idct_row(blk + 8 * r);
    for (int c = 0; c < 8; ++c) idct_col(blk + c, px + c, 8);
}

// channel 0 of the BGR pixel VideoCapture gives for (Y, Cb)
MJPEG_HD uint8_t blue(int y, int cb) { return clip_u8((y * 8192 + (cb - 128) * 14516) >> 13); }

// Pixels of Y block (by, bx) into the frame out[rows][cols], cropped: grey, or blue from Y and the covering Cb block.
// coef: the frame's blocks (Header::blocks() layout); the blocks read are copied, not changed.
MJPEG_HD void put_y_block(const Header &h, const int16_t *coef, int by, int bx, uint8_t *out) {
    int16_t blk[64];
    uint8_t y[64], cb[64];
    const int16_t *src = coef + ((int64_t)by * h.y_blocks_x() + bx) * 64;
    for (int k = 0; k < 64; ++k) blk[k] = src[k];
    idct_block(blk, y);
    const int r0 = by * 8, c0 = bx * 8;
    if (h.ncomp == 3) {
        const int my = by / h.vy, mx = bx / h.hy;
        const int16_t *cs = coef + ((int64_t)h.y_blocks_x() * h.y_blocks_y() + (int64_t)my * h.mcus_x() + mx) * 64;
        for (int k = 0; k < 64; ++k) blk[k] = cs[k];
        idct_block(blk, cb);
        const int oy = (by % h.vy) * 8, ox = (bx % h.hy) * 8;  // the Y block's corner in the MCU, in Y samples
        for (int r = 0; r < 8; ++r)
            for (int c = 0; c < 8; ++c) y[r * 8 + c] = blue(y[r * 8 + c], cb[((oy + r) / h.vy) * 8 + (ox + c) / h.hy]);
    }
    for (int r = 0; r < 8 && r0 + r < h.rows; ++r)
        for (int c = 0; c < 8 && c0 + c < h.cols; ++c) out[(int64_t)(r0 + r) * h.cols + c0 + c] = y[r * 8 + c];
}

}  // namespace mjpeg
