// mpeg4_format.h — MPEG-4 Part 2 video (Simple / Advanced Simple profile streams as libavcodec's 'mpeg4' encoder writes them:
// cv2.VideoWriter 'mp4v' and 'XVID') as libavcodec's 'mpeg4' decoder reads them, reduced to channel 0 of the BGR frame
// cv::VideoCapture delivers.
//
// Shared by the host (the video index parses the VOL and every frame's VOP header; lmh_decode_mpeg4 runs the whole decode on
// the CPU for the tests) and by k_mpeg4.cu (k_mpeg4_locate runs parse() per frame, k_mpeg4_entropy runs decode_vop() per
// frame, k_mpeg4_recon runs build_mb() / put_mb() per macroblock).  Every function that touches stream bytes is bounded by
// the frame it reads: bytes past the end read as zero and are counted, every loop consumes input, and malformed data ends
// the frame with an LM_MPEG4_* status.
//
// The rules (libavcodec's mpeg4 decoder for streams whose user data names libavcodec, or none; see DESIGN §8):
//   - VLC tables of ISO/IEC 14496-2 Annex B; intra DC by the DC size VLCs (or in the TCOEF table when intra_dc_vlc_thr says
//     so, judged on the quantiser before the macroblock's dquant); DC / AC prediction on quantised levels with the
//     direction from the DC gradients, neighbours outside the VOP or not intra count as DC 1024 and AC 0, AC of a
//     neighbour with another quantiser rescaled by ROUNDED_DIV; H.263 dequantisation (intra after prediction, inter inside
//     the TCOEF decode, escape-3 inter levels clipped to -2048..2047); DC times the MPEG-4 dc_scaler.
//   - 1MV motion vectors: median prediction with libavcodec's first-row rule, f_code 1..7 and the wrap to 5 + f_code bits.
//   - Reconstruction: libavcodec's 8-bit simple IDCT (mjpeg_format.h) put for intra blocks, add over the half-pel
//     prediction for inter blocks.  The prediction reads the previous frame clamped to its macroblock-aligned size (the
//     unrestricted-vector edge of libavcodec without its old-encoder workaround).  rounding_type 1 uses the no-rounding
//     averages that libavcodec's x86 builds use outside bitexact mode (one operand lowered by one before a rounded average).
//   - Chroma vector of a 1MV macroblock: (v >> 1) | (v & 1) per component, half-pel on the chroma plane.
//   - A not-coded VOP (vop_coded = 0) gives no frame: libavcodec returns none for it, so VideoCapture reads one frame less.
//     The readers leave such frames out; the decoders refuse them.
//   - Channel 0: clip(((Y - 16) * 8 * 9539 >> 16) + ((Cb - 128) * 8 * 16525 >> 16)) with Cb nearest (one Cb per 2 x 2 Y).
//     Cr is entropy-decoded (the bit stream runs through it) but never reconstructed.
//   - Refused: B-VOPs, S-VOPs / sprites / GMC, quarter-pel, 4MV macroblocks, interlaced, non-rectangular shape, not-8-bit,
//     quant_type 1, complexity estimation, resync markers, data partitioning, newpred, reduced resolution, scalability,
//     short-header (H.263) frames, a VOL that differs from the stream's first, a VOL size other than the video's, and user
//     data that names XviD, DivX or a libavcodec build old enough to get bug workarounds.
#pragma once
#include <cstdint>

#include "mjpeg_format.h"

#ifdef __CUDACC__
#define MPEG4_HD __host__ __device__ __forceinline__
#else
#define MPEG4_HD inline
#endif

namespace mpeg4 {

// Per-frame status codes (k_mpeg4_locate / k_mpeg4_entropy write one per frame; -1 = not decoded)
enum {
    LM_MPEG4_OK = 0, LM_MPEG4_NO_VOP, LM_MPEG4_NO_VOL, LM_MPEG4_HEADER, LM_MPEG4_SHORT_HEADER, LM_MPEG4_SHAPE, LM_MPEG4_INTERLACED,
    LM_MPEG4_NOT_8BIT, LM_MPEG4_QUANT_TYPE, LM_MPEG4_QPEL, LM_MPEG4_SPRITE, LM_MPEG4_COMPLEXITY, LM_MPEG4_RESYNC, LM_MPEG4_PARTITIONED,
    LM_MPEG4_NEWPRED, LM_MPEG4_REDUCED, LM_MPEG4_SCALABILITY, LM_MPEG4_ENCODER, LM_MPEG4_VOL_CHANGE, LM_MPEG4_SIZE, LM_MPEG4_B_VOP,
    LM_MPEG4_S_VOP, LM_MPEG4_INTER4V, LM_MPEG4_FIRST_NOT_I, LM_MPEG4_CODE, LM_MPEG4_DC, LM_MPEG4_RUN, LM_MPEG4_MARKER,
    LM_MPEG4_TRUNCATED, LM_MPEG4_NOT_CODED, LM_MPEG4_ODD_HEIGHT
};

inline const char *status_text(int st) {
    switch (st) {
        case LM_MPEG4_OK: return "ok";
        case LM_MPEG4_NO_VOP: return "no VOP start code in the frame";
        case LM_MPEG4_NO_VOL: return "no video object layer (VOL) header before the first VOP, in the stream or its extradata";
        case LM_MPEG4_HEADER: return "truncated or malformed VOL / VOP header";
        case LM_MPEG4_SHORT_HEADER: return "short-header (H.263) MPEG-4 frames are not decoded";
        case LM_MPEG4_SHAPE: return "only rectangular video object layers are decoded (binary / grey shape)";
        case LM_MPEG4_INTERLACED: return "interlaced MPEG-4 video is not decoded";
        case LM_MPEG4_NOT_8BIT: return "only 8-bit MPEG-4 video is decoded (not_8_bit)";
        case LM_MPEG4_QUANT_TYPE: return "MPEG quantisation (quant_type 1) is not decoded, only H.263 quantisation";
        case LM_MPEG4_QPEL: return "quarter-pel motion compensation is not decoded";
        case LM_MPEG4_SPRITE: return "sprites and global motion compensation (S-VOPs) are not decoded";
        case LM_MPEG4_COMPLEXITY: return "complexity estimation headers are not decoded";
        case LM_MPEG4_RESYNC: return "resync markers / video packets are not decoded (resync_marker_disable is 0)";
        case LM_MPEG4_PARTITIONED: return "data partitioning and reversible VLC are not decoded";
        case LM_MPEG4_NEWPRED: return "newpred is not decoded";
        case LM_MPEG4_REDUCED: return "reduced-resolution VOPs are not decoded";
        case LM_MPEG4_SCALABILITY: return "scalable MPEG-4 video is not decoded";
        case LM_MPEG4_ENCODER:
            return "the stream's user data names XviD, DivX or an old libavcodec build, for which libavcodec switches IDCT or applies "
                   "bug workarounds that are not restated here";
        case LM_MPEG4_VOL_CHANGE: return "the frame carries a VOL that differs from the stream's first";
        case LM_MPEG4_SIZE: return "the VOL's frame size differs from the video's";
        case LM_MPEG4_B_VOP: return "B-VOPs are not decoded";
        case LM_MPEG4_S_VOP: return "S-VOPs (sprite / GMC) are not decoded";
        case LM_MPEG4_INTER4V: return "4MV (inter4v) macroblocks are not decoded";
        case LM_MPEG4_FIRST_NOT_I: return "the first frame is not an I-VOP";
        case LM_MPEG4_CODE: return "invalid VLC code in the macroblock data";
        case LM_MPEG4_DC: return "intra DC size out of range, or a negative intra DC, in the macroblock data";
        case LM_MPEG4_RUN: return "coefficient run past coefficient 63";
        case LM_MPEG4_MARKER: return "marker bit missing";
        case LM_MPEG4_TRUNCATED: return "the frame's data ends before its last macroblock";
        case LM_MPEG4_NOT_CODED:
            return "not-coded VOP (vop_coded 0): VideoCapture returns no frame for it, so it must be left out of the frames "
                   "(the video readers do)";
        case LM_MPEG4_ODD_HEIGHT: return "odd frame heights are not decoded (VideoCapture's frames of them follow another rule)";
        case -1: return "not decoded";
        default: return "unknown error";
    }
}

enum { VOP_I = 0, VOP_P = 1, VOP_N = 2 };  // N: not coded (no frame)

// What the VOL says; two VOLs of one stream must be equal in every field
struct Vol {
    int32_t width, height, time_res, time_bits, ver_id, vo_type, valid;
    MPEG4_HD bool same(const Vol &o) const {
        return width == o.width && height == o.height && time_res == o.time_res && ver_id == o.ver_id && vo_type == o.vo_type;
    }
};

struct Vop {
    int32_t type;      // VOP_I / VOP_P / VOP_N
    int32_t rounding;  // rounding_type (P)
    int32_t dc_thr;    // intra_dc_vlc_thr as a quantiser threshold (99: always the DC size VLCs, 0: never)
    int32_t quant, fcode;
    int64_t data_bit;  // macroblock data starts at this bit of the frame
};

// Per macroblock of a decoded frame: motion vector (half-pel) and what the coefficient blocks hold
struct MbInfo {
    int16_t mvx, mvy;
    uint8_t flags;  // bit 0: intra; bit 1 + b: block b (Y0..Y3, Cb) has coefficients (intra: all five)
    uint8_t pad_[3];
};
constexpr int BLOCKS_PER_MB = 5;  // Y0..Y3, Cb stored; Cr is decoded and dropped

// ---- bit reader -----------------------------------------------------------------------------------------------------
struct BitReader {
    const uint8_t *p, *end;
    uint64_t acc;  // MSB-first: the next bit is bit 63
    int nbits;
    int pad;       // zero bits fed past the data
    MPEG4_HD void init(const uint8_t *b, const uint8_t *e, int64_t bit) {
        p = b + (bit >> 3);
        end = e;
        acc = 0;
        nbits = 0;
        pad = 0;
        if (p > end) {
            pad = (int)((p - end) * 8 > 64 ? 64 : (p - end) * 8);
            p = end;
        }
        refill();
        skip((int)(bit & 7));
    }
    MPEG4_HD void refill() {  // at least 57 bits in acc
        if (nbits <= 56 && p + 8 <= end) {
            // eight bytes at once (independent loads); the bits past the whole bytes counted are the stream's next bits, which
            // a later refill ORs in again
            uint64_t w = 0;
            for (int i = 0; i < 8; ++i) w = (w << 8) | p[i];
            acc |= w >> nbits;
            const int k = (63 - nbits) >> 3;
            p += k;
            nbits += 8 * k;
            return;
        }
        while (nbits <= 56) {
            uint32_t b = 0;
            if (p < end) b = *p++;
            else pad += 8;
            acc |= (uint64_t)b << (56 - nbits);
            nbits += 8;
        }
    }
    MPEG4_HD uint32_t peek(int n) const { return n ? (uint32_t)(acc >> (64 - n)) : 0u; }
    MPEG4_HD void skip(int n) {
        acc <<= n;
        nbits -= n;
    }
    MPEG4_HD uint32_t get(int n) {  // n <= 32, refill() done by the caller for the bits asked
        const uint32_t v = peek(n);
        skip(n);
        return v;
    }
    MPEG4_HD uint32_t bits(int n) {  // with its own refill
        if (nbits < n) refill();
        return get(n);
    }
    MPEG4_HD bool overrun() const { return nbits < pad; }
    MPEG4_HD int64_t consumed_to(const uint8_t *begin) const { return (int64_t)(p - begin) * 8 - nbits + pad; }
};

// ---- VLC tables (ISO/IEC 14496-2 Annex B) ---------------------------------------------------------------------------
// Each table: {code, length} per symbol.  Table ids for code() / count():
enum { T_MCBPC_I = 0, T_MCBPC_P, T_CBPY, T_MVD, T_DC_LUM, T_DC_CHROM, T_TCOEF_INTRA, T_TCOEF_INTER, T_COUNT };
constexpr int TCOEF_ESC = 102;     // the escape symbol of both TCOEF tables
constexpr int MCBPC_I_STUFF = 8;   // I-VOP MCBPC: 0..3 intra cbpc, 4..7 intra+q cbpc, 8 stuffing
constexpr int MCBPC_P_STUFF = 20;  // P-VOP MCBPC: type * 4 + cbpc, types inter, inter+q, inter4v, intra, intra+q; 20 stuffing

MPEG4_HD int count(int t) {
    constexpr int n[T_COUNT] = {9, 21, 16, 33, 13, 13, 103, 103};
    return n[t];
}

// {code, length} of symbol s of table t
MPEG4_HD void code(int t, int s, int &c, int &len) {
    constexpr uint8_t mcbpc_i[9][2] = {{1, 1}, {1, 3}, {2, 3}, {3, 3}, {1, 4}, {1, 6}, {2, 6}, {3, 6}, {1, 9}};
    constexpr uint8_t mcbpc_p[21][2] = {{1, 1}, {3, 4}, {2, 4}, {5, 6}, {3, 3}, {7, 7}, {6, 7}, {5, 9}, {2, 3}, {5, 7}, {4, 7},
                                        {5, 8}, {3, 5}, {4, 8}, {3, 8}, {3, 7}, {4, 6}, {4, 9}, {3, 9}, {2, 9}, {1, 9}};
    constexpr uint8_t cbpy[16][2] = {{3, 4}, {5, 5}, {4, 5}, {9, 4}, {3, 5}, {7, 4}, {2, 6}, {11, 4},
                                     {2, 5}, {3, 6}, {5, 4}, {10, 4}, {4, 4}, {8, 4}, {6, 4}, {3, 2}};
    constexpr uint8_t mvd[33][2] = {{1, 1}, {1, 2}, {1, 3}, {1, 4}, {3, 6}, {5, 7}, {4, 7}, {3, 7}, {11, 9}, {10, 9}, {9, 9},
                                    {17, 10}, {16, 10}, {15, 10}, {14, 10}, {13, 10}, {12, 10}, {11, 10}, {10, 10}, {9, 10}, {8, 10}, {7, 10},
                                    {6, 10}, {5, 10}, {4, 10}, {7, 11}, {6, 11}, {5, 11}, {4, 11}, {3, 11}, {2, 11}, {3, 12}, {2, 12}};
    constexpr uint8_t dc_lum[13][2] = {{3, 3}, {3, 2}, {2, 2}, {2, 3}, {1, 3}, {1, 4}, {1, 5}, {1, 6}, {1, 7}, {1, 8}, {1, 9}, {1, 10}, {1, 11}};
    constexpr uint8_t dc_chrom[13][2] = {{3, 2}, {2, 2}, {1, 2}, {1, 3}, {1, 4}, {1, 5}, {1, 6}, {1, 7}, {1, 8}, {1, 9}, {1, 10}, {1, 11}, {1, 12}};
    constexpr uint8_t intra[103][2] = {
        {0x2, 2}, {0x6, 3}, {0xf, 4}, {0xd, 5}, {0xc, 5}, {0x15, 6}, {0x13, 6}, {0x12, 6}, {0x17, 7}, {0x1f, 8}, {0x1e, 8},
        {0x1d, 8}, {0x25, 9}, {0x24, 9}, {0x23, 9}, {0x21, 9}, {0x21, 10}, {0x20, 10}, {0xf, 10}, {0xe, 10}, {0x7, 11}, {0x6, 11},
        {0x20, 11}, {0x21, 11}, {0x50, 12}, {0x51, 12}, {0x52, 12}, {0xe, 4}, {0x14, 6}, {0x16, 7}, {0x1c, 8}, {0x20, 9}, {0x1f, 9},
        {0xd, 10}, {0x22, 11}, {0x53, 12}, {0x55, 12}, {0xb, 5}, {0x15, 7}, {0x1e, 9}, {0xc, 10}, {0x56, 12}, {0x11, 6}, {0x1b, 8},
        {0x1d, 9}, {0xb, 10}, {0x10, 6}, {0x22, 9}, {0xa, 10}, {0xd, 6}, {0x1c, 9}, {0x8, 10}, {0x12, 7}, {0x1b, 9}, {0x54, 12},
        {0x14, 7}, {0x1a, 9}, {0x57, 12}, {0x19, 8}, {0x9, 10}, {0x18, 8}, {0x23, 11}, {0x17, 8}, {0x19, 9}, {0x18, 9}, {0x7, 10},
        {0x58, 12}, {0x7, 4}, {0xc, 6}, {0x16, 8}, {0x17, 9}, {0x6, 10}, {0x5, 11}, {0x4, 11}, {0x59, 12}, {0xf, 6}, {0x16, 9},
        {0x5, 10}, {0xe, 6}, {0x4, 10}, {0x11, 7}, {0x24, 11}, {0x10, 7}, {0x25, 11}, {0x13, 7}, {0x5a, 12}, {0x15, 8}, {0x5b, 12},
        {0x14, 8}, {0x13, 8}, {0x1a, 8}, {0x15, 9}, {0x14, 9}, {0x13, 9}, {0x12, 9}, {0x11, 9}, {0x26, 11}, {0x27, 11}, {0x5c, 12},
        {0x5d, 12}, {0x5e, 12}, {0x5f, 12}, {0x3, 7}};
    constexpr uint8_t inter[103][2] = {
        {0x2, 2}, {0xf, 4}, {0x15, 6}, {0x17, 7}, {0x1f, 8}, {0x25, 9}, {0x24, 9}, {0x21, 10}, {0x20, 10}, {0x7, 11}, {0x6, 11},
        {0x20, 11}, {0x6, 3}, {0x14, 6}, {0x1e, 8}, {0xf, 10}, {0x21, 11}, {0x50, 12}, {0xe, 4}, {0x1d, 8}, {0xe, 10}, {0x51, 12},
        {0xd, 5}, {0x23, 9}, {0xd, 10}, {0xc, 5}, {0x22, 9}, {0x52, 12}, {0xb, 5}, {0xc, 10}, {0x53, 12}, {0x13, 6}, {0xb, 10},
        {0x54, 12}, {0x12, 6}, {0xa, 10}, {0x11, 6}, {0x9, 10}, {0x10, 6}, {0x8, 10}, {0x16, 7}, {0x55, 12}, {0x15, 7}, {0x14, 7},
        {0x1c, 8}, {0x1b, 8}, {0x21, 9}, {0x20, 9}, {0x1f, 9}, {0x1e, 9}, {0x1d, 9}, {0x1c, 9}, {0x1b, 9}, {0x1a, 9}, {0x22, 11},
        {0x23, 11}, {0x56, 12}, {0x57, 12}, {0x7, 4}, {0x19, 9}, {0x5, 11}, {0xf, 6}, {0x4, 11}, {0xe, 6}, {0xd, 6}, {0xc, 6},
        {0x13, 7}, {0x12, 7}, {0x11, 7}, {0x10, 7}, {0x1a, 8}, {0x19, 8}, {0x18, 8}, {0x17, 8}, {0x16, 8}, {0x15, 8}, {0x14, 8},
        {0x13, 8}, {0x18, 9}, {0x17, 9}, {0x16, 9}, {0x15, 9}, {0x14, 9}, {0x13, 9}, {0x12, 9}, {0x11, 9}, {0x7, 10}, {0x6, 10},
        {0x5, 10}, {0x4, 10}, {0x24, 11}, {0x25, 11}, {0x26, 11}, {0x27, 11}, {0x58, 12}, {0x59, 12}, {0x5a, 12}, {0x5b, 12},
        {0x5c, 12}, {0x5d, 12}, {0x5e, 12}, {0x5f, 12}, {0x3, 7}};
    const uint8_t *e = t == T_MCBPC_I ? mcbpc_i[s] : t == T_MCBPC_P ? mcbpc_p[s] : t == T_CBPY ? cbpy[s] : t == T_MVD ? mvd[s]
                     : t == T_DC_LUM ? dc_lum[s] : t == T_DC_CHROM ? dc_chrom[s] : t == T_TCOEF_INTRA ? intra[s] : inter[s];
    c = e[0];
    len = e[1];
}

// (last, run, level) of TCOEF symbol s (not the escape); intra: the intra table
MPEG4_HD void tcoef_event(int intra, int s, int &last, int &run, int &level) {
    constexpr int8_t intra_level[102] = {1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 1, 2, 3, 4, 5, 1, 2, 3, 4, 1, 2, 3, 1, 2, 3, 1, 2, 3, 1, 2, 3, 1, 2, 1, 2, 1, 1, 1, 1, 1, 1, 2, 3, 4, 5, 6, 7, 8, 1, 2, 3, 1, 2, 1, 2, 1, 2, 1, 2, 1, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1};
    constexpr int8_t intra_run[102] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1,
                                       1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 5, 5, 5, 6, 6, 6, 7, 7, 7, 8, 8, 9, 9, 10, 11,
                                       12, 13, 14, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 8, 9, 10, 11, 12, 13, 14,
                                       15, 16, 17, 18, 19, 20};
    constexpr int8_t inter_level[102] = {1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 1, 2, 3, 4, 5, 6, 1, 2, 3, 4, 1, 2, 3, 1, 2, 3, 1, 2, 3, 1,
                                         2, 3, 1, 2, 1, 2, 1, 2, 1, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 3, 1, 2, 1,
                                         1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                                         1, 1, 1, 1, 1, 1};
    constexpr int8_t inter_run[102] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 4, 4, 4, 5, 5, 5, 6,
                                       6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 0, 0, 0, 1,
                                       1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30,
                                       31, 32, 33, 34, 35, 36, 37, 38, 39, 40};
    last = s >= (intra ? 67 : 58);
    run = intra ? intra_run[s] : inter_run[s];
    level = intra ? intra_level[s] : inter_level[s];
}

// Scans: 0 zigzag, 1 alternate horizontal (AC predicted from above), 2 alternate vertical (from the left)
MPEG4_HD int scan_pos(int which, int k) {
    constexpr uint8_t alt_h[64] = {0,  1,  2,  3,  8,  9,  16, 17, 10, 11, 4,  5,  6,  7,  15, 14, 13, 12, 19, 18, 24, 25,
                                   32, 33, 26, 27, 20, 21, 22, 23, 28, 29, 30, 31, 34, 35, 40, 41, 48, 49, 42, 43, 36, 37,
                                   38, 39, 44, 45, 46, 47, 50, 51, 56, 57, 58, 59, 52, 53, 54, 55, 60, 61, 62, 63};
    constexpr uint8_t alt_v[64] = {0,  8,  16, 24, 1,  9,  2,  10, 17, 25, 32, 40, 48, 56, 57, 49, 41, 33, 26, 18, 3,  11,
                                   4,  12, 19, 27, 34, 42, 50, 58, 35, 43, 51, 59, 20, 28, 5,  13, 6,  14, 21, 29, 36, 44,
                                   52, 60, 37, 45, 53, 61, 22, 30, 7,  15, 23, 31, 38, 46, 54, 62, 39, 47, 55, 63};
    return which == 0 ? mjpeg::zigzag(k) : which == 1 ? alt_h[k] : alt_v[k];
}

// Lookahead tables of every VLC table, the scans and the escape limits: built once (build_tables), read by decode_vop.
// A lookahead entry is length << 8 | symbol, 0 for a prefix no code has.
constexpr int LUT_BITS = 12;
struct Tables {
    uint16_t tcoef[2][1 << LUT_BITS];  // [intra]
    uint16_t mvd[1 << LUT_BITS];
    uint16_t dc[2][1 << LUT_BITS];     // [chroma]
    uint16_t mcbpc[2][1 << 9];         // [P]
    uint16_t cbpy[1 << 6];
    uint8_t scan[3][64];
    uint8_t run[2][103], level[2][103], last[2][103];
    int8_t max_level[2][2][64];        // [intra][last][run]
    int8_t max_run[2][2][32];          // [intra][last][level]
};

MPEG4_HD uint16_t *lut_of(Tables &T, int t, int &bits) {
    switch (t) {
        case T_MCBPC_I: bits = 9; return T.mcbpc[0];
        case T_MCBPC_P: bits = 9; return T.mcbpc[1];
        case T_CBPY: bits = 6; return T.cbpy;
        case T_MVD: bits = LUT_BITS; return T.mvd;
        case T_DC_LUM: bits = LUT_BITS; return T.dc[0];
        case T_DC_CHROM: bits = LUT_BITS; return T.dc[1];
        case T_TCOEF_INTRA: bits = LUT_BITS; return T.tcoef[1];
        default: bits = LUT_BITS; return T.tcoef[0];
    }
}

// Phase 0 clears the lookahead tables, phase 1 fills them and the rest; work item i of n (threads of a CTA, or 0 of 1).
// Codes of one table are prefix-free, so the ranges phase 1 writes are disjoint.
MPEG4_HD void build_tables(Tables &T, int phase, int i, int n) {
    if (phase == 0) {
        uint16_t *w = &T.tcoef[0][0];
        const int words = (int)((sizeof(T.tcoef) + sizeof(T.mvd) + sizeof(T.dc) + sizeof(T.mcbpc) + sizeof(T.cbpy)) / 2);
        for (int k = i; k < words; k += n) w[k] = 0;
        return;
    }
    int item = 0;
    for (int t = 0; t < T_COUNT; ++t)
        for (int s = 0; s < count(t); ++s, ++item) {
            if (item % n != i) continue;
            int c, len, bits;
            code(t, s, c, len);
            uint16_t *lut = lut_of(T, t, bits);
            const int lo = c << (bits - len), hi = (c + 1) << (bits - len);
            for (int j = lo; j < hi; ++j) lut[j] = (uint16_t)((len << 8) | s);
        }
    if (i == 0) {
        for (int w = 0; w < 3; ++w)
            for (int k = 0; k < 64; ++k) T.scan[w][k] = (uint8_t)scan_pos(w, k);
        for (int intra = 0; intra < 2; ++intra) {
            for (int l = 0; l < 2; ++l) {
                for (int r = 0; r < 64; ++r) T.max_level[intra][l][r] = 0;
                for (int v = 0; v < 32; ++v) T.max_run[intra][l][v] = 0;
            }
            for (int s = 0; s < TCOEF_ESC; ++s) {
                int last, run, level;
                tcoef_event(intra, s, last, run, level);
                T.run[intra][s] = (uint8_t)run;
                T.level[intra][s] = (uint8_t)level;
                T.last[intra][s] = (uint8_t)last;
                if (level > T.max_level[intra][last][run]) T.max_level[intra][last][run] = (int8_t)level;
                if (run > T.max_run[intra][last][level]) T.max_run[intra][last][level] = (int8_t)run;
            }
        }
    }
}

// ---- headers --------------------------------------------------------------------------------------------------------

// Bytes [p, end) of one start-code segment: from after its 00 00 01 xx to the next start code (or the end)
MPEG4_HD int64_t next_start(const uint8_t *d, int64_t p, int64_t len) {
    for (; p + 3 < len; ++p)
        if (d[p] == 0 && d[p + 1] == 0 && d[p + 2] == 1) return p;
    return len;
}

MPEG4_HD bool prefix(const uint8_t *d, int64_t n, const char *s) {
    int64_t i = 0;
    for (; s[i]; ++i)
        if (i >= n || d[i] != (uint8_t)s[i]) return false;
    return true;
}

// User data that makes libavcodec change its decoding: XviD / DivX builds, and libavcodec builds that get workarounds
// (those up to 4712, and the 'FFmpeg' / 'ffmpeg' strings of old builds).  0 = fine, else LM_MPEG4_ENCODER.
MPEG4_HD int check_user_data(const uint8_t *d, int64_t n) {
    if (prefix(d, n, "XviD") || prefix(d, n, "DivX") || prefix(d, n, "FFmpe") || prefix(d, n, "ffmpeg")) return LM_MPEG4_ENCODER;
    if (prefix(d, n, "Lavc")) {
        int v[3] = {0, 0, 0}, k = 0;
        int64_t i = 4;
        for (; k < 3; ++k) {
            if (i >= n || d[i] < '0' || d[i] > '9') break;
            while (i < n && d[i] >= '0' && d[i] <= '9' && v[k] < 100000) v[k] = v[k] * 10 + (d[i++] - '0');
            if (k < 2) {
                if (i >= n || d[i] != '.') { ++k; break; }
                ++i;
            }
        }
        if (k == 3 && v[0] <= 255 && v[1] <= 255 && v[2] <= 255 && (v[0] << 16) + (v[1] << 8) + v[2] <= 4712) return LM_MPEG4_ENCODER;
    }
    return LM_MPEG4_OK;
}

// The video object layer header after its start code (bytes [0, n))
MPEG4_HD int parse_vol(const uint8_t *d, int64_t n, Vol &v) {
    BitReader br;
    br.init(d, d + n, 0);
    br.bits(1);  // random_accessible_vol
    v.vo_type = (int)br.bits(8);
    if (br.bits(1)) {
        v.ver_id = (int)br.bits(4);
        br.bits(3);
    } else {
        v.ver_id = 1;
    }
    if (br.bits(4) == 15) br.bits(16);  // extended pixel aspect ratio
    if (br.bits(1)) {                   // vol_control_parameters
        br.bits(2);                     // chroma_format
        br.bits(1);                     // low_delay
        if (br.bits(1)) {               // vbv_parameters
            br.bits(32);
            br.bits(32);
            br.bits(15);
        }
    }
    const int shape = (int)br.bits(2);
    if (shape != 0) return LM_MPEG4_SHAPE;
    br.bits(1);
    const int res = (int)br.bits(16);
    if (res == 0) return LM_MPEG4_HEADER;
    v.time_res = res;
    int tb = 0;
    while ((1 << tb) < res) ++tb;  // av_log2(res - 1) + 1
    v.time_bits = tb < 1 ? 1 : tb;
    br.bits(1);
    if (br.bits(1)) br.bits(v.time_bits);  // fixed_vop_rate
    br.bits(1);
    v.width = (int)br.bits(13);
    br.bits(1);
    v.height = (int)br.bits(13);
    br.bits(1);
    if (br.bits(1)) return LM_MPEG4_INTERLACED;
    br.bits(1);  // obmc_disable
    if (br.bits(v.ver_id == 1 ? 1 : 2)) return LM_MPEG4_SPRITE;
    if (br.bits(1)) return LM_MPEG4_NOT_8BIT;
    if (br.bits(1)) return LM_MPEG4_QUANT_TYPE;
    if (v.ver_id != 1 && br.bits(1)) return LM_MPEG4_QPEL;
    if (!br.bits(1)) return LM_MPEG4_COMPLEXITY;
    if (!br.bits(1)) return LM_MPEG4_RESYNC;
    if (br.bits(1)) return LM_MPEG4_PARTITIONED;
    if (v.ver_id != 1) {
        if (br.bits(1)) return LM_MPEG4_NEWPRED;
        if (br.bits(1)) return LM_MPEG4_REDUCED;
    }
    if (br.bits(1)) return LM_MPEG4_SCALABILITY;
    if (br.overrun() || v.width <= 0 || v.height <= 0) return LM_MPEG4_HEADER;
    if (v.height & 1) return LM_MPEG4_ODD_HEIGHT;
    v.valid = 1;
    return LM_MPEG4_OK;
}

// The VOP header after its start code; vop.data_bit is relative to d
MPEG4_HD int parse_vop(const uint8_t *d, int64_t n, const Vol &vol, Vop &vop) {
    BitReader br;
    br.init(d, d + n, 0);
    const int type = (int)br.bits(2);
    if (type == 2) return LM_MPEG4_B_VOP;
    if (type == 3) return LM_MPEG4_S_VOP;
    for (int k = 0; br.bits(1); ++k)  // modulo_time_base
        if (br.overrun()) return LM_MPEG4_HEADER;
    if (!br.bits(1)) return LM_MPEG4_MARKER;
    br.bits(vol.time_bits);
    if (!br.bits(1)) return LM_MPEG4_MARKER;  // libavcodec would guess another increment width
    vop.type = type;
    vop.rounding = 0;
    vop.fcode = 1;
    vop.dc_thr = 99;
    vop.quant = 1;
    if (!br.bits(1)) {  // vop_coded = 0
        vop.type = VOP_N;
        vop.data_bit = br.consumed_to(d);
        return br.overrun() ? LM_MPEG4_HEADER : LM_MPEG4_OK;
    }
    if (type == VOP_P) vop.rounding = (int)br.bits(1);
    constexpr int thr[8] = {99, 13, 15, 17, 19, 21, 23, 0};
    vop.dc_thr = thr[br.bits(3)];
    vop.quant = (int)br.bits(5);
    if (vop.quant == 0) return LM_MPEG4_HEADER;
    if (type == VOP_P) {
        vop.fcode = (int)br.bits(3);
        if (vop.fcode == 0) return LM_MPEG4_HEADER;
    }
    vop.data_bit = br.consumed_to(d);
    return br.overrun() ? LM_MPEG4_HEADER : LM_MPEG4_OK;
}

// Walks the start codes of a frame (want_vop) or of extradata (!want_vop).  vol: the stream's VOL so far (vol.valid = 0:
// none yet; a VOL found here becomes it; a VOL that differs from it is refused).  rows / cols: the video's size (0: any).
// For a frame, decodes its VOP header into vop (data_bit relative to d).
MPEG4_HD int parse(const uint8_t *d, int64_t len, int rows, int cols, bool want_vop, Vol &vol, Vop &vop) {
    if (want_vop && len >= 3 && d[0] == 0 && d[1] == 0 && (d[2] & 0xFC) == 0x80) return LM_MPEG4_SHORT_HEADER;
    int64_t p = next_start(d, 0, len);
    bool vol_here = false;
    while (p < len) {
        const int c = d[p + 3];
        const int64_t s = p + 4;
        if (c == 0xB6) {
            if (!want_vop) return LM_MPEG4_HEADER;
            if (!vol.valid) return LM_MPEG4_NO_VOL;
            const int st = parse_vop(d + s, len - s, vol, vop);
            vop.data_bit += s * 8;
            return st;
        }
        const int64_t e = next_start(d, s, len);
        if (c >= 0x20 && c <= 0x2F) {
            if (!vol_here) {  // libavcodec reads the first VOL of a packet and ignores others
                Vol v;
                v.valid = 0;
                const int st = parse_vol(d + s, e - s, v);
                if (st) return st;
                if (vol.valid && !vol.same(v)) return LM_MPEG4_VOL_CHANGE;
                if ((rows || cols) && (v.width != cols || v.height != rows)) return LM_MPEG4_SIZE;
                vol = v;
                vol_here = true;
            }
        } else if (c == 0xB2) {
            if (int st = check_user_data(d + s, e - s)) return st;
        }
        p = e;
    }
    return want_vop ? LM_MPEG4_NO_VOP : LM_MPEG4_OK;
}

// ---- macroblock layer -----------------------------------------------------------------------------------------------

MPEG4_HD int vlc(BitReader &br, const uint16_t *lut, int bits) {  // symbol or -1; refill() done by the caller
    const uint16_t e = lut[br.peek(bits)];
    if (!e) return -1;
    br.skip(e >> 8);
    return e & 255;
}

MPEG4_HD int y_dc_scale(int q) { return q < 5 ? 8 : q < 9 ? 2 * q : q < 25 ? q + 8 : 2 * q - 16; }
MPEG4_HD int c_dc_scale(int q) { return q < 5 ? 8 : q < 25 ? (q + 13) / 2 : q - 6; }
MPEG4_HD int rounded_div(int a, int b) { return (a >= 0 ? a + (b >> 1) : a - (b >> 1)) / b; }
MPEG4_HD int median(int a, int b, int c) {
    const int mx = a > b ? a : b, mn = a < b ? a : b;
    return c > mx ? mx : c < mn ? mn : c;
}

// Prediction state of one block position: its DC (times dc_scaler, clipped as libavcodec stores it) and the first column
// (col, block[8 i]) and row (row, block[i]) of its quantised levels, i = 1..7
struct Pred {
    int16_t dc;
    int16_t col[7];
    int16_t row[7];
    int16_t pad_;
    MPEG4_HD void reset() {
        dc = 1024;
        for (int i = 0; i < 7; ++i) col[i] = row[i] = 0;
    }
};

// Working memory of decode_vop for one frame: what the macroblock row above left behind
struct Lines {
    Pred *ytop;      // [2 * mbw]: blocks 2 and 3 of each macroblock of the row above
    Pred *ctop;      // [2][mbw]: Cb, Cr of each macroblock of the row above
    int8_t *qtop;    // [mbw]: quantiser of each macroblock of the row above
    int32_t *mvtop;  // [mbw + 1]: motion vector (x | y << 16) of each macroblock of the row above; the last entry stays 0
};
MPEG4_HD int64_t lines_bytes(int mbw) { return (int64_t)mbw * (4 * (int64_t)sizeof(Pred) + 1 + 4) + 4 + 64; }
MPEG4_HD Lines lines_at(uint8_t *base, int mbw) {
    Lines L;
    L.ytop = reinterpret_cast<Pred *>(base);
    L.ctop = L.ytop + 2 * mbw;
    L.mvtop = reinterpret_cast<int32_t *>(L.ctop + 2 * mbw);
    L.qtop = reinterpret_cast<int8_t *>(L.mvtop + mbw + 1);
    return L;
}

// One TCOEF event, escapes resolved: quantised level (signed), run, last; esc3 set for the fixed-length escape.
MPEG4_HD int tcoef(BitReader &br, const Tables &T, int intra, int &last, int &run, int &level, bool &esc3) {
    br.refill();
    const uint16_t *lut = T.tcoef[intra];
    int s = vlc(br, lut, LUT_BITS);
    if (s < 0) return LM_MPEG4_CODE;
    esc3 = false;
    if (s != TCOEF_ESC) {
        last = T.last[intra][s];
        run = T.run[intra][s];
        level = T.level[intra][s];
    } else if (br.peek(1) == 0) {  // escape 1: level + LMAX(last, run)
        br.skip(1);
        s = vlc(br, lut, LUT_BITS);
        if (s < 0 || s == TCOEF_ESC) return LM_MPEG4_CODE;
        last = T.last[intra][s];
        run = T.run[intra][s];
        level = T.level[intra][s] + T.max_level[intra][last][run];
    } else if (br.peek(2) == 2) {  // escape 2: run + RMAX(last, level) + 1
        br.skip(2);
        s = vlc(br, lut, LUT_BITS);
        if (s < 0 || s == TCOEF_ESC) return LM_MPEG4_CODE;
        last = T.last[intra][s];
        level = T.level[intra][s];
        run = T.run[intra][s] + T.max_run[intra][last][level] + 1;
    } else {  // escape 3: last, run, level fixed-length between marker bits
        br.skip(2);
        last = (int)br.get(1);
        run = (int)br.get(6);
        if (!br.get(1)) return LM_MPEG4_MARKER;
        level = (int)(br.get(12) << 20) >> 20;
        if (!br.get(1)) return LM_MPEG4_MARKER;
        esc3 = true;
        return LM_MPEG4_OK;
    }
    if (br.get(1)) level = -level;
    return LM_MPEG4_OK;
}

// Decodes the macroblocks of one coded VOP.  For every macroblock calls info(mb, MbInfo) and, for each stored block with
// coefficients, block(mb, b, blk) with blk the dequantised coefficients in natural order (b: 0..3 Y, 4 Cb).
// mbw x mbh macroblocks; L: lines_at() of lines_bytes(mbw) bytes.  Returns a status.
template <class Info, class Block>
MPEG4_HD int decode_vop(const Tables &T, const Vop &vop, int mbw, int mbh, const uint8_t *frame, int64_t len, Lines L, Info &&info,
                        Block &&block) {
    BitReader br;
    br.init(frame, frame + len, vop.data_bit);
    for (int x = 0; x < 2 * mbw; ++x) L.ytop[x].reset();
    for (int x = 0; x < 2 * mbw; ++x) L.ctop[x].reset();
    for (int x = 0; x <= mbw; ++x) L.mvtop[x] = 0;
    int q = vop.quant;
    const bool P = vop.type == VOP_P;
    for (int my = 0; my < mbh; ++my) {
        Pred yleft[2], cleft[2], ydiag, cdiag[2];  // left: blocks 1 and 3 of the macroblock to the left; diag: above-left
        yleft[0].reset(), yleft[1].reset(), cleft[0].reset(), cleft[1].reset(), ydiag.reset(), cdiag[0].reset(), cdiag[1].reset();
        int qleft = q, mvleft = 0;
        for (int mx = 0; mx < mbw; ++mx) {
            const int mb = my * mbw + mx;
            MbInfo mi;
            mi.mvx = mi.mvy = 0;
            mi.flags = 0;
            mi.pad_[0] = mi.pad_[1] = mi.pad_[2] = 0;
            bool intra = true, skipped = false;
            int cbpc = 0, dquant = 0;
            for (;;) {  // stuffing repeats the macroblock header
                br.refill();
                if (P) {
                    if (br.get(1)) {
                        skipped = true;
                        break;
                    }
                    const int s = vlc(br, T.mcbpc[1], 9);
                    if (s < 0) return LM_MPEG4_CODE;
                    if (s == MCBPC_P_STUFF) continue;
                    const int type = s >> 2;
                    if (type == 2) return LM_MPEG4_INTER4V;
                    intra = type >= 3;
                    dquant = type == 1 || type == 4;
                    cbpc = s & 3;
                } else {
                    const int s = vlc(br, T.mcbpc[0], 9);
                    if (s < 0) return LM_MPEG4_CODE;
                    if (s == MCBPC_I_STUFF) continue;
                    dquant = s >= 4;
                    cbpc = s & 3;
                }
                break;
            }
            if (br.overrun()) return LM_MPEG4_TRUNCATED;
            Pred ycur[4], ccur[2];
            if (skipped || !intra) {
                for (int b = 0; b < 4; ++b) ycur[b].reset();
                ccur[0].reset(), ccur[1].reset();
            }
            int mv = 0;
            if (!skipped) {
                const int ac_pred = intra ? (int)br.get(1) : 0;
                const int cs = vlc(br, T.cbpy, 6);
                if (cs < 0) return LM_MPEG4_CODE;
                const int cbpy = intra ? cs : cs ^ 15;
                const bool dc_vlc = q < vop.dc_thr;
                if (dquant) {
                    constexpr int dq[4] = {-1, -2, 1, 2};
                    q += dq[br.get(2)];
                    q = q < 1 ? 1 : q > 31 ? 31 : q;
                }
                const int cbp = (cbpy << 2) | cbpc;  // bit 5 - b: block b coded
                if (!intra) {
                    int px, py;
                    if (my == 0) {
                        px = mx ? (int16_t)(mvleft & 0xFFFF) : 0;
                        py = mx ? (mvleft >> 16) : 0;
                    } else {
                        const int a = mx ? mvleft : 0, b = L.mvtop[mx], c = L.mvtop[mx + 1];
                        px = median((int16_t)(a & 0xFFFF), (int16_t)(b & 0xFFFF), (int16_t)(c & 0xFFFF));
                        py = median(a >> 16, b >> 16, c >> 16);
                    }
                    int v[2];
                    const int pr[2] = {px, py};
                    for (int k = 0; k < 2; ++k) {
                        br.refill();
                        const int m = vlc(br, T.mvd, LUT_BITS);
                        if (m < 0) return LM_MPEG4_CODE;
                        int val = pr[k];
                        if (m) {
                            const int sign = (int)br.get(1), shift = vop.fcode - 1;
                            int d = m;
                            if (shift) d = (((d - 1) << shift) | (int)br.get(shift)) + 1;
                            val += sign ? -d : d;
                            const int w = 5 + vop.fcode;  // wrap to w bits, signed
                            val = (int)((uint32_t)val << (32 - w)) >> (32 - w);
                        }
                        v[k] = val;
                    }
                    mi.mvx = (int16_t)v[0];
                    mi.mvy = (int16_t)v[1];
                    mv = (v[0] & 0xFFFF) | (v[1] << 16);
                    const int qmul = 2 * q, qadd = (q - 1) | 1;
                    for (int b = 0; b < 6; ++b) {
                        if (!(cbp & (32 >> b))) continue;
                        alignas(16) int16_t blk[64];
                        for (int k = 0; k < 64; ++k) blk[k] = 0;
                        for (int pos = -1;;) {
                            int last, run, level;
                            bool esc3;
                            if (int st = tcoef(br, T, 0, last, run, level, esc3)) return st;
                            pos += run + 1;
                            if (pos > 63 || (!last && pos > 62)) return LM_MPEG4_RUN;
                            int dq = level > 0 ? level * qmul + qadd : level * qmul - qadd;
                            if (esc3) dq = dq < -2048 ? -2048 : dq > 2047 ? 2047 : dq;
                            blk[T.scan[0][pos]] = (int16_t)dq;
                            if (last) break;
                        }
                        if (br.overrun()) return LM_MPEG4_TRUNCATED;
                        if (b < 5) {
                            mi.flags |= (uint8_t)(2 << b);
                            block(mb, b, blk);
                        }
                    }
                } else {
                    mi.flags = 1 | (31 << 1);
                    const int qmul = 2 * q, qadd = (q - 1) | 1;
                    for (int b = 0; b < 6; ++b) {
                        const bool chroma = b >= 4;
                        const int scale = chroma ? c_dc_scale(q) : y_dc_scale(q);
                        // neighbours A (left), B (above-left), C (above), and whether the AC of A / C needs rescaling
                        const Pred *A, *B, *C;
                        int qa = q, qc = q;
                        if (b == 0) A = &yleft[0], B = &ydiag, C = &L.ytop[2 * mx], qa = qleft, qc = L.qtop[mx];
                        else if (b == 1) A = &ycur[0], B = &L.ytop[2 * mx], C = &L.ytop[2 * mx + 1], qc = L.qtop[mx];
                        else if (b == 2) A = &yleft[1], B = &yleft[0], C = &ycur[0], qa = qleft;
                        else if (b == 3) A = &ycur[2], B = &ycur[0], C = &ycur[1];
                        else A = &cleft[b - 4], B = &cdiag[b - 4], C = &L.ctop[(b - 4) * mbw + mx], qa = qleft, qc = L.qtop[mx];
                        if (mx == 0) qa = q;  // outside: DC 1024, AC 0 (the reset states), never rescaled
                        if (my == 0) qc = q;
                        const int a = A->dc, bb = B->dc, c = C->dc;
                        const int ab = a - bb < 0 ? bb - a : a - bb, bc = bb - c < 0 ? c - bb : bb - c;
                        const int dir = ab < bc;  // 1: from above (C), 0: from the left (A)
                        const int pred = ((dir ? c : a) + (scale >> 1)) / scale;
                        alignas(16) int16_t blk[64];
                        for (int k = 0; k < 64; ++k) blk[k] = 0;
                        int pos = -1;
                        br.refill();
                        if (dc_vlc) {
                            const int size = vlc(br, T.dc[chroma], LUT_BITS);
                            if (size < 0) return LM_MPEG4_CODE;
                            if (size > 9) return LM_MPEG4_DC;
                            int diff = 0;
                            if (size) {
                                const int v = (int)br.get(size);
                                diff = v < (1 << (size - 1)) ? v - (1 << size) + 1 : v;
                                if (size > 8) br.get(1);  // marker (libavcodec does not insist)
                            }
                            if (diff + pred < 0) return LM_MPEG4_DC;  // libavcodec: an error, not a clip
                            blk[0] = (int16_t)(diff + pred);
                            pos = 0;
                        }
                        if (cbp & (32 >> b)) {
                            const uint8_t *scan = T.scan[ac_pred ? (dir ? 1 : 2) : 0];
                            for (;;) {
                                int last, run, level;
                                bool esc3;
                                if (int st = tcoef(br, T, 1, last, run, level, esc3)) return st;
                                pos += run + 1;
                                if (pos > 63 || (!last && pos > 62)) return LM_MPEG4_RUN;
                                blk[scan[pos]] = (int16_t)level;
                                if (last) break;
                            }
                        }
                        if (br.overrun()) return LM_MPEG4_TRUNCATED;
                        if (!dc_vlc) blk[0] = (int16_t)(blk[0] + pred);
                        int dcs = blk[0] * scale;  // the predictor libavcodec stores
                        if (dcs & ~2047) dcs = dcs < 0 ? 0 : 2047;
                        if (ac_pred) {
                            if (dir == 0) {
                                for (int i = 1; i < 8; ++i)
                                    blk[8 * i] = (int16_t)(blk[8 * i] + (qa == q ? A->col[i - 1] : rounded_div(A->col[i - 1] * qa, q)));
                            } else {
                                for (int i = 1; i < 8; ++i)
                                    blk[i] = (int16_t)(blk[i] + (qc == q ? C->row[i - 1] : rounded_div(C->row[i - 1] * qc, q)));
                            }
                        }
                        Pred &own = chroma ? ccur[b - 4] : ycur[b];
                        own.dc = (int16_t)dcs;
                        for (int i = 1; i < 8; ++i) own.col[i - 1] = blk[8 * i], own.row[i - 1] = blk[i];
                        if (b < 5) {
                            blk[0] = (int16_t)(blk[0] * scale);
                            for (int k = 1; k < 64; ++k) {
                                const int l = blk[k];
                                if (l) blk[k] = (int16_t)(l > 0 ? l * qmul + qadd : l * qmul - qadd);
                            }
                            block(mb, b, blk);
                        }
                    }
                }
            }
            info(mb, mi);
            // what the next macroblock and the next row see
            ydiag = L.ytop[2 * mx + 1];
            cdiag[0] = L.ctop[mx];
            cdiag[1] = L.ctop[mbw + mx];
            yleft[0] = ycur[1];
            yleft[1] = ycur[3];
            cleft[0] = ccur[0];
            cleft[1] = ccur[1];
            L.ytop[2 * mx] = ycur[2];
            L.ytop[2 * mx + 1] = ycur[3];
            L.ctop[mx] = ccur[0];
            L.ctop[mbw + mx] = ccur[1];
            L.qtop[mx] = (int8_t)q;
            qleft = q;
            L.mvtop[mx] = mvleft = mv;
        }
    }
    return LM_MPEG4_OK;
}

// ---- reconstruction -------------------------------------------------------------------------------------------------

// libavcodec simple_idct add: column x of the row-transformed block added to 8 pixels at px[0], px[stride], ...
MPEG4_HD void idct_col_add(const int16_t *c, uint8_t *px, int stride) {
    using namespace mjpeg;
    const int32_t x0 = c[0], x1 = c[8], x2 = c[16], x3 = c[24], x4 = c[32], x5 = c[40], x6 = c[48], x7 = c[56];
    uint32_t a0 = (uint32_t)(W4 * (x0 + ((1 << 19) / W4))), a1 = a0, a2 = a0, a3 = a0;
    a0 += (uint32_t)(W2 * x2); a1 += (uint32_t)(W6 * x2); a2 += (uint32_t)(-W6 * x2); a3 += (uint32_t)(-W2 * x2);
    uint32_t b0 = (uint32_t)(W1 * x1), b1 = (uint32_t)(W3 * x1), b2 = (uint32_t)(W5 * x1), b3 = (uint32_t)(W7 * x1);
    b0 += (uint32_t)(W3 * x3); b1 += (uint32_t)(-W7 * x3); b2 += (uint32_t)(-W1 * x3); b3 += (uint32_t)(-W5 * x3);
    if (x4) { a0 += (uint32_t)(W4 * x4); a1 += (uint32_t)(-W4 * x4); a2 += (uint32_t)(-W4 * x4); a3 += (uint32_t)(W4 * x4); }
    if (x5) { b0 += (uint32_t)(W5 * x5); b1 += (uint32_t)(-W1 * x5); b2 += (uint32_t)(W7 * x5); b3 += (uint32_t)(W3 * x5); }
    if (x6) { a0 += (uint32_t)(W6 * x6); a1 += (uint32_t)(-W2 * x6); a2 += (uint32_t)(W2 * x6); a3 += (uint32_t)(-W6 * x6); }
    if (x7) { b0 += (uint32_t)(W7 * x7); b1 += (uint32_t)(-W5 * x7); b2 += (uint32_t)(W3 * x7); b3 += (uint32_t)(-W1 * x7); }
    px[0] = clip_u8(px[0] + ((int32_t)(a0 + b0) >> 20)); px[7 * stride] = clip_u8(px[7 * stride] + ((int32_t)(a0 - b0) >> 20));
    px[stride] = clip_u8(px[stride] + ((int32_t)(a1 + b1) >> 20)); px[6 * stride] = clip_u8(px[6 * stride] + ((int32_t)(a1 - b1) >> 20));
    px[2 * stride] = clip_u8(px[2 * stride] + ((int32_t)(a2 + b2) >> 20)); px[5 * stride] = clip_u8(px[5 * stride] + ((int32_t)(a2 - b2) >> 20));
    px[3 * stride] = clip_u8(px[3 * stride] + ((int32_t)(a3 + b3) >> 20)); px[4 * stride] = clip_u8(px[4 * stride] + ((int32_t)(a3 - b3) >> 20));
}

// Half-pel prediction of the 8 x 8 block at (x0, y0) of a w x h plane (w, h multiples of 8) displaced by (vx, vy) half
// pels, reading the plane clamped to its edges.  rnd = 0: rounding_type 1.  Without rounding, one operand of a two-tap
// average is lowered by one (saturating) before the rounded average: the left one across, and the one of odd row parity
// (counted from the block's first source row) down -- libavcodec's x86 no-rounding averages, exact for the four-tap one.
MPEG4_HD void predict(const uint8_t *ref, int w, int h, int x0, int y0, int vx, int vy, int rounding, uint8_t out[64]) {
    const int sx = x0 + (vx >> 1), sy = y0 + (vy >> 1), dx = vx & 1, dy = vy & 1;
    for (int r = 0; r < 8; ++r) {
        const int ya = sy + r < 0 ? 0 : sy + r >= h ? h - 1 : sy + r;
        const int yb = sy + r + 1 < 0 ? 0 : sy + r + 1 >= h ? h - 1 : sy + r + 1;
        const uint8_t *ra = ref + (int64_t)ya * w, *rb = ref + (int64_t)yb * w;
        for (int c = 0; c < 8; ++c) {
            const int xa = sx + c < 0 ? 0 : sx + c >= w ? w - 1 : sx + c;
            const int xb = sx + c + 1 < 0 ? 0 : sx + c + 1 >= w ? w - 1 : sx + c + 1;
            int v;
            if (!dx && !dy) {
                v = ra[xa];
            } else if (dx && !dy) {
                const int a = ra[xa], b = ra[xb];
                v = rounding ? ((a > 0 ? a - 1 : 0) + b + 1) >> 1 : (a + b + 1) >> 1;
            } else if (!dx) {
                int a = ra[xa], b = rb[xa];
                if (rounding) {
                    if (r & 1) a = a > 0 ? a - 1 : 0;
                    else b = b > 0 ? b - 1 : 0;
                    v = (a + b + 1) >> 1;
                } else {
                    v = (a + b + 1) >> 1;
                }
            } else {
                v = (ra[xa] + ra[xb] + rb[xa] + rb[xb] + 2 - rounding) >> 2;
            }
            out[r * 8 + c] = (uint8_t)v;
        }
    }
}

// Macroblock (mx, my) of a frame into its Y plane cy [16 mbh][16 mbw] and Cb plane cc [8 mbh][8 mbw]: intra blocks by IDCT
// put, the others as the prediction from the previous frame's planes ry / rc plus the IDCT of their coefficients.
// coef: the macroblock's five blocks of 64 (those mi.flags marks).
MPEG4_HD void build_mb(int mbw, int mbh, int mx, int my, const MbInfo &mi, const int16_t *coef, int rounding, const uint8_t *ry,
                       const uint8_t *rc, uint8_t *cy, uint8_t *cc) {
    const int wy = 16 * mbw, hy = 16 * mbh, wc = 8 * mbw, hc = 8 * mbh;
    const bool intra = mi.flags & 1;
    const int cvx = (mi.mvx >> 1) | (mi.mvx & 1), cvy = (mi.mvy >> 1) | (mi.mvy & 1);
    for (int b = 0; b < BLOCKS_PER_MB; ++b) {
        const bool luma = b < 4;
        const int x0 = luma ? 16 * mx + 8 * (b & 1) : 8 * mx, y0 = luma ? 16 * my + 8 * (b >> 1) : 8 * my;
        const int w = luma ? wy : wc;
        uint8_t *dst = (luma ? cy : cc) + (int64_t)y0 * w + x0;
        alignas(16) uint8_t px[64];
        alignas(16) int16_t blk[64];
        const bool coded = mi.flags & (2 << b);
        if (coded)
            for (int k = 0; k < 64; ++k) blk[k] = coef[b * 64 + k];
        if (intra) {
            mjpeg::idct_block(blk, px);
        } else {
            predict(luma ? ry : rc, w, luma ? hy : hc, x0, y0, luma ? mi.mvx : cvx, luma ? mi.mvy : cvy, rounding, px);
            if (coded) {
                for (int r = 0; r < 8; ++r) mjpeg::idct_row(blk + 8 * r);
                for (int c = 0; c < 8; ++c) idct_col_add(blk + c, px + c, 8);
            }
        }
        for (int r = 0; r < 8; ++r)
            for (int c = 0; c < 8; ++c) dst[(int64_t)r * w + c] = px[r * 8 + c];
    }
}

// channel 0 of the BGR pixel VideoCapture gives for (Y, Cb) of 4:2:0 MPEG-4 video (libswscale's yuv420p -> bgr24)
MPEG4_HD uint8_t blue(int y, int cb) { return mjpeg::clip_u8(((((y - 16) * 8) * 9539) >> 16) + ((((cb - 128) * 8) * 16525) >> 16)); }

// The displayed part of macroblock (mx, my) from the planes into out [rows][cols]
MPEG4_HD void put_mb(int mbw, int mx, int my, const uint8_t *cy, const uint8_t *cc, int rows, int cols, uint8_t *out) {
    const int wy = 16 * mbw, wc = 8 * mbw;
    for (int r = 16 * my; r < 16 * my + 16 && r < rows; ++r)
        for (int c = 16 * mx; c < 16 * mx + 16 && c < cols; ++c)
            out[(int64_t)r * cols + c] = blue(cy[(int64_t)r * wy + c], cc[(int64_t)(r >> 1) * wc + (c >> 1)]);
}

}  // namespace mpeg4
