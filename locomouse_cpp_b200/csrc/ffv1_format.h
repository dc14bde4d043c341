// ffv1_format.h — FFV1 version 3 (RFC 9043) as libavcodec writes it into AVI files: the configuration record, the range
// coder, the Golomb-Rice sample coder and the serial decode of one slice chain.
//
// Shared by the host (the AVI reader checks the record and reads each frame's keyframe bit; the C ABI checks the record
// before any launch) and by k_ffv1.cu, whose threads each run decode_chain().  Every function that touches stream bytes
// is bounded by the slice it reads: bytes past the end read as zero and are counted, every loop consumes input or
// produces output, and malformed data ends the chain with an LM_FFV1_* status.
//
// The decode follows libavcodec's ffv1dec.c step for step, including the parts that are not in the RFC's prose: the
// two-line sample ring whose edge samples come from the line above, the 5-input context that reads line y - 2 out of the
// ring before it is overwritten, the run mode that keeps the context and sign of the pixel where the run started, and
// the VlcState update with its 16-bit error sum.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>

#ifdef __CUDACC__
#define FFV1_HD __host__ __device__ __forceinline__
#else
#define FFV1_HD inline
#endif

namespace ffv1 {

constexpr int CONTEXT_SIZE = 32;       // bytes of range-coder state per context
constexpr int MAX_QUANT_TABLES = 8;
constexpr int MAX_SLICES = 1024;
constexpr int MAX_CTX_PLANES = 3;      // context planes of version 3: luma / green, chroma / blue + red, alpha
constexpr int MAX_CONTEXTS = 16384;    // (32768 + 1) / 2: the largest context count a record can give

// Per-slice status codes (k_ffv1.cu writes one per frame and slice; -1 = not decoded)
enum {
    LM_FFV1_OK = 0, LM_FFV1_FOOTER, LM_FFV1_CRC, LM_FFV1_KEYFRAME, LM_FFV1_SLICE_HEADER, LM_FFV1_QUANT_INDEX,
    LM_FFV1_SYMBOL, LM_FFV1_TRUNCATED, LM_FFV1_SLICE_END
};

inline const char *status_text(int st) {
    switch (st) {
        case LM_FFV1_OK: return "ok";
        case LM_FFV1_FOOTER: return "the slice footers do not chain back to the start of the frame (truncated or corrupt frame)";
        case LM_FFV1_CRC: return "slice CRC mismatch";
        case LM_FFV1_KEYFRAME: return "keyframe bit differs from the frame's first decision";
        case LM_FFV1_SLICE_HEADER: return "slice header places the slice off its grid cell";
        case LM_FFV1_QUANT_INDEX: return "quant table index out of range, or changed inside a GOP";
        case LM_FFV1_SYMBOL: return "malformed range-coded symbol";
        case LM_FFV1_TRUNCATED: return "the slice data ends before its last sample";
        case LM_FFV1_SLICE_END: return "the range-coded slice does not end where its footer says";
        case -1: return "not decoded (an earlier frame of its GOP failed)";
        default: return "unknown error";
    }
}

// Tables the decoder reads per decision / per pixel (k_ffv1.cu keeps them in shared memory).
struct Tables {
    int16_t quant[MAX_QUANT_TABLES][5][256];
    uint8_t one_default[256], zero_default[256];  // ff_build_rac_states(0.05 * 2^32, 256 - 8)
    uint8_t one_slice[256], zero_slice[256];      // the slices' transitions: the default, or coder_type 2's custom table
};

struct Record {
    int version = 0, micro_version = 0, ac = 0, colorspace = 0, bits = 0, chroma_planes = 0, h_shift = 0, v_shift = 0;
    int transparency = 0, h_slices = 0, v_slices = 0, quant_table_count = 0, ec = 0, intra = 0, plane_count = 0;
    int context_count[MAX_QUANT_TABLES] = {};
    int64_t initial_offset[MAX_QUANT_TABLES] = {};  // byte offset of table i's initial states in the initial-state block, -1: all 128
    alignas(16) Tables t;  // copied to shared memory in 16-byte words
    FFV1_HD int slices() const { return h_slices * v_slices; }
    FFV1_HD int coded_planes() const { return colorspace == 0 ? 1 : 3 + transparency; }  // sample planes per slice
    FFV1_HD int ctx_planes() const { return colorspace == 0 ? 1 : 2 + transparency; }    // context planes they use
};

// ---- range coder (libavcodec rangecoder.h) -------------------------------------------------------------------------
struct RangeDec {
    const uint8_t *p, *end;
    uint32_t low, range;
    int overread;
    FFV1_HD void init(const uint8_t *buf, const uint8_t *e) {
        end = e;
        p = buf;
        low = 0;
        for (int i = 0; i < 2; ++i) low = (low << 8) | (p < end ? *p : 0u), ++p;
        range = 0xFF00;
        overread = 0;
        if (low >= 0xFF00) {
            low = 0xFF00;
            end = p;
        }
    }
    FFV1_HD int get(uint8_t &state, const uint8_t *one, const uint8_t *zero) {
        const uint32_t r1 = (range * state) >> 8;
        range -= r1;
        int bit;
        if (low < range) {
            state = zero[state];
            bit = 0;
        } else {
            low -= range;
            range = r1;
            state = one[state];
            bit = 1;
        }
        if (range < 0x100) {
            range <<= 8;
            low <<= 8;
            if (p < end) low += *p++;
            else ++overread;
        }
        return bit;
    }
    // get_symbol(); a run of more than 31 exponent bits sets `bad`
    FFV1_HD int symbol(uint8_t *st, bool is_signed, const uint8_t *one, const uint8_t *zero, bool &bad) {
        if (get(st[0], one, zero)) return 0;
        int e = 0;
        while (get(st[1 + (e < 9 ? e : 9)], one, zero)) {
            if (++e > 31) {
                bad = true;
                return 0;
            }
        }
        uint32_t a = 1;
        for (int i = e - 1; i >= 0; --i) a = 2 * a + get(st[22 + (i < 9 ? i : 9)], one, zero);
        const int neg = is_signed && get(st[11 + (e < 10 ? e : 10)], one, zero);
        return neg ? -(int)a : (int)a;
    }
};

inline void build_rac_states(uint8_t one_state[256], uint8_t zero_state[256]) {
    const int64_t one = 1LL << 32, factor = (int64_t)(0.05 * (double)(1LL << 32));
    const int max_p = 256 - 8;
    memset(one_state, 0, 256);
    memset(zero_state, 0, 256);
    int64_t p = one / 2;
    int last_p8 = 0;
    for (int i = 0; i < 128; ++i) {
        int p8 = (int)((256 * p + one / 2) >> 32);
        if (p8 <= last_p8) p8 = last_p8 + 1;
        if (last_p8 && last_p8 < 256 && p8 <= max_p) one_state[last_p8] = (uint8_t)p8;
        p += ((one - p) * factor + one / 2) >> 32;
        last_p8 = p8;
    }
    for (int i = 256 - max_p; i <= max_p; ++i) {
        if (one_state[i]) continue;
        int64_t q = (i * one + 128) >> 8;
        q += ((one - q) * factor + one / 2) >> 32;
        int p8 = (int)((256 * q + one / 2) >> 32);
        if (p8 <= i) p8 = i + 1;
        if (p8 > max_p) p8 = max_p;
        one_state[i] = (uint8_t)p8;
    }
    for (int i = 1; i < 255; ++i) zero_state[i] = (uint8_t)(256 - one_state[256 - i]);
}

// CRC-32, polynomial 0x04C11DB7, MSB first, initial value 0 (libavcodec's AV_CRC_32_IEEE as FFV1 uses it): a record or a
// slice that carries its CRC gives 0 over its whole length.
inline void crc_table(uint32_t t[256]) {
    for (uint32_t i = 0; i < 256; ++i) {
        uint32_t c = i << 24;
        for (int k = 0; k < 8; ++k) c = (c << 1) ^ (c & 0x80000000u ? 0x04C11DB7u : 0u);
        t[i] = c;
    }
}
FFV1_HD uint32_t crc_update(const uint32_t *t, uint32_t crc, uint8_t b) { return (crc << 8) ^ t[(crc >> 24) ^ b]; }

// The keyframe flag of a frame: its first range-coded decision (state 128, default transitions), from its first 2 bytes.
FFV1_HD int keyframe_bit(const uint8_t *p, int64_t len) {
    const uint32_t low = len >= 2 ? ((uint32_t)p[0] << 8) | p[1] : len == 1 ? (uint32_t)p[0] << 8 : 0u;
    return (low >= 0xFF00 ? 0xFF00u : low) >= 0xFF00u - ((0xFF00u * 128) >> 8);
}

// ---- configuration record --------------------------------------------------------------------------------------------
// Parses and checks an FFV1 record (AVI 'strf' bytes after the BITMAPINFOHEADER) for a rows x cols video.  Returns 0, or
// -1 with `why` naming the reason.  initial_states (may be null) receives the coded initial context states of every
// table that has them, CONTEXT_SIZE bytes per context, at rec.initial_offset[i].
inline int parse_record(const uint8_t *d, int64_t n, int rows, int cols, Record &rec, uint8_t *initial_states,
                        int64_t *initial_bytes, char *why, size_t why_cap) {
    auto fail = [&](const char *msg, long long a = 0, long long b = 0) {
        snprintf(why, why_cap, msg, a, b);
        return -1;
    };
    rec = Record();
    if (n <= 0) return fail("no FFV1 configuration record: FFV1 versions 0 and 1 are not decoded, only version 3");
    Tables &T = rec.t;
    build_rac_states(T.one_default, T.zero_default);
    RangeDec c;
    c.init(d, d + n);
    uint8_t st[CONTEXT_SIZE];
    memset(st, 128, sizeof st);
    bool bad = false;
    auto sym = [&](uint8_t *s, bool sg) { return c.symbol(s, sg, T.one_default, T.zero_default, bad); };
    rec.version = sym(st, false);
    if (rec.version != 3) return fail("FFV1 version %lld: only version 3 is decoded", rec.version);
    if (n < 4) return fail("configuration record of %lld bytes is too short", n);
    uint32_t ct[256], crc = 0;
    crc_table(ct);
    for (int64_t i = 0; i < n; ++i) crc = crc_update(ct, crc, d[i]);
    if (crc) return fail("configuration record CRC mismatch");
    c.end = d + n - 4;
    rec.micro_version = sym(st, false);
    rec.ac = sym(st, false);
    if (rec.ac < 0 || rec.ac > 2) return fail("coder_type %lld is not 0, 1 or 2", rec.ac);
    memcpy(T.one_slice, T.one_default, 256);
    memcpy(T.zero_slice, T.zero_default, 256);
    if (rec.ac == 2) {
        for (int i = 1; i < 256; ++i) {
            T.one_slice[i] = (uint8_t)(sym(st, true) + T.one_default[i]);
        }
        for (int i = 1; i < 256; ++i) T.zero_slice[256 - i] = (uint8_t)(256 - T.one_slice[i]);
    }
    rec.colorspace = sym(st, false);
    rec.bits = sym(st, false);
    rec.chroma_planes = c.get(st[0], T.one_default, T.zero_default);
    rec.h_shift = sym(st, false);
    rec.v_shift = sym(st, false);
    rec.transparency = c.get(st[0], T.one_default, T.zero_default);
    rec.plane_count = 2 + rec.transparency;  // 1 + (chroma_planes || version < 4) + transparency
    rec.h_slices = 1 + sym(st, false);
    rec.v_slices = 1 + sym(st, false);
    if (bad) return fail("malformed configuration record");
    if (rec.bits != 8) return fail("%lld bits per sample: only 8-bit video is decoded", rec.bits);
    if (rec.colorspace == 0 && rec.chroma_planes)
        return fail("YUV with chroma planes is not decoded (VideoCapture's answer passes through swscale's YUV to BGR conversion)");
    if (rec.colorspace == 0 && rec.transparency) return fail("grey with an alpha plane is not decoded");
    if (rec.colorspace == 1 && (rec.h_shift || rec.v_shift)) return fail("RGB with chroma subsampling is invalid");
    if (rec.colorspace != 0 && rec.colorspace != 1) return fail("colorspace %lld is not 0 (YUV / grey) or 1 (RGB)", rec.colorspace);
    if (rec.h_slices < 1 || rec.v_slices < 1 || rec.h_slices > cols || rec.v_slices > rows || rec.h_slices * rec.v_slices > MAX_SLICES)
        return fail("invalid slice grid %lld x %lld", rec.h_slices, rec.v_slices);
    rec.quant_table_count = sym(st, false);
    if (rec.quant_table_count < 1 || rec.quant_table_count > MAX_QUANT_TABLES) return fail("quant_table_count %lld", rec.quant_table_count);
    for (int q = 0; q < rec.quant_table_count; ++q) {
        int64_t count = 1;
        for (int k = 0; k < 5; ++k) {
            int16_t *t = T.quant[q][k];
            uint8_t qs[CONTEXT_SIZE];
            memset(qs, 128, sizeof qs);
            int i = 0, v = 0;
            for (; i < 128; ++v) {
                const uint32_t len = (uint32_t)sym(qs, false) + 1u;
                if (bad || len > (uint32_t)(128 - i) || !len) return fail("malformed quant table %lld", q);
                for (uint32_t j = 0; j < len; ++j) t[i++] = (int16_t)(count * v);
            }
            for (i = 1; i < 128; ++i) t[256 - i] = (int16_t)-t[i];
            t[128] = (int16_t)-t[127];
            count *= 2 * v - 1;
            if (count > 32768) return fail("quant table %lld gives more than 32768 contexts", q);
        }
        rec.context_count[q] = (int)((count + 1) / 2);
    }
    int64_t off = 0;
    uint8_t st2[CONTEXT_SIZE][CONTEXT_SIZE];
    memset(st2, 128, sizeof st2);
    for (int q = 0; q < rec.quant_table_count; ++q) {
        rec.initial_offset[q] = -1;
        if (!c.get(st[0], T.one_default, T.zero_default)) continue;
        rec.initial_offset[q] = off;
        for (int j = 0; j < rec.context_count[q]; ++j)
            for (int k = 0; k < CONTEXT_SIZE; ++k) {
                const int64_t at = off + (int64_t)j * CONTEXT_SIZE + k;
                const int pred = j ? (initial_states ? initial_states[at - CONTEXT_SIZE] : 128) : 128;
                const int v = (pred + sym(st2[k], true)) & 0xFF;
                if (initial_states) initial_states[at] = (uint8_t)v;
            }
        off += (int64_t)rec.context_count[q] * CONTEXT_SIZE;
    }
    if (initial_bytes) *initial_bytes = off;
    rec.ec = sym(st, false);
    if (rec.micro_version > 2) rec.intra = sym(st, false);
    if (bad) return fail("malformed configuration record");
    if (rec.ec < 0 || rec.ec > 1) return fail("error-correction mode %lld is not 0 or 1", rec.ec);
    return 0;
}

// ---- samples --------------------------------------------------------------------------------------------------------
struct alignas(8) VlcState {
    int16_t drift;
    uint16_t error_sum;
    int16_t bias;   // int8 range
    uint16_t count; // uint8 range
};

// MSB-first bit reader over [p, end); bytes past the end read as zero.  `left` counts the bits not yet consumed.
struct BitReader {
    uint64_t cache;
    int nbits;
    const uint8_t *p, *end;
    int64_t left;
    FFV1_HD void init(const uint8_t *b, const uint8_t *e) {
        p = b;
        end = e;
        cache = 0;
        nbits = 0;
        left = (int64_t)(e - b) * 8;
    }
    FFV1_HD void refill() {
        while (nbits <= 56) {
            const uint64_t byte = p < end ? *p++ : 0u;
            cache |= byte << (56 - nbits);
            nbits += 8;
        }
    }
    FFV1_HD uint32_t show32() const { return (uint32_t)(cache >> 32); }
    FFV1_HD void skip(int n) {
        cache <<= n;
        nbits -= n;
        left -= n;
    }
    FFV1_HD uint32_t get(int n) {  // 1 <= n <= 32, after refill
        const uint32_t v = (uint32_t)(cache >> (64 - n));
        skip(n);
        return v;
    }
};

FFV1_HD int clz32(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __clz(x);
#else
    return __builtin_clz(x);
#endif
}
FFV1_HD int log2_run(int i) { return i < 16 ? i >> 2 : i < 24 ? 4 + ((i - 16) >> 1) : i - 16; }  // ff_log2_run[i], i <= 40
FFV1_HD int mid_pred(int a, int b, int c) {
    const int lo = a < b ? a : b, hi = a < b ? b : a;
    return c < lo ? lo : c > hi ? hi : c;
}
FFV1_HD int fold(int v, int bits) { return (int)((uint32_t)v << (32 - bits)) >> (32 - bits); }

// get_vlc_symbol(): Golomb-Rice with limit 12 and an escape of `bits` bits, then the VlcState bias / drift update
FFV1_HD int vlc_symbol(BitReader &g, VlcState &s, int bits) {
    int k = 0;
    for (int i = s.count; i < (int)s.error_sum; i += i) ++k;
    g.refill();
    uint32_t buf = g.show32();
    uint32_t u;
    const int lg = buf ? 31 - clz32(buf) : 0;
    if (lg > 31 - 12) {
        buf >>= lg - k;
        buf += (uint32_t)(30 - lg) << k;
        g.skip(32 + k - lg);
        u = buf;
    } else {
        g.skip(12);
        u = g.get(bits) + 11;
    }
    int v = (int)(u >> 1) ^ -(int)(u & 1);
    v ^= (2 * s.drift + (int)s.count) >> 31;
    const int ret = fold(v + s.bias, bits);
    int drift = s.drift + v, count = s.count;
    uint16_t es = (uint16_t)(s.error_sum + (v < 0 ? -v : v));
    if (count == 128) {
        count >>= 1;
        drift >>= 1;
        es >>= 1;
    }
    ++count;
    int bias = s.bias;
    if (drift <= -count) {
        bias = bias - 1 < -128 ? -128 : bias - 1;
        drift = drift + count > -count + 1 ? drift + count : -count + 1;
    } else if (drift > 0) {
        bias = bias + 1 > 127 ? 127 : bias + 1;
        drift = drift - count < 0 ? drift - count : 0;
    }
    s.drift = (int16_t)drift;
    s.error_sum = es;
    s.bias = (int16_t)bias;
    s.count = (uint16_t)count;
    return ret;
}


// ---- slices and chains ----------------------------------------------------------------------------------------------
// Walks a frame's slice footers back from its end (3-byte big-endian size, then an error byte and a CRC when ec = 1).
// Slice i of the frame is fr[off[i], off[i] + len[i]), footer included; the walk must land exactly on byte 0.
FFV1_HD int locate_slices(const uint8_t *fr, int64_t n, int S, int ec, int64_t *off, int32_t *len) {
    const int trailer = 3 + 5 * ec;
    int64_t end = n;
    for (int i = S - 1; i >= 0; --i) {
        if (end < trailer) return LM_FFV1_FOOTER;
        const uint8_t *t = fr + end - trailer;
        const int64_t v = (((int64_t)t[0] << 16) | ((int64_t)t[1] << 8) | t[2]) + trailer;
        if (v > end) return LM_FFV1_FOOTER;
        end -= v;
        off[i] = end;
        len[i] = (int32_t)v;
    }
    return end == 0 ? LM_FFV1_OK : LM_FFV1_FOOTER;
}

// Per-chain work memory: context states (one block of ctx_stride bytes per context plane) and the sample line ring.
FFV1_HD int64_t ctx_stride(const Record &R) {
    int m = 1;
    for (int q = 0; q < R.quant_table_count; ++q) m = R.context_count[q] > m ? R.context_count[q] : m;
    return (int64_t)m * (R.ac ? CONTEXT_SIZE : (int)sizeof(VlcState));
}
FFV1_HD int line_stride(const Record &R, int cols) { return (cols + R.h_slices - 1) / R.h_slices + 6; }
FFV1_HD int64_t line_bytes(const Record &R, int cols) { return (int64_t)R.coded_planes() * 2 * line_stride(R, cols) * (int64_t)sizeof(int16_t); }

// decode_line(): one line of one plane.  L0 is the line above (with its edge samples set), L1 the line being decoded; in
// the 5-input context model L1 still holds line y - 2 where it has not been overwritten yet.
template <bool RANGE>
FFV1_HD int decode_line(RangeDec &c, BitReader &g, const Tables &T, const int16_t (*q)[256], bool five, uint8_t *rst,
                        VlcState *vst, int w, const int16_t *L0, int16_t *L1, int bits, int &run_index) {
    const int mask = (1 << bits) - 1;
    int run_count = 0, run_mode = 0;
    for (int x = 0; x < w; ++x) {
        if (!(x & 1023) && (RANGE ? c.overread > 2 : g.left < 1)) return LM_FFV1_TRUNCATED;
        const int LT = L0[x - 1], Tp = L0[x], L = L1[x - 1];
        int ctx = q[0][(L - LT) & 0xFF] + q[1][(LT - Tp) & 0xFF] + q[2][(Tp - L0[x + 1]) & 0xFF];
        if (five) ctx += q[3][(L1[x - 2] - L) & 0xFF] + q[4][(L1[x] - Tp) & 0xFF];
        const bool sign = ctx < 0;
        if (sign) ctx = -ctx;
        int diff;
        if (RANGE) {
            bool bad = false;
            diff = c.symbol(rst + (int64_t)ctx * CONTEXT_SIZE, true, T.one_slice, T.zero_slice, bad);
            if (bad) return LM_FFV1_SYMBOL;
        } else {
            if (ctx == 0 && run_mode == 0) run_mode = 1;
            if (run_mode) {
                if (run_count == 0 && run_mode == 1) {
                    g.refill();
                    const int lr = log2_run(run_index);
                    if (g.get(1)) {
                        run_count = 1 << lr;
                        if (x + run_count <= w && run_index < 40) ++run_index;
                    } else {
                        run_count = lr ? (int)g.get(lr) : 0;
                        if (run_index) --run_index;
                        run_mode = 2;
                    }
                }
                if (L1[x - 1] == L0[x - 1]) {
                    while (run_count > 1 && w - x > 1) {
                        L1[x] = L0[x];
                        ++x;
                        --run_count;
                    }
                } else {
                    while (run_count > 1 && w - x > 1) {
                        L1[x] = (int16_t)mid_pred(L1[x - 1], L1[x - 1] + L0[x] - L0[x - 1], L0[x]);
                        ++x;
                        --run_count;
                    }
                }
                if (--run_count < 0) {
                    run_mode = 0;
                    run_count = 0;
                    diff = vlc_symbol(g, vst[ctx], bits);
                    if (diff >= 0) ++diff;
                } else {
                    diff = 0;
                }
            } else {
                diff = vlc_symbol(g, vst[ctx], bits);
            }
        }
        if (sign) diff = -diff;
        const int l = L1[x - 1];
        L1[x] = (int16_t)((mid_pred(l, l + L0[x] - L0[x - 1], L0[x]) + diff) & mask);
    }
    return LM_FFV1_OK;
}

// One slice [sb, se) (footer included) of one frame: slice header, then every plane; channel 0 of the pixels goes to
// `frame` ([rows][cols]).  qpack holds the chain's quant table per context plane (3 bits each), set on the keyframe.
// hs: CONTEXT_SIZE bytes for the header's states (memory, not an array on the stack: the kernel keeps no local memory).
template <bool RANGE>
FFV1_HD int decode_slice(const Record &R, const Tables &T, const uint8_t *initial, const uint8_t *sb, const uint8_t *se, bool key,
                         int s, int rows, int cols, uint8_t *frame, uint8_t *hs, uint8_t *state, int64_t ctx_stride, int16_t *lines,
                         int ls, int &qpack) {
    RangeDec c;
    c.init(sb, se);
    if (s == 0) {
        uint8_t ks = 128;
        if (c.get(ks, T.one_default, T.zero_default) != (int)key) return LM_FFV1_KEYFRAME;
    }
    const uint8_t *one = T.one_slice, *zero = T.zero_slice;
    for (int i = 0; i < CONTEXT_SIZE; ++i) hs[i] = 128;
    bool bad = false;
    const int sx = c.symbol(hs, false, one, zero, bad), sy = c.symbol(hs, false, one, zero, bad);
    const int sw = c.symbol(hs, false, one, zero, bad), sh = c.symbol(hs, false, one, zero, bad);
    if (bad) return LM_FFV1_SYMBOL;
    if (sx != s % R.h_slices || sy != s / R.h_slices || sw != 0 || sh != 0) return LM_FFV1_SLICE_HEADER;
    const int np = R.ctx_planes();
    for (int j = 0; j < R.plane_count; ++j) {
        const int idx = c.symbol(hs, false, one, zero, bad);
        if (bad || idx < 0 || idx >= R.quant_table_count) return LM_FFV1_QUANT_INDEX;
        if (j >= np) continue;
        if (key) qpack = (qpack & ~(7 << (3 * j))) | (idx << (3 * j));
        else if (((qpack >> (3 * j)) & 7) != idx) return LM_FFV1_QUANT_INDEX;
    }
    for (int k = 0; k < 3; ++k) c.symbol(hs, false, one, zero, bad);  // picture structure, sample aspect ratio
    if (bad) return LM_FFV1_SYMBOL;
    const int x0 = (int)((int64_t)cols * sx / R.h_slices), w = (int)((int64_t)cols * (sx + 1) / R.h_slices) - x0;
    const int y0 = (int)((int64_t)rows * sy / R.v_slices), h = (int)((int64_t)rows * (sy + 1) / R.v_slices) - y0;
    if (key) {
        for (int j = 0; j < np; ++j) {
            const int q = (qpack >> (3 * j)) & 7, n = R.context_count[q];
            uint8_t *st = state + j * ctx_stride;
            if (RANGE) {
                const int64_t io = R.initial_offset[q];
                for (int64_t i = 0; i < (int64_t)n * CONTEXT_SIZE; ++i) st[i] = io >= 0 ? initial[io + i] : 128;
            } else {
                VlcState *v = reinterpret_cast<VlcState *>(st);
                for (int i = 0; i < n; ++i) v[i] = VlcState{0, 4, 0, 1};
            }
        }
    }
    BitReader g;
    g.init(se, se);
    if (!RANGE) {
        if (R.micro_version > 1) {
            uint8_t t = 129;
            c.get(t, one, zero);
        }
        if (c.p - 1 > se) return LM_FFV1_TRUNCATED;
        g.init(c.p - 1, se);  // the Golomb-Rice bits start after the range coder's last byte
    }
    const int npc = R.coded_planes();
    for (int i = 0; i < npc * 2 * ls; ++i) lines[i] = 0;
    // plane p's two lines are lines + (2p) * ls + 3 and lines + (2p + 1) * ls + 3; the first is the current line on even y
    int run_index = 0;
    const int bits = R.colorspace == 0 ? 8 : 9;
    for (int y = 0; y < h; ++y) {
        const int cur = y & 1;
        for (int p = 0; p < npc; ++p) {
            int16_t *L1 = lines + (2 * p + cur) * ls + 3, *L0 = lines + (2 * p + (cur ^ 1)) * ls + 3;
            L1[-1] = L0[0];
            L0[w] = L0[w - 1];
            const int cp = (p + 1) >> 1;
            const int16_t(*q)[256] = T.quant[(qpack >> (3 * cp)) & 7];
            const bool five = q[3][127] || q[4][127];
            uint8_t *st = state + cp * ctx_stride;
            const int e = decode_line<RANGE>(c, g, T, q, five, st, reinterpret_cast<VlcState *>(st), w, L0, L1, bits, run_index);
            if (e) return e;
        }
        uint8_t *o = frame + (int64_t)(y0 + y) * cols + x0;
        const int16_t *S0 = lines + cur * ls + 3;
        if (R.colorspace == 0) {
            for (int x = 0; x < w; ++x) o[x] = (uint8_t)S0[x];
        } else {
            const int16_t *S1 = S0 + 2 * ls, *S2 = S0 + 4 * ls;
            for (int x = 0; x < w; ++x) {
                const int b = S1[x] - 256, r = S2[x] - 256;
                o[x] = (uint8_t)(b + S0[x] - ((b + r) >> 2));
            }
        }
    }
    if (RANGE) {
        uint8_t t = 129;
        c.get(t, one, zero);
        if (se - c.p - 2 - 5 * R.ec != 0) return LM_FFV1_SLICE_END;
    } else if (g.left < 0) {
        return LM_FFV1_TRUNCATED;
    }
    return LM_FFV1_OK;
}

// Per-chain work memory: header states, context states (one block of ctx_stride bytes per context plane), sample lines.
FFV1_HD int64_t work_bytes(const Record &R, int cols) { return CONTEXT_SIZE + R.ctx_planes() * ctx_stride(R) + line_bytes(R, cols); }

// One (GOP, slice) chain: slice s of frames f0 .. f0 + nf - 1, f0 a keyframe and the others not.  Slice i = f * S + s is
// payload[soff[i], soff[i] + slen[i]); status[i] is -1 until it is decoded, or an error found before the decode.
// work: work_bytes() bytes, 16-byte aligned.
template <bool RANGE>
FFV1_HD void decode_chain(const Record &R, const Tables &T, const uint8_t *initial, const uint8_t *payload, const int64_t *soff,
                          const int32_t *slen, int32_t *status, uint8_t *out, int rows, int cols, int64_t f0, int nf, int s,
                          uint8_t *work) {
    const int S = R.slices();
    const int64_t cs = ctx_stride(R);
    uint8_t *state = work + CONTEXT_SIZE;
    int16_t *lines = reinterpret_cast<int16_t *>(state + R.ctx_planes() * cs);
    const int ls = line_stride(R, cols);
    int qpack = 0;
    for (int k = 0; k < nf; ++k) {
        const int64_t f = f0 + k, i = f * S + s;
        if (status[i] != -1) return;
        const uint8_t *sb = payload + soff[i];
        const int e = decode_slice<RANGE>(R, T, initial, sb, sb + slen[i], k == 0, s, rows, cols, out + f * rows * (int64_t)cols, work,
                                          state, cs, lines, ls, qpack);
        status[i] = e;
        if (e) return;
    }
}

}  // namespace ffv1
