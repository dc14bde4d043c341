// k_png.cu — PNG frames (the '00dc' chunks of an 'MPNG' / 'png ' AVI) inflated and unfiltered on the device into raw
// [n][rows][cols] frames, channel 0 of what cv::VideoCapture delivers (grey, or blue of RGB / RGBA).
//
// One warp per frame.  Lane 0 runs the serial part of inflate (zlib header, block headers, Huffman decoding, literals and
// stored bytes); the warp copies LZ77 matches and fills the Huffman lookup tables.  The bit stream is read straight from
// the PNG file: the 12 bytes of chunk framing between consecutive IDAT chunks are skipped by the byte reader.  The whole
// filtered stream of a frame is inflated into a scratch slot first, because back-references point into FILTERED bytes
// up to 32 kB back; only then is it unfiltered, as a diagonal wavefront: lane i owns row r0 + i and runs one pixel
// behind lane i - 1, whose last two pixels (the row above at x and x - 1) arrive by shuffle.  Lane 31 writes its
// unfiltered row back into the scratch slot, where lane 0 of the next group of 32 rows reads it.
//
// The input is untrusted: every read is bounded by the frame's payload, every write by its scratch slot and output
// frame, every loop consumes input or produces output, and each error ends the frame with a status code (LM_PNG_*).
#include "lm_internal.h"

namespace {

constexpr int FL = 10, FD = 8;  // bits resolved by one lookup in the literal / length and the distance tables

struct PngSmem {
    uint16_t fast_l[1 << FL];  // (symbol << 4) | code length; 0 = longer code or none: canonical walk
    uint16_t fast_d[1 << FD];
    uint16_t sym_l[288], sym_d[32];  // symbols sorted by code length (canonical order)
    uint16_t cnt_l[16], cnt_d[16], offs[16];
    uint8_t lens[288 + 32];  // code lengths: literal / length, then distance
    uint8_t cl[20];
};

__constant__ uint16_t c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
                                     4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

__device__ __forceinline__ uint32_t be32(const uint8_t *p) {
    return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
}
__device__ __forceinline__ bool is_tag(const uint8_t *p, char a, char b, char c, char d) {
    return p[0] == (uint8_t)a && p[1] == (uint8_t)b && p[2] == (uint8_t)c && p[3] == (uint8_t)d;
}

// Bytes of the IDAT sequence of one PNG file.  p .. ce is the rest of the current chunk body, fe the end of the file.
struct Src {
    const uint8_t *p, *ce, *fe;
    __device__ int next() {
        while (p == ce) {  // p is at the CRC of the finished chunk: step over it and the next chunk's length and type
            if (fe - p < 12 || !is_tag(p + 8, 'I', 'D', 'A', 'T')) {
                fe = ce;  // end of the IDAT sequence: stays exhausted
                return -1;
            }
            const uint32_t len = be32(p + 4);
            p += 12;
            ce = (uint64_t)len > (uint64_t)(fe - p) ? fe : p + len;
        }
        return *p++;
    }
};

// LSB-first bit buffer.  When the input runs out, zero bytes are appended and counted in `pad`; consuming any of them
// (nb < pad) means the stream was truncated.
struct Bits {
    uint64_t bb;
    int nb, pad;
    __device__ void refill(Src &s) {
        while (nb <= 56) {
            int c = s.next();
            if (c < 0) {
                c = 0;
                pad += 8;
            }
            bb |= (uint64_t)c << nb;
            nb += 8;
        }
    }
    __device__ uint32_t get(int n) {  // n <= 32, after refill with room for it
        const uint32_t v = (uint32_t)(bb & ((1ull << n) - 1));
        bb >>= n;
        nb -= n;
        return v;
    }
    __device__ bool over() const { return nb < pad; }
};

// Canonical Huffman decode, one bit at a time (codes longer than the lookup table, the code-length code)
__device__ int decode_slow(Bits &B, const uint16_t *cnt, const uint16_t *sym) {
    int code = 0, first = 0, index = 0;
    uint64_t b = B.bb;
    for (int len = 1; len <= 15; ++len) {
        code |= (int)(b & 1);
        b >>= 1;
        const int c = cnt[len];
        if (code - c < first) {
            B.bb >>= len;
            B.nb -= len;
            return sym[index + (code - first)];
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return -1;
}
__device__ __forceinline__ int decode(Bits &B, const uint16_t *fast, int fb, const uint16_t *cnt, const uint16_t *sym) {
    const uint16_t e = fast[B.bb & ((1u << fb) - 1)];
    if (e) {
        const int l = e & 15;
        B.bb >>= l;
        B.nb -= l;
        return e >> 4;
    }
    return decode_slow(B, cnt, sym);
}

// Counts and canonical symbol order of one code; zlib's acceptance rule (inflate_table): no over-subscribed set, and no
// incomplete set except a single code of length 1 (not for the code-length code); an empty set is accepted.
__device__ bool build_counts(const uint8_t *len, int n, uint16_t *cnt, uint16_t *sym, bool is_cl, uint16_t *offs) {
    for (int l = 0; l < 16; ++l) cnt[l] = 0;
    for (int s = 0; s < n; ++s) ++cnt[len[s]];
    int max = 15;
    while (max > 0 && cnt[max] == 0) --max;
    if (max == 0) return !is_cl;
    int left = 1;
    for (int l = 1; l < 16; ++l) {
        left = (left << 1) - cnt[l];
        if (left < 0) return false;
    }
    if (left > 0 && (is_cl || max != 1)) return false;
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + cnt[l];
    for (int s = 0; s < n; ++s)
        if (len[s]) sym[offs[len[s]]++] = (uint16_t)s;
    return true;
}

// The warp fills the lookup table of one code from its counts and canonical order.
__device__ void fill_fast(const uint8_t *len, const uint16_t *cnt, const uint16_t *sym, uint16_t *fast, int fb, int lane) {
    int total = 0;
    for (int l = 1; l < 16; ++l) total += cnt[l];
    for (int k = lane; k < total; k += 32) {
        const int s = sym[k], L = len[s];
        if (L > fb) continue;
        int nc = 0, idx = 0;
        for (int l = 1; l < L; ++l) {
            nc = (nc + cnt[l]) << 1;
            idx += cnt[l];
        }
        const uint32_t rev = __brev((uint32_t)(nc + k - idx)) >> (32 - L);
        for (uint32_t e = rev; e < (1u << fb); e += 1u << L) fast[e] = (uint16_t)((s << 4) | L);
    }
}

enum { OP_NONE = 0, OP_COPY = 1, OP_BUILD = 2, OP_END = 3 };
enum { M_HEADER = 0, M_DATA = 1 };

__global__ void __launch_bounds__(128) k_png_decode(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs, int64_t base, int n,
                                                    int rows, int cols, uint8_t *__restrict__ scratch, int64_t slot, uint8_t *__restrict__ out,
                                                    int32_t *__restrict__ status) {
    __shared__ PngSmem smem[4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t f = (int64_t)blockIdx.x * 4 + warp;
    if (f >= n) return;
    PngSmem &S = smem[warp];
    const uint8_t *fp = payload + (offs[f] - base);
    const int64_t flen = offs[f + 1] - offs[f];
    uint8_t *dst = scratch + f * slot;

    // ---- signature, IHDR, first IDAT (checked on the host too; repeated here so that no input can mislead the kernel)
    int err = 0, bpp = 1;
    int64_t total = 0;
    Src src{};
    if (lane == 0) {
        if (flen < 45 || be32(fp) != 0x89504e47u || be32(fp + 4) != 0x0d0a1a0au || be32(fp + 8) != 13 || !is_tag(fp + 12, 'I', 'H', 'D', 'R') ||
            be32(fp + 16) != (uint32_t)cols || be32(fp + 20) != (uint32_t)rows || fp[24] != 8 || fp[26] || fp[27] || fp[28] ||
            (fp[25] != 0 && fp[25] != 2 && fp[25] != 6)) {
            err = LM_PNG_HEADER;
        } else {
            bpp = fp[25] == 0 ? 1 : fp[25] == 2 ? 3 : 4;
            total = (int64_t)rows * (1 + (int64_t)cols * bpp);
            if (total > slot) err = LM_PNG_HEADER;
            const uint8_t *fe = fp + flen, *p = fp + 33;
            for (;;) {  // chunks before the first IDAT (PLTE, tEXt, ...) are skipped
                if (fe - p < 12 || is_tag(p + 4, 'I', 'E', 'N', 'D')) {
                    if (!err) err = LM_PNG_NO_IDAT;
                    break;
                }
                const uint64_t len = be32(p);
                if (is_tag(p + 4, 'I', 'D', 'A', 'T')) {
                    src.p = p + 8;
                    src.ce = len > (uint64_t)(fe - src.p) ? fe : src.p + len;
                    src.fe = fe;
                    break;
                }
                if (len + 12 > (uint64_t)(fe - p)) {
                    if (!err) err = LM_PNG_TRUNCATED;
                    break;
                }
                p += 12 + len;
            }
        }
    }

    // ---- inflate: lane 0 decodes until it needs the warp (a match to copy, tables to fill) or the stream ends
    Bits B{0, 0, 0};
    int mode = M_HEADER, last = 0;
    int32_t pos = 0;
    if (lane == 0 && !err) {
        B.refill(src);
        const uint32_t cmf = B.get(8), flg = B.get(8);
        if ((cmf & 15) != 8 || (cmf >> 4) > 7 || ((cmf << 8) | flg) % 31 != 0 || (flg & 0x20)) err = LM_PNG_ZLIB;  // FDICT: no preset dictionary in PNG
        if (B.over()) err = LM_PNG_TRUNCATED;
    }
    for (;;) {
        int op = OP_NONE, c_len = 0, c_dist = 0, c_pos = 0;
        if (lane == 0) {
            while (op == OP_NONE) {
                if (err) {
                    op = OP_END;
                    break;
                }
                B.refill(src);
                if (mode == M_HEADER) {
                    if (last) {
                        op = OP_END;
                        break;
                    }
                    last = (int)B.get(1);
                    const int type = (int)B.get(2);
                    if (type == 0) {  // stored: byte aligned LEN, NLEN, then LEN raw bytes
                        B.get(B.nb & 7);
                        B.refill(src);
                        const uint32_t ln = B.get(16), nln = B.get(16);
                        if (B.over()) err = LM_PNG_TRUNCATED;
                        else if (ln != (~nln & 0xffffu)) err = LM_PNG_STORED;
                        else if (pos + (int64_t)ln > total) err = LM_PNG_TOO_LONG;
                        for (uint32_t i = 0; i < ln && !err; ++i) {
                            B.refill(src);
                            dst[pos++] = (uint8_t)B.get(8);
                            if (B.over()) err = LM_PNG_TRUNCATED;
                        }
                    } else if (type == 1) {  // fixed Huffman codes (RFC 1951 3.2.6); distances 30, 31 and lengths 286, 287 are invalid
                        for (int i = 0; i < 288; ++i) S.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
                        for (int i = 0; i < 32; ++i) S.lens[288 + i] = 5;
                        build_counts(S.lens, 288, S.cnt_l, S.sym_l, false, S.offs);
                        build_counts(S.lens + 288, 32, S.cnt_d, S.sym_d, false, S.offs);
                        mode = M_DATA;
                        op = OP_BUILD;
                    } else if (type == 2) {  // dynamic: code-length code, then the literal / length and distance code lengths
                        const int nlen = (int)B.get(5) + 257, ndist = (int)B.get(5) + 1, ncode = (int)B.get(4) + 4;
                        if (nlen > 286 || ndist > 30) {
                            err = LM_PNG_CODES;
                            continue;
                        }
                        for (int i = 0; i < 19; ++i) S.cl[c_clorder[i]] = 0;
                        for (int i = 0; i < ncode; ++i) {
                            B.refill(src);
                            S.cl[c_clorder[i]] = (uint8_t)B.get(3);
                        }
                        if (!build_counts(S.cl, 19, S.cnt_l, S.sym_l, true, S.offs)) {
                            err = LM_PNG_CODES;
                            continue;
                        }
                        for (int i = 0; i < nlen + ndist && !err;) {
                            B.refill(src);
                            const int sym = decode_slow(B, S.cnt_l, S.sym_l);
                            int rep = 0, val = 0;
                            if (sym < 0) err = LM_PNG_CODES;
                            else if (sym < 16) val = sym, rep = 1;
                            else if (sym == 16) {
                                if (i == 0) err = LM_PNG_CODES;
                                else val = S.lens[i - 1 < nlen ? i - 1 : 288 + i - 1 - nlen], rep = 3 + (int)B.get(2);
                            } else if (sym == 17) rep = 3 + (int)B.get(3);
                            else rep = 11 + (int)B.get(7);
                            if (B.over()) err = LM_PNG_TRUNCATED;
                            if (!err && i + rep > nlen + ndist) err = LM_PNG_CODES;
                            for (; rep > 0 && !err; --rep, ++i) S.lens[i < nlen ? i : 288 + i - nlen] = (uint8_t)val;
                        }
                        if (err) continue;
                        for (int i = nlen; i < 288; ++i) S.lens[i] = 0;
                        for (int i = ndist; i < 32; ++i) S.lens[288 + i] = 0;
                        if (S.lens[256] == 0 || !build_counts(S.lens, 288, S.cnt_l, S.sym_l, false, S.offs) ||
                            !build_counts(S.lens + 288, 32, S.cnt_d, S.sym_d, false, S.offs)) {
                            err = LM_PNG_CODES;  // no end-of-block code, or an over-subscribed / incomplete set
                            continue;
                        }
                        mode = M_DATA;
                        op = OP_BUILD;
                    } else {
                        err = LM_PNG_BLOCK_TYPE;
                    }
                    continue;
                }
                // M_DATA: literals until a match or the end of the block
                const int sym = decode(B, S.fast_l, FL, S.cnt_l, S.sym_l);
                if (sym < 0) {
                    err = LM_PNG_SYMBOL;
                } else if (sym < 256) {
                    if (pos >= total) err = LM_PNG_TOO_LONG;
                    else dst[pos++] = (uint8_t)sym;
                } else if (sym == 256) {
                    mode = M_HEADER;
                } else if (sym - 257 >= 29) {
                    err = LM_PNG_SYMBOL;
                } else {
                    const int l = sym - 257;
                    const int len = c_lbase[l] + (int)B.get(c_lext[l]);
                    const int d = decode(B, S.fast_d, FD, S.cnt_d, S.sym_d);
                    if (d < 0 || d >= 30) {
                        err = LM_PNG_SYMBOL;
                    } else {
                        const int dist = c_dbase[d] + (int)B.get(c_dext[d]);
                        if (!B.over() && dist > pos) err = LM_PNG_DISTANCE;
                        else if (pos + (int64_t)len > total) err = LM_PNG_TOO_LONG;
                        else op = OP_COPY, c_len = len, c_dist = dist, c_pos = pos, pos += len;
                    }
                }
                if (B.over()) err = LM_PNG_TRUNCATED, op = OP_NONE;
            }
        }
        op = __shfl_sync(0xffffffffu, op, 0);
        __syncwarp();
        if (op == OP_COPY) {
            c_len = __shfl_sync(0xffffffffu, c_len, 0);
            c_dist = __shfl_sync(0xffffffffu, c_dist, 0);
            c_pos = __shfl_sync(0xffffffffu, c_pos, 0);
            uint8_t *o = dst + c_pos;
            for (int j = lane; j < c_len; j += 32) o[j] = o[(c_dist >= c_len ? j : j % c_dist) - c_dist];
        } else if (op == OP_BUILD) {
            for (int i = lane; i < (1 << FL); i += 32) S.fast_l[i] = 0;
            for (int i = lane; i < (1 << FD); i += 32) S.fast_d[i] = 0;
            __syncwarp();
            fill_fast(S.lens, S.cnt_l, S.sym_l, S.fast_l, FL, lane);
            fill_fast(S.lens + 288, S.cnt_d, S.sym_d, S.fast_d, FD, lane);
        } else {
            break;
        }
        __syncwarp();
    }
    if (lane == 0 && !err && pos != total) err = LM_PNG_TOO_SHORT;
    err = __shfl_sync(0xffffffffu, err, 0);
    bpp = __shfl_sync(0xffffffffu, bpp, 0);
    if (err) {
        if (lane == 0) status[f] = err;
        return;
    }

    // ---- unfilter: every filter type is checked first, then rows in groups of 32, one lane per row
    const int64_t stride = 1 + (int64_t)cols * bpp;
    bool bad = false;
    for (int r = lane; r < rows; r += 32) bad |= dst[r * stride] > 4;
    if (__any_sync(0xffffffffu, bad)) {
        if (lane == 0) status[f] = LM_PNG_FILTER;
        return;
    }
    const int ch = bpp == 1 ? 0 : 2;  // channel 0 of the BGR frame = blue = third byte of RGB / RGBA
    uint8_t *of = out + f * (int64_t)rows * cols;
    for (int r0 = 0; r0 < rows; r0 += 32) {
        const int r = r0 + lane;
        const bool valid = r < rows;
        uint8_t *row = dst + (valid ? r : 0) * stride;
        const int ft = valid ? row[0] : 0;
        ++row;
        const uint8_t *above = r0 > 0 ? dst + (int64_t)(r0 - 1) * stride + 1 : nullptr;  // lane 0: the previous group's last row
        const bool keep = lane == 31 && r0 + 32 < rows;
        uint32_t a = 0, a2 = 0, cprev = 0;
        for (int t = 0; t < cols + 31; ++t) {
            const int x = t - lane;
            uint32_t b = __shfl_up_sync(0xffffffffu, a, 1), c = __shfl_up_sync(0xffffffffu, a2, 1);
            if (lane == 0) {
                b = 0;
                if (above && x < cols)
                    for (int k = 0; k < bpp; ++k) b |= (uint32_t)above[x * bpp + k] << (8 * k);
                c = cprev;
                cprev = b;
            }
            if (!valid || x < 0 || x >= cols) continue;
            uint32_t px = 0;
            for (int k = 0; k < bpp; ++k) {
                const int ak = (a >> (8 * k)) & 255, bk = (b >> (8 * k)) & 255, ck = (c >> (8 * k)) & 255;
                int pred;
                switch (ft) {
                    case 0: pred = 0; break;
                    case 1: pred = ak; break;
                    case 2: pred = bk; break;
                    case 3: pred = (ak + bk) >> 1; break;
                    default: {
                        const int pa = abs(bk - ck), pb = abs(ak - ck), pc = abs(ak + bk - 2 * ck);
                        pred = (pa <= pb && pa <= pc) ? ak : (pb <= pc ? bk : ck);
                    }
                }
                const uint32_t v = (uint32_t)(row[x * bpp + k] + pred) & 255u;
                if (keep) row[x * bpp + k] = (uint8_t)v;
                px |= v << (8 * k);
            }
            a2 = a;
            a = px;
            of[(int64_t)r * cols + x] = (uint8_t)(px >> (8 * ch));
        }
        __syncwarp();
    }
    if (lane == 0) status[f] = LM_PNG_OK;
}

// The first 45 bytes of every frame (signature, IHDR, the next chunk header) for the host's checks, zero-padded
__global__ void k_png_headers(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs, int64_t base, int64_t n,
                              uint8_t *__restrict__ hdr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * LM_PNG_HDR_BYTES) return;
    const int64_t f = i / LM_PNG_HDR_BYTES, k = i % LM_PNG_HDR_BYTES;
    hdr[i] = k < offs[f + 1] - offs[f] ? payload[offs[f] - base + k] : 0;
}

}  // namespace

int lm_launch_png_decode(const uint8_t *payload, const int64_t *offs, int64_t base, int n, int rows, int cols, uint8_t *scratch, int64_t slot,
                         uint8_t *out, int32_t *status, cudaStream_t s) {
    if (n <= 0) return 0;
    k_png_decode<<<(n + 3) / 4, 128, 0, s>>>(payload, offs, base, n, rows, cols, scratch, slot, out, status);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int lm_launch_png_headers(const uint8_t *payload, const int64_t *offs, int64_t base, int64_t n, uint8_t *hdr, cudaStream_t s) {
    if (n <= 0) return 0;
    const int64_t total = n * LM_PNG_HDR_BYTES;
    k_png_headers<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(payload, offs, base, n, hdr);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

const char *lm_png_status_text(int st) {
    switch (st) {
        case LM_PNG_OK: return "ok";
        case LM_PNG_HEADER: return "bad PNG signature or IHDR";
        case LM_PNG_TRUNCATED: return "the compressed data ends early (truncated frame or missing end-of-block)";
        case LM_PNG_ZLIB: return "bad zlib header (or a preset dictionary)";
        case LM_PNG_BLOCK_TYPE: return "invalid deflate block type 3";
        case LM_PNG_CODES: return "invalid Huffman code lengths (over-subscribed, incomplete or no end-of-block code)";
        case LM_PNG_SYMBOL: return "invalid Huffman code or length / distance symbol";
        case LM_PNG_DISTANCE: return "a back-reference reaches before the start of the stream";
        case LM_PNG_TOO_LONG: return "the image data is longer than rows x (1 + cols x bytes per pixel)";
        case LM_PNG_TOO_SHORT: return "the image data is shorter than rows x (1 + cols x bytes per pixel)";
        case LM_PNG_STORED: return "stored block length does not match its complement";
        case LM_PNG_FILTER: return "unknown row filter type";
        case LM_PNG_NO_IDAT: return "no IDAT chunk";
        default: return "not decoded";
    }
}
