// k_mpeg4.cu — MPEG-4 Part 2 video (cv2.VideoWriter 'mp4v' / 'XVID', libavcodec's mpeg4 encoder) decoded on the device into
// raw [n][rows][cols] frames, channel 0 of what cv::VideoCapture delivers (mpeg4_format.h).
//
// All prediction inside a frame (DC, AC, motion vectors) happens on coefficients and vectors, so the entropy decode of one
// frame does not need any other frame; only pixel reconstruction runs from frame to frame, and inside a frame it is parallel
// over macroblocks.  So, per piece of frames:
//   k_mpeg4_locate   one thread per frame: walks the frame's start codes (frames are untrusted) into its VOP header, checking
//                    any VOL it carries against the call's (only for payloads already on the device; the host parses the
//                    headers of a host payload itself);
//   k_mpeg4_entropy  one thread per frame (8 frames per CTA): builds the VLC lookahead tables in shared memory, then decodes
//                    every macroblock of its frame into motion vectors and dequantised Y / Cb coefficients after DC / AC
//                    prediction, in the piece's scratch;
//   k_mpeg4_recon    launched once per position in a segment (a run of frames from an I-VOP, or from the piece's first frame,
//                    to the frame before the next I-VOP): one thread per macroblock of every segment's frame at that
//                    position builds the macroblock from the segment's previous frame (half-pel prediction, IDCT, add) into
//                    the segment's reference planes and writes its displayed pixels through the colour rule.
// A segment that starts with a P-VOP continues the previous piece's last frame, whose planes are carried over.
#include "mpeg4_format.h"
#include "lm_internal.h"

namespace {

__global__ void __launch_bounds__(128) k_mpeg4_locate(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs, int n, int rows,
                                                      int cols, const mpeg4::Vol *__restrict__ vol0, mpeg4::Vop *__restrict__ vop,
                                                      int32_t *__restrict__ status) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    mpeg4::Vol vol = *vol0;
    mpeg4::Vop v{};
    int st = mpeg4::parse(payload + offs[f], offs[f + 1] - offs[f], rows, cols, true, vol, v);
    if (st == mpeg4::LM_MPEG4_OK && v.type == mpeg4::VOP_N) st = mpeg4::LM_MPEG4_NOT_CODED;
    if (st == mpeg4::LM_MPEG4_OK && f == 0 && v.type != mpeg4::VOP_I) st = mpeg4::LM_MPEG4_FIRST_NOT_I;
    vop[f] = v;
    status[f] = st;
}

// The VOL of the call when the extradata has none: frame 0's (one thread)
__global__ void k_mpeg4_vol(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs, int rows, int cols, mpeg4::Vol *__restrict__ vol,
                            int32_t *__restrict__ status) {
    mpeg4::Vop v{};
    const int st = mpeg4::parse(payload + offs[0], offs[1] - offs[0], rows, cols, true, *vol, v);
    if (st != mpeg4::LM_MPEG4_OK) status[0] = st;
}

__global__ void __launch_bounds__(LM_MPEG4_FRAMES_PER_CTA) k_mpeg4_entropy(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs,
                                                                          int64_t base, int n, const mpeg4::Vop *__restrict__ vop, int mbw, int mbh,
                                                                          mpeg4::MbInfo *__restrict__ info, int16_t *__restrict__ coef,
                                                                          uint8_t *__restrict__ lines, int64_t lines_bytes, int32_t *__restrict__ status) {
    extern __shared__ __align__(16) uint8_t smem[];
    mpeg4::Tables &T = *reinterpret_cast<mpeg4::Tables *>(smem);
    mpeg4::build_tables(T, 0, threadIdx.x, blockDim.x);
    __syncthreads();
    mpeg4::build_tables(T, 1, threadIdx.x, blockDim.x);
    __syncthreads();
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n || status[f] != mpeg4::LM_MPEG4_OK) return;
    const int nmb = mbw * mbh;
    mpeg4::MbInfo *fi = info + (int64_t)f * nmb;
    const mpeg4::Vop v = vop[f];
    int16_t *fc = coef + (int64_t)f * nmb * mpeg4::BLOCKS_PER_MB * 64;
    status[f] = mpeg4::decode_vop(
        T, v, mbw, mbh, payload + (offs[f] - base), offs[f + 1] - offs[f], mpeg4::lines_at(lines + (int64_t)f * lines_bytes, mbw),
        [&](int m, const mpeg4::MbInfo &mi) { fi[m] = mi; },
        [&](int m, int b, const int16_t *blk) {
            const uint4 *s = reinterpret_cast<const uint4 *>(blk);
            uint4 *d = reinterpret_cast<uint4 *>(fc + ((int64_t)m * mpeg4::BLOCKS_PER_MB + b) * 64);
#pragma unroll
            for (int k = 0; k < 8; ++k) d[k] = s[k];
        });
}

// Position j of every segment: frame seg[2 s] + j of the piece when j < seg[2 s + 1].  Planes of segment s: 2 s + (j & 1)
// (the frame built) and 2 s + ((j - 1) & 1) (its predecessor); at j = 0 the predecessor is the carried plane.
__global__ void __launch_bounds__(128) k_mpeg4_recon(const int32_t *__restrict__ seg, int j, const mpeg4::Vop *__restrict__ vop,
                                                     const mpeg4::MbInfo *__restrict__ info, const int16_t *__restrict__ coef, int mbw, int mbh,
                                                     uint8_t *__restrict__ planes, const uint8_t *__restrict__ carry, int64_t plane_bytes,
                                                     const int32_t *__restrict__ status, uint8_t *__restrict__ out, int rows, int cols) {
    const int s = blockIdx.y, m = blockIdx.x * blockDim.x + threadIdx.x, nmb = mbw * mbh;
    if (m >= nmb || j >= seg[2 * s + 1]) return;
    const int f = seg[2 * s] + j;
    if (status[f] != mpeg4::LM_MPEG4_OK) return;
    const uint8_t *ref = j == 0 ? carry : planes + (2 * s + ((j - 1) & 1)) * plane_bytes;
    uint8_t *cur = planes + (2 * s + (j & 1)) * plane_bytes;
    const int64_t ybytes = (int64_t)nmb * 256;
    const int my = m / mbw, mx = m - my * mbw;
    mpeg4::build_mb(mbw, mbh, mx, my, info[(int64_t)f * nmb + m], coef + ((int64_t)f * nmb + m) * mpeg4::BLOCKS_PER_MB * 64, vop[f].rounding, ref,
                    ref + ybytes, cur, cur + ybytes);
    mpeg4::put_mb(mbw, mx, my, cur, cur + ybytes, rows, cols, out + (int64_t)f * rows * cols);
}

}  // namespace

size_t lm_mpeg4_vol_bytes() { return sizeof(mpeg4::Vol); }
size_t lm_mpeg4_vop_bytes() { return sizeof(mpeg4::Vop); }
size_t lm_mpeg4_info_bytes() { return sizeof(mpeg4::MbInfo); }

int lm_launch_mpeg4_locate(const uint8_t *payload, const int64_t *offs, int n, int rows, int cols, uint8_t *vol, int need_vol, uint8_t *vop,
                           int32_t *status, cudaStream_t s) {
    if (n <= 0) return 0;
    auto *V = reinterpret_cast<mpeg4::Vol *>(vol);
    if (need_vol) k_mpeg4_vol<<<1, 1, 0, s>>>(payload, offs, rows, cols, V, status);
    k_mpeg4_locate<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(payload, offs, n, rows, cols, V, reinterpret_cast<mpeg4::Vop *>(vop), status);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int lm_launch_mpeg4_decode(const uint8_t *payload, const int64_t *offs, int64_t base, int n, const uint8_t *vop, int rows, int cols, uint8_t *info,
                           int16_t *coef, uint8_t *lines, const int32_t *seg, int nseg, int seg_len, uint8_t *planes, const uint8_t *carry,
                           int32_t *status, uint8_t *out, cudaStream_t s) {
    if (n <= 0) return 0;
    const int mbw = (cols + 15) / 16, mbh = (rows + 15) / 16, nmb = mbw * mbh;
    const auto *V = reinterpret_cast<const mpeg4::Vop *>(vop);
    auto *I = reinterpret_cast<mpeg4::MbInfo *>(info);
    const int64_t lb = (mpeg4::lines_bytes(mbw) + 15) & ~(int64_t)15;
    const size_t smem = sizeof(mpeg4::Tables);
    static LmDevOnce once;
    if (auto setup = once.first())
        if (lm_allow_max_dynamic_smem(k_mpeg4_entropy) != cudaSuccess) return -1;
    k_mpeg4_entropy<<<(unsigned)((n + LM_MPEG4_FRAMES_PER_CTA - 1) / LM_MPEG4_FRAMES_PER_CTA), LM_MPEG4_FRAMES_PER_CTA, smem, s>>>(
        payload, offs, base, n, V, mbw, mbh, I, coef, lines, lb, status);
    const int64_t plane = lm_mpeg4_plane_bytes(rows, cols);
    for (int j = 0; j < seg_len; ++j)
        k_mpeg4_recon<<<dim3((unsigned)((nmb + 127) / 128), (unsigned)nseg), 128, 0, s>>>(seg, j, V, I, coef, mbw, mbh, planes, carry, plane,
                                                                                         status, out, rows, cols);
    return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int64_t lm_mpeg4_lines_bytes(int cols) { return (mpeg4::lines_bytes((cols + 15) / 16) + 15) & ~(int64_t)15; }
