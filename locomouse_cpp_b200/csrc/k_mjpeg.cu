// k_mjpeg.cu — Motion-JPEG frames (baseline JPEG, the chunks of an 'MJPG' AVI or the samples of a Matroska / QuickTime
// track) decoded on the device into raw [n][rows][cols] frames, channel 0 of what cv::VideoCapture delivers (mjpeg_format.h).
//
// Three kernels per piece of frames, because the serial part and the parallel part want different shapes:
//   k_mjpeg_locate   one thread per frame: walks the frame's marker segments (frames are untrusted) into a Header (tables,
//                    geometry, start of the entropy-coded data) and a status;
//   k_mjpeg_entropy  one thread per frame (8 frames per CTA, so that a piece of frames spreads over every SM): builds the 9-bit lookahead of each Huffman table in its own slice of shared
//                    memory, then Huffman-decodes every block of the frame with a word-based bit reader into dequantised
//                    int16 coefficients (Y and Cb) in the piece's scratch;
//   k_mjpeg_idct     one thread per Y block: libavcodec's simple IDCT of the block (and of the Cb block that covers it),
//                    the colour rule and the crop to the frame.
// A restart interval is decoded inside its frame's thread (the predictor reset and the RSTn check are in decode_scan).
#include "mjpeg_format.h"
#include "lm_internal.h"

namespace {

constexpr int LOOKAHEAD = 4 << mjpeg::FAST_BITS;  // entries of one frame's four lookahead tables

__global__ void __launch_bounds__(128) k_mjpeg_locate(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs, int64_t base,
                                                      int n, int rows, int cols, mjpeg::Header *__restrict__ hdr,
                                                      int32_t *__restrict__ status, int32_t *__restrict__ dht0, int first_piece) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    status[f] = mjpeg::parse(payload + (offs[f] - base), offs[f + 1] - offs[f], rows, cols, hdr[f]);
    if (first_piece && f == 0) *dht0 = hdr[0].dht_mask;  // the call's frame 0: the Huffman tables every frame must define
}

__global__ void __launch_bounds__(LM_MJPEG_FRAMES_PER_CTA) k_mjpeg_entropy(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs,
                                                                          int64_t base, int n, const mjpeg::Header *__restrict__ hdr,
                                                                          int16_t *__restrict__ coef, int64_t slot_blocks,
                                                                          int32_t *__restrict__ status, const int32_t *__restrict__ dht0) {
    extern __shared__ uint16_t fast_all[];
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n || status[f] != mjpeg::LM_MJPEG_OK) return;
    const mjpeg::Header &h = hdr[f];
    if (h.dht_mask != *dht0) {  // libavcodec would carry the tables over from frame to frame
        status[f] = mjpeg::LM_MJPEG_DHT_CHANGE;
        return;
    }
    if (h.blocks() > slot_blocks) {  // parse() allows only layouts max_blocks() bounds; the slot is never overrun
        status[f] = mjpeg::LM_MJPEG_SAMPLING;
        return;
    }
    uint16_t *fast = fast_all + threadIdx.x * LOOKAHEAD;
    for (int t = 0; t < 4; ++t)
        if (!mjpeg::build_fast(h.tab[t], fast + t * (1 << mjpeg::FAST_BITS))) {
            status[f] = mjpeg::LM_MJPEG_TABLE;
            return;
        }
    const uint8_t *fr = payload + (offs[f] - base);
    int16_t *out = coef + (int64_t)f * slot_blocks * 64;
    const int st = mjpeg::decode_scan(h, fr + h.ecs, fr + (offs[f + 1] - offs[f]), fast, [&](int64_t b, const int16_t *blk) {
        const uint4 *s = reinterpret_cast<const uint4 *>(blk);
        uint4 *d = reinterpret_cast<uint4 *>(out + b * 64);
#pragma unroll
        for (int k = 0; k < 8; ++k) d[k] = s[k];
    });
    status[f] = st;
}

__global__ void __launch_bounds__(256, 2) k_mjpeg_idct(const mjpeg::Header *__restrict__ hdr, const int16_t *__restrict__ coef, int64_t slot_blocks,
                                                    int slot_yblocks, int n, const int32_t *__restrict__ status, uint8_t *__restrict__ out,
                                                    int rows, int cols) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)n * slot_yblocks) return;
    const int f = (int)(i / slot_yblocks), b = (int)(i - (int64_t)f * slot_yblocks);
    if (status[f] != mjpeg::LM_MJPEG_OK) return;
    const mjpeg::Header &h = hdr[f];
    const int bx_n = h.y_blocks_x();
    if (b >= bx_n * h.y_blocks_y()) return;
    const int by = b / bx_n, bx = b - by * bx_n;
    mjpeg::put_y_block(h, coef + (int64_t)f * slot_blocks * 64, by, bx, out + (int64_t)f * rows * cols);
}

}  // namespace

size_t lm_mjpeg_header_bytes() { return sizeof(mjpeg::Header); }

int lm_launch_mjpeg_decode(const uint8_t *payload, const int64_t *offs, int64_t base, int n, int rows, int cols, uint8_t *hdr, int16_t *coef,
                           int32_t *status, int32_t *dht0, int first_piece, uint8_t *out, cudaStream_t s) {
    if (n <= 0) return 0;
    auto *H = reinterpret_cast<mjpeg::Header *>(hdr);
    const int64_t slot_blocks = mjpeg::max_blocks(rows, cols);
    const int slot_yblocks = (int)(((cols + 15) / 16) * 2 * (int64_t)((rows + 15) / 16) * 2);
    const size_t smem = (size_t)LM_MJPEG_FRAMES_PER_CTA * LOOKAHEAD * sizeof(uint16_t);
    static LmDevOnce once;
    if (auto setup = once.first())
        if (lm_allow_max_dynamic_smem(k_mjpeg_entropy) != cudaSuccess) return -1;
    k_mjpeg_locate<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(payload, offs, base, n, rows, cols, H, status, dht0, first_piece);
    k_mjpeg_entropy<<<(unsigned)((n + LM_MJPEG_FRAMES_PER_CTA - 1) / LM_MJPEG_FRAMES_PER_CTA), LM_MJPEG_FRAMES_PER_CTA, smem, s>>>(
        payload, offs, base, n, H, coef, slot_blocks, status, dht0);
    const int64_t threads = (int64_t)n * slot_yblocks;
    k_mjpeg_idct<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(H, coef, slot_blocks, slot_yblocks, n, status, out, rows, cols);
    if (cudaGetLastError() != cudaSuccess) return -1;
    return 1;
}
