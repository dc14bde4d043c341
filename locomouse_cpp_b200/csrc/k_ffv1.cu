// k_ffv1.cu — FFV1 version 3 frames (the '00dc' chunks of an 'FFV1' AVI) decoded on the device into raw [n][rows][cols]
// frames, channel 0 of what cv::VideoCapture delivers (grey, or blue of RGB / RGBA).
//
// The serial unit of FFV1 is a (GOP, slice) chain: within a GOP, slice s of each frame continues the context state that
// slice s of the previous frame ended with, and every decision depends on the one before.  So one THREAD runs one chain
// (ffv1_format.h decode_chain): a 10 000-frame video at GOP 12 with 8 slices has about 6 700 chains, each up to about a
// million dependent pixel steps, which is about one thread per chain across the whole GPU.  Two small kernels run first:
// k_ffv1_locate walks each frame's slice footers (one thread per frame), and k_ffv1_crc checks every slice's CRC (one
// thread per slice), so that a corrupt slice is reported before anything is decoded from it.
//
// Each chain's work memory (header states, context states, two sample lines per plane) sits in shared memory when the
// launch still fits in one wave that way, otherwise in a per-chain global slot (guarded in guard mode).  The record's
// quant tables and state transitions sit in shared memory.  The input is untrusted: see ffv1_format.h.
#include "ffv1_format.h"
#include "lm_internal.h"

namespace {

__global__ void __launch_bounds__(256) k_ffv1_locate(const uint8_t *__restrict__ payload, const int64_t *__restrict__ offs, int64_t base,
                                                     int64_t n, int S, int ec, int64_t *__restrict__ soff, int32_t *__restrict__ slen,
                                                     int32_t *__restrict__ status) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    const int64_t b = offs[f] - base;
    const int e = ffv1::locate_slices(payload + b, offs[f + 1] - offs[f], S, ec, soff + f * S, slen + f * S);
    for (int s = 0; s < S; ++s) {
        if (e) status[f * S + s] = ffv1::LM_FFV1_FOOTER;
        else soff[f * S + s] += b;
    }
}

__global__ void __launch_bounds__(256) k_ffv1_crc(const uint8_t *__restrict__ payload, const int64_t *__restrict__ soff,
                                                  const int32_t *__restrict__ slen, int64_t ns, int32_t *__restrict__ status) {
    __shared__ uint32_t t[256];
    {
        uint32_t c = threadIdx.x << 24;
        for (int k = 0; k < 8; ++k) c = (c << 1) ^ (c & 0x80000000u ? 0x04C11DB7u : 0u);
        t[threadIdx.x] = c;
    }
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns || status[i] != -1) return;
    const uint8_t *p = payload + soff[i];
    const int32_t n = slen[i];
    uint32_t crc = 0;
    int32_t k = 0;
    for (; k < n && ((uintptr_t)(p + k) & 3); ++k) crc = ffv1::crc_update(t, crc, p[k]);
    for (; k + 4 <= n; k += 4) {  // aligned words, bytes in stream order
        const uint32_t w = *reinterpret_cast<const uint32_t *>(p + k);
        crc = ffv1::crc_update(t, crc, (uint8_t)w);
        crc = ffv1::crc_update(t, crc, (uint8_t)(w >> 8));
        crc = ffv1::crc_update(t, crc, (uint8_t)(w >> 16));
        crc = ffv1::crc_update(t, crc, (uint8_t)(w >> 24));
    }
    for (; k < n; ++k) crc = ffv1::crc_update(t, crc, p[k]);
    if (crc) status[i] = ffv1::LM_FFV1_CRC;
}

template <bool RANGE>
__global__ void __launch_bounds__(LM_FFV1_CHAINS_PER_CTA, 1) k_ffv1_decode(const ffv1::Record *__restrict__ rec, const uint8_t *__restrict__ initial,
                                                                        const uint8_t *__restrict__ payload, const int64_t *__restrict__ soff,
                                                                        const int32_t *__restrict__ slen, int32_t *__restrict__ status,
                                                                        uint8_t *__restrict__ out, int rows, int cols,
                                                                        const LmFfv1Chain *__restrict__ chains, int nchains,
                                                                        uint8_t *__restrict__ work, int64_t work_bytes, int work_in_smem) {
    extern __shared__ uint4 smem[];
    ffv1::Tables &T = *reinterpret_cast<ffv1::Tables *>(smem);
    const uint4 *src = reinterpret_cast<const uint4 *>(&rec->t);
    for (int i = threadIdx.x; i < (int)(sizeof(ffv1::Tables) / 16); i += blockDim.x) smem[i] = src[i];
    __syncthreads();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nchains) return;
    uint8_t *w = work_in_smem ? reinterpret_cast<uint8_t *>(smem) + sizeof(ffv1::Tables) + threadIdx.x * work_bytes : work + (int64_t)c * work_bytes;
    const LmFfv1Chain d = chains[c];
    ffv1::decode_chain<RANGE>(*rec, T, initial, payload, soff, slen, status, out, rows, cols, d.f0, d.nf, d.s, w);
}

static_assert(sizeof(ffv1::Tables) % 16 == 0, "the tables are copied to shared memory in 16-byte words");

}  // namespace

size_t lm_ffv1_smem_tables() { return sizeof(ffv1::Tables); }

int lm_launch_ffv1_locate(const uint8_t *payload, const int64_t *offs, int64_t base, int64_t n, int S, int ec, int64_t *soff, int32_t *slen,
                          int32_t *status, cudaStream_t s) {
    if (n <= 0) return 0;
    k_ffv1_locate<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(payload, offs, base, n, S, ec, soff, slen, status);
    if (cudaGetLastError() != cudaSuccess) return -1;
    return 1;
}

int lm_launch_ffv1_crc(const uint8_t *payload, const int64_t *soff, const int32_t *slen, int64_t ns, int32_t *status, cudaStream_t s) {
    if (ns <= 0) return 0;
    k_ffv1_crc<<<(unsigned)((ns + 255) / 256), 256, 0, s>>>(payload, soff, slen, ns, status);
    if (cudaGetLastError() != cudaSuccess) return -1;
    return 1;
}

int lm_launch_ffv1_decode(const ffv1::Record *rec, int ac, const uint8_t *initial, const uint8_t *payload, const int64_t *soff,
                          const int32_t *slen, int32_t *status, uint8_t *out, int rows, int cols, const LmFfv1Chain *chains, int nchains,
                          uint8_t *work, int64_t work_bytes, int work_in_smem, cudaStream_t s) {
    if (nchains <= 0) return 0;
    const size_t smem = sizeof(ffv1::Tables) + (work_in_smem ? (size_t)LM_FFV1_CHAINS_PER_CTA * work_bytes : 0);
    auto kern = ac ? k_ffv1_decode<true> : k_ffv1_decode<false>;
    static LmDevOnce once;
    if (auto setup = once.first())
        if (lm_allow_max_dynamic_smem(k_ffv1_decode<true>) != cudaSuccess || lm_allow_max_dynamic_smem(k_ffv1_decode<false>) != cudaSuccess) return -1;
    const unsigned blocks = (unsigned)((nchains + LM_FFV1_CHAINS_PER_CTA - 1) / LM_FFV1_CHAINS_PER_CTA);
    kern<<<blocks, LM_FFV1_CHAINS_PER_CTA, smem, s>>>(rec, initial, payload, soff, slen, status, out, rows, cols, chains, nchains, work,
                                                      work_bytes, work_in_smem);
    if (cudaGetLastError() != cudaSuccess) return -1;
    return 1;
}
