// ingest.cuh -- PCM16 ingest on the GPU (SURVEY.md 8f row f2).
//
// Replaces the per-clip CPU prologue of the reference, src/utils/audio.py:19-38 as used by
// src/features/cache.py:66-67:
//   soundfile.read(dtype="float32") of a PCM16 file  ->  x = int16 / 32768        (exact in float32)
//   normalize_audio: peak = max|x|; x / peak if peak > 0                             (float32 division)
// The division is the correctly rounded float32 quotient, so the result is bit-identical to NumPy's.
// One CTA per clip: pass 1 reduces the peak, pass 2 re-reads the clip (L2-resident) and writes float32.
// Shipping int16 over PCIe instead of float32 halves the host->device bytes of the end-to-end path.
#pragma once

#include "dspx_internal.cuh"

namespace dspx {

#if defined(__CUDACC__)
__global__ void __launch_bounds__(256) pcm16_to_float_kernel(const int16_t *pcm, int64_t clip_len, int64_t pcm_stride,
                                                            int normalize, float *out, int64_t out_stride)
{
    const int16_t *src = pcm + (size_t)blockIdx.x * pcm_stride;
    float *dst = out + (size_t)blockIdx.x * out_stride;
    __shared__ int s_peak[8];
    float peak = 1.0f;
    if (normalize) {
        int m = 0;
        for (int64_t i = threadIdx.x; i < clip_len; i += 256) {
            const int v = src[i];
            m = max(m, v < 0 ? -v : v);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
        if ((threadIdx.x & 31) == 0) s_peak[threadIdx.x >> 5] = m;
        __syncthreads();
        m = s_peak[0];
#pragma unroll
        for (int w = 1; w < 8; w++) m = max(m, s_peak[w]);
        peak = m > 0 ? (float)m * (1.0f / 32768.0f) : 1.0f;            // peak == 0: leave the clip as it is
    }
    for (int64_t i = threadIdx.x; i < clip_len; i += 256) {
        const float x = (float)src[i] * (1.0f / 32768.0f);             // exact
        dst[i] = normalize ? __fdiv_rn(x, peak) : x;
    }
}
// max |sample| of every clip: all the fused PCM16 path needs before the feature kernel converts the samples in its
// own loads (w8_pcm_to_float).  One CTA per clip; the clip was just copied to the device, so this read is L2-warm.
// rtab (ragged batches): clip b is rtab[b].length samples from rtab[b].start instead of clip_len from b * pcm_stride.
__global__ void __launch_bounds__(256) pcm16_peak_kernel(const int16_t *pcm, int64_t clip_len, int64_t pcm_stride, int *peaks,
                                                         const dspx_ragged_clip *rtab = nullptr)
{
    const int16_t *src = pcm + (rtab ? rtab[blockIdx.x].start : (int64_t)blockIdx.x * pcm_stride);
    if (rtab) clip_len = rtab[blockIdx.x].length;
    __shared__ int s_peak[8];
    int m = 0;
    const int64_t pairs = ((reinterpret_cast<uintptr_t>(src) & 3) == 0) ? clip_len / 2 : 0;      // 32-bit loads when aligned
    const int *src2 = reinterpret_cast<const int *>(src);
    for (int64_t i = threadIdx.x; i < pairs; i += 256) {
        const int v = src2[i];
        const int lo = (int)(short)(v & 0xffff), hi = v >> 16;
        m = max(m, max(lo < 0 ? -lo : lo, hi < 0 ? -hi : hi));
    }
    for (int64_t i = 2 * pairs + threadIdx.x; i < clip_len; i += 256) {
        const int v = src[i];
        m = max(m, v < 0 ? -v : v);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
    if ((threadIdx.x & 31) == 0) s_peak[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 1; w < 8; w++) m = max(m, s_peak[w]);
        peaks[blockIdx.x] = m;
    }
}
#endif

}  // namespace dspx
