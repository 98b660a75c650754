// w8_lab.cu -- standalone timing harness for the headline instantiation of feat_warp8_kernel
// (MFCC + log-mel, frame 1024 / hop 512, 2000 x 5 s clips), for quick A/B runs of kernel variants:
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -DDSPX_W8_LAB [-DDSPX_ABL=n] \
//        -o benchmarks/lab/w8_lab benchmarks/lab/w8_lab.cu -cudart shared
//   ./w8_lab [clips] [reps]        prints ms per launch, audio-s/s and checksums of both outputs
//
// The checksums let two variants be compared for identical results; numerical parity against the oracle is
// the job of tests/ (CPU replay of the same phase functions + the GPU tests), not of this harness.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../dsp_final_b200/csrc/dspx_internal.cuh"
#include "../../dsp_final_b200/csrc/tables.cuh"
#include "../../dsp_final_b200/csrc/feat_warp8.cuh"

namespace dspx {
static char g_err[512];
void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char *get_error() { return g_err; }
}  // namespace dspx

__global__ void synth_kernel(float *x, int64_t n_clips, int64_t len)
{
    const int64_t clip = blockIdx.x;
    float *dst = x + clip * len;
    unsigned s = 1234567u + 7919u * (unsigned)clip;
    const float f0 = 6.2831853f * (80.f + 37.f * (clip % 50)) / 44100.f;
    for (int64_t i = threadIdx.x; i < len; i += blockDim.x) {
        unsigned h = (unsigned)i * 2654435761u ^ s;
        h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
        const float noise = (float)(h & 0xffff) / 32768.f - 1.f;
        dst[i] = 0.5f * __sinf(f0 * (float)i) + 0.2f * __sinf(3.7f * f0 * (float)i + 1.f) + 0.1f * noise;
    }
}

__global__ void checksum_kernel(const float *x, int64_t n, double *out)
{
    double s = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s += (double)x[i] * (double)(1 + (i % 7));
    atomicAdd(out, s);
}

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); return 1; } } while (0)

int main(int argc, char **argv)
{
    using namespace dspx;
    const int64_t n_clips = argc > 1 ? atoll(argv[1]) : 2000, len = 220500;
    const int reps = argc > 2 ? atoi(argv[2]) : 20;
    const bool mfcc_only = argc > 4 && atoi(argv[4]) != 0;      // 4th argument: 1 = no log-mel output (the sweep's setting)
    dspx_plan pl;
    pl.cfg = dspx_config{44100, 1024, 512, 0, argc > 3 ? atoi(argv[3]) : 40, 13, 0.0, -1.0, 0.97, DSPX_WINDOW_HANN, 0};
    pl.P = 1024; pl.M = 512; pl.n_bins = 513; pl.device = 0;
    build_window(pl.cfg.window, pl.cfg.frame_length, pl.host.window);
    build_filterbank(pl.cfg.n_mels, pl.P, pl.cfg.sample_rate, 0.0, 22050.0, pl.host);
    build_dct2(pl.cfg.n_mfcc, pl.cfg.n_mels, pl.host.dct2);
    cudaDeviceProp prop{};
    CK(cudaGetDeviceProperties(&prop, 0));
    pl.sm_count = prop.multiProcessorCount;
    if (!warp8_supported(&pl)) { printf("unsupported\n"); return 1; }
    if (warp8_prepare(&pl) != DSPX_OK) { printf("prepare failed: %s\n", get_error()); return 1; }
    const int64_t T = 1 + (len - 1024) / 512;
    float *clips, *lm, *mf;
    double *cs;
    CK(cudaMalloc(&clips, n_clips * len * 4));
    CK(cudaMalloc(&lm, n_clips * T * pl.cfg.n_mels * 4));
    CK(cudaMalloc(&mf, n_clips * T * 13 * 4));
    CK(cudaMalloc(&cs, 16));
    synth_kernel<<<(unsigned)n_clips, 256>>>(clips, n_clips, len);
    CK(cudaDeviceSynchronize());
    const W8Params p = w8_batch_params(&pl, clips, n_clips, len, T, mfcc_only ? nullptr : lm, mf, 0);
    for (int i = 0; i < 3; i++)
        if (launch_warp8(&pl, W8_SHARE, p, true, 0) != DSPX_OK) { printf("launch failed: %s\n", get_error()); return 1; }
    CK(cudaDeviceSynchronize());
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0);
    for (int i = 0; i < reps; i++) launch_warp8(&pl, W8_SHARE, p, true, 0);
    cudaEventRecord(e1);
    CK(cudaDeviceSynchronize());
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    ms /= reps;
    double h[2] = {0, 0};
    CK(cudaMemset(cs, 0, 16));
    checksum_kernel<<<296, 256>>>(lm, n_clips * T * pl.cfg.n_mels, cs);
    checksum_kernel<<<296, 256>>>(mf, n_clips * T * 13, cs + 1);
    CK(cudaMemcpy(h, cs, 16, cudaMemcpyDeviceToHost));
    const double bytes = (double)n_clips * (4.0 * len + 4.0 * T * (13 + pl.cfg.n_mels));
    printf("abl=%d ms=%.4f audio_s_per_s=%.4e GBps=%.1f frac=%.4f lm_sum=%.10e mf_sum=%.10e\n",
#ifdef DSPX_ABL
           DSPX_ABL,
#else
           0,
#endif
           ms, n_clips * 5.0 / (ms * 1e-3), bytes / (ms * 1e-3) / 1e9, bytes / (ms * 1e-3) / 1e9 / 6534.8, h[0], h[1]);
    return 0;
}
