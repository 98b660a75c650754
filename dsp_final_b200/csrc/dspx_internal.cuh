// dspx_internal.cuh -- plan object, error plumbing and small helpers shared by
// the kernels of libdspx.so.  Not part of the public ABI (include/dspx.h is).
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dspx.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

// Host/device portability shims: the "phase" functions of the kernels are
// __host__ __device__ so that csrc/emu.cu can replay them thread by thread on
// the CPU (tests only).  On the device the rounding-exact intrinsics are used;
// the host build is compiled with -ffp-contract=off so plain ops round the same.
#if defined(__CUDA_ARCH__)
#define DSPX_FMUL_RN(a, b) __fmul_rn((a), (b))
#define DSPX_FSUB_RN(a, b) __fsub_rn((a), (b))
#else
#define DSPX_FMUL_RN(a, b) ((float)((float)(a) * (float)(b)))
#define DSPX_FSUB_RN(a, b) ((float)((float)(a) - (float)(b)))
#endif
#define DSPX_HD __host__ __device__ __forceinline__

namespace dspx {

void set_error(const char *fmt, ...);
const char *get_error();

#define DSPX_CUDA_CHECK(expr)                                                            \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            ::dspx::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                              __FILE__, __LINE__);                                       \
            return DSPX_ECUDA;                                                           \
        }                                                                                \
    } while (0)

#define DSPX_REQUIRE(cond, ...)                 \
    do {                                        \
        if (!(cond)) {                          \
            ::dspx::set_error(__VA_ARGS__);     \
            return DSPX_EINVAL;                 \
        }                                       \
    } while (0)

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// A caller's workspace moved up to the next 256-byte boundary: the workspace size queries leave 256 bytes for this
inline char *ws_align(void *p)
{
    char *c = static_cast<char *>(p);
    return c ? c + ((256 - (reinterpret_cast<uintptr_t>(c) & 255)) & 255) : nullptr;
}

// Opt-in dynamic shared memory: a per-function, per-device attribute shared by every plan and thread.  It is
// set once per (kernel, device) to the architectural maximum and never lowered, so launches of plans with
// different shared-memory sizes cannot race on it (the size actually used is a launch argument).
constexpr size_t MAX_OPTIN_SMEM = 227 * 1024;
#if defined(__CUDACC__)
template <class Kernel>
inline cudaError_t optin_max_smem(Kernel kernel, std::atomic<unsigned char> (&done)[64], int device)
{
    std::atomic<unsigned char> &flag = done[device & 63];
    if (flag.load(std::memory_order_acquire)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MAX_OPTIN_SMEM);
    if (e == cudaSuccess) flag.store(1, std::memory_order_release);
    return e;
}
#endif

// Tables built on the host in float64 with the reference's formulas, rounded
// once to float32 (SURVEY.md appendix A.7: the mel bin floor is only safe in
// float64).  See tables.cuh for the file:line of each formula.
struct HostTables {
    std::vector<double> window;        // [frame_length]
    std::vector<double> fbank;         // dense [n_mels, n_bins]
    std::vector<double> dct2;          // [n_mfcc, n_mels], already times 2
    std::vector<int32_t> fb_start;     // per filter: first non-zero bin
    std::vector<int32_t> fb_cnt;       //             number of bins from there to the last non-zero
    std::vector<int32_t> fb_off;       //             offset into fb_w
    std::vector<float> fb_w;           // weights, row after row
    // per-bin view of the same filterbank (each bin feeds at most two adjacent
    // filters; see tables.cuh): filter index of the falling edge and weights
    std::vector<int32_t> bin_filt;     // [n_bins] index f such that the bin feeds f (fall) and f+1 (rise); -1.. allowed
    std::vector<float> bin_wfall;      // [n_bins]
    std::vector<float> bin_wrise;      // [n_bins]
    bool two_band_ok = false;          // per-bin form is exact for this filterbank
    // float32 tables the generic kernel reads besides fb_*: window, DCT, twiddles exp(-2 pi i j / P)
    std::vector<float> window32, dct2_32;
    std::vector<float2> tw;
};

}  // namespace dspx

struct dspx_plan {
    dspx_config cfg;
    int device = 0;
    int sm_count = 0;
    int P = 0;              // transform length (power of two)
    int M = 0;              // P / 2: complex FFT length of the packed real transform
    int n_bins = 0;
    int take_feat = 0;
    int take_stft = 0;
    int kernel = DSPX_KERNEL_GENERIC;
    int n_stages = 0;
    int radix[16] = {0};
    dspx::HostTables host;
    // device tables
    float *d_window = nullptr;          // [frame_length]
    float2 *d_tw = nullptr;             // [P]  exp(-2*pi*i*j/P)
    int32_t *d_fb_start = nullptr, *d_fb_cnt = nullptr, *d_fb_off = nullptr;
    float *d_fb_w = nullptr;
    float *d_dct2 = nullptr;            // [n_mfcc, n_mels]
    int32_t *d_bin_filt = nullptr;
    float *d_bin_wfall = nullptr, *d_bin_wrise = nullptr;
    void *d_fast_tables = nullptr;      // packed tables of the warp8 kernel (feat_warp8.cuh)
    size_t fast_tables_bytes = 0;
    void *fast_host = nullptr;          // host-side descriptor of those tables (W8PlanData)
    // host pipeline state (pinned staging, streams), created lazily by the *_host calls
    void *host_pipe = nullptr;
};
