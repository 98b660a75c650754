// feat_select.cuh -- which feature kernel a plan uses (plan_derive), and per feature call the steps around it
// (feat_steps) and the layout of their scratch (feat_ws_carve).  Host code only, no launches: dspx.cu runs what it says
// (run_features), and the test-only replay library (emu.cu) exposes it so that the choice and the workspace can be
// checked on machines without a GPU.
#pragma once

#include <algorithm>

#include "dspx_internal.cuh"
#include "tables.cuh"
#include "feat_warp8.cuh"

namespace dspx {

// The host part of dspx_plan_create: transform geometry, tables (float64, rounded once to float32) and the kernel.
// warp8 when the configuration allows it and its tables fit in shared memory, else the generic kernel; a plan that asks
// for warp8 by name fails instead.  A warp8 plan's tables are in p->fast_host (warp8_release frees them).
inline int plan_derive(const dspx_config *cfg, dspx_plan *p)
{
    p->cfg = *cfg;
    const int nfft_raw = cfg->n_fft > 0 ? cfg->n_fft : cfg->frame_length;
    const int64_t P = next_pow_two(nfft_raw);
    if (P < 16 || P > 8192) {
        set_error("transform length %lld unsupported (power of two in [16, 8192])", (long long)P);
        return DSPX_EUNSUPPORTED;
    }
    p->P = (int)P;
    p->M = p->P / 2;
    p->n_bins = p->P / 2 + 1;
    p->take_feat = cfg->frame_length < p->P ? cfg->frame_length : p->P;       // mfcc.py:89-98
    p->take_stft = cfg->frame_length < nfft_raw ? cfg->frame_length : nfft_raw; // fft.py:32-33
    int m = p->M, ns = 0;
    while (m > 1) {
        if (m % 4 == 0) { p->radix[ns++] = 4; m /= 4; }
        else { p->radix[ns++] = 2; m /= 2; }
    }
    p->n_stages = ns;

    HostTables &h = p->host;
    if (!build_window(cfg->window, cfg->frame_length, h.window)) {
        set_error("Unsupported window: %d", cfg->window);
        return DSPX_EINVAL;
    }
    const double f_max = cfg->f_max < 0.0 ? (double)cfg->sample_rate / 2.0 : cfg->f_max;
    build_filterbank(cfg->n_mels, p->P, cfg->sample_rate, cfg->f_min, f_max, h);
    build_dct2(cfg->n_mfcc, cfg->n_mels, h.dct2);
    h.window32.assign(h.window.begin(), h.window.end());
    h.dct2_32.assign(h.dct2.begin(), h.dct2.end());
    h.tw.resize(p->P);
    for (int j = 0; j < p->P; j++) {
        const double a = -2.0 * M_PI * (double)j / (double)p->P;
        h.tw[j] = make_float2((float)std::cos(a), (float)std::sin(a));
    }

    p->kernel = DSPX_KERNEL_GENERIC;
    if (cfg->kernel == DSPX_KERNEL_GENERIC) return DSPX_OK;
    if (!warp8_supported(p)) {
        if (cfg->kernel != DSPX_KERNEL_WARP8) return DSPX_OK;
        set_error("warp8 kernel does not support this configuration");
        return DSPX_EUNSUPPORTED;
    }
    auto *pd = new W8PlanData();
    warp8_build_tables(p, pd->blob, pd->tb);
    static_cast<W8Shapes &>(*pd) = warp8_shapes(pd->tb, cfg->n_mels);
    if (pd->smem > MAX_OPTIN_SMEM) {
        // tables too large for shared memory (e.g. 256 mels at n_fft 1024, 128 mels at 4096): the generic kernel
        delete pd;
        set_error("warp8: tables too large for shared memory");
        return cfg->kernel == DSPX_KERNEL_WARP8 ? DSPX_EUNSUPPORTED : DSPX_OK;
    }
    p->fast_host = pd;
    p->kernel = DSPX_KERNEL_WARP8;
    return DSPX_OK;
}

// The clips of a feature call: n_clips rows of clip_len samples of dtype, stride samples apart, from samples; or a
// ragged batch (tab on the host, tab_dev the same dspx_ragged_layout table on the device; clip_len and stride 0).
// samples may be null for rows that will sit at the start of a cudaMalloc'd buffer: only its alignment is read here.
struct FeatBatch {
    const void *samples;
    int dtype;
    int normalize;            // PCM16: divide every clip by its peak (0 or 1)
    int64_t n_clips, clip_len, stride;
    const dspx_ragged_clip *tab, *tab_dev;
};

// What a feature call runs, in this order (run_features): the ragged first-pair array, the PCM16 peaks or the float32
// conversion, the zeroed embedding sums, the feature kernel, the embeddings.
struct FeatSteps {
    int64_t T;                // frames per clip; a ragged batch: of its longest clip
    W8Path path;              // the feature kernel (W8_UNSUPPORTED when per_clip: each clip's call chooses its own)
    bool convert;             // PCM16 converted by pcm16_to_float_kernel into scratch first (ragged: clip by clip)
    bool peaks;               // pcm16_peak_kernel first: the kernel converts in its loads and normalises by the peaks
    bool fused;               // embeddings alone, accumulated inside the kernel and finalised by embed_finalize_kernel
    bool mfcc_scratch;        // embeddings alone that do not fuse: the statistics of an MFCC tensor in scratch
    bool per_clip;            // a ragged batch on a plan without a ragged kernel (generic, n_fft 4096): one call per clip
};

// The one place that decides a feature call's steps; warp8_select picks the kernel.  want_mfcc / want_embed: the call
// has an MFCC / an embedding output.  PCM16 converts inside the kernel's loads wherever a kernel does (warp8 at n_fft
// 512 / 1024 / 2048); embeddings alone fuse into float32 kernels on the 8-byte grid, for clips of at most
// w8_embed_max_frames frames.
inline FeatSteps feat_steps(const dspx_plan *pl, const FeatBatch &b, bool want_mfcc, bool want_embed)
{
    FeatSteps s{};
    const bool ragged = b.tab != nullptr, pcm = b.dtype == DSPX_DTYPE_PCM16, alone = want_embed && !want_mfcc;
    if (ragged)
        for (int64_t i = 0; i < b.n_clips; i++) s.T = std::max(s.T, b.tab[i].n_frames);
    else
        s.T = 1 + (b.clip_len - pl->cfg.frame_length) / pl->cfg.hop_length;
    auto select = [&](W8Want want) { return warp8_select(pl, b.samples, b.stride, b.dtype, ragged, b.n_clips, s.T, want); };
    s.fused = alone && select(W8_WANT_EMBED) != W8_UNSUPPORTED;
    s.mfcc_scratch = alone && !s.fused;
    s.path = select(s.fused ? W8_WANT_EMBED : W8_WANT_FEATURES);
    s.per_clip = ragged && s.path == W8_UNSUPPORTED;
    s.convert = pcm && s.path == W8_UNSUPPORTED;
    if (s.convert && !ragged)       // the float32 copy: rows of clip_len at the start of the scratch
        s.path = warp8_select(pl, nullptr, b.clip_len, DSPX_DTYPE_F32, false, b.n_clips, s.T, W8_WANT_FEATURES);
    s.peaks = pcm && !s.convert && b.normalize;
    return s;
}

// Scratch of a feature call; null where no step needs it
struct FeatWs {
    uint32_t *rpairs = nullptr;   // [n_clips + 1] first frame pair of every clip of a ragged batch, then the total
    int *peaks = nullptr;         // [n_clips]
    long long *eacc = nullptr;    // [n_clips][2][n_mfcc] fixed-point embedding sums
    float *mfcc = nullptr;        // [frames][n_mfcc]
    float *f32 = nullptr;         // converted clips; a ragged batch: one clip at a time
};

// One layout of a call's scratch for the size queries and the launches, every region 256-byte aligned from a 256-byte
// aligned base.  Returns the size dspx_features_ragged_workspace reports; with base, also the pointers.
inline size_t feat_ws_carve(const dspx_plan *pl, const FeatBatch &b, const FeatSteps &s, char *base, FeatWs *ws)
{
    const int64_t n = b.n_clips, C = pl->cfg.n_mfcc;
    int64_t frames = n * s.T, samples = n * b.clip_len;
    if (b.tab) {
        frames = n > 0 ? b.tab[n - 1].first_frame + b.tab[n - 1].n_frames : 0;
        samples = 0;
        for (int64_t i = 0; i < n; i++) samples = std::max(samples, b.tab[i].length);
    }
    size_t off = 0;
    auto take = [&](size_t bytes) -> char * {
        char *p = bytes && base ? base + off : nullptr;
        off += align256(bytes);
        return p;
    };
    FeatWs w;
    w.rpairs = reinterpret_cast<uint32_t *>(take(b.tab && !s.per_clip ? (size_t)(n + 1) * sizeof(uint32_t) : 0));
    w.peaks = reinterpret_cast<int *>(take(s.peaks ? (size_t)n * sizeof(int) : 0));
    w.eacc = reinterpret_cast<long long *>(take(s.fused ? (size_t)n * 2 * C * sizeof(long long) : 0));
    w.mfcc = reinterpret_cast<float *>(take(s.mfcc_scratch ? (size_t)frames * C * sizeof(float) : 0));
    w.f32 = reinterpret_cast<float *>(take(s.convert ? (size_t)samples * sizeof(float) : 0));
    if (ws) *ws = w;
    return off + 256;
}

}  // namespace dspx
