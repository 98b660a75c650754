// dspx.cu -- C ABI of libdspx.so (include/dspx.h): plan management, kernel
// launches and the host-buffer pipeline.  All numerical work is in the .cuh
// kernels included below; this file only validates arguments and launches.
#include <cstdarg>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <thread>

#include "dspx_internal.cuh"
#include "tables.cuh"
#include "feat_generic.cuh"
#include "feat_warp8.cuh"
#include "feat_warp8_x2.cuh"
#include "fft_generic.cuh"
#include "retrieval.cuh"
#include "retrieval_f32.cuh"
#include "retrieval_tc.cuh"
#include "ingest.cuh"

// the ctypes binding (dsp_final_b200/_lib.py) mirrors these layouts; tests assert the same numbers
static_assert(sizeof(dspx_config) == 56 && offsetof(dspx_config, f_min) == 24 && offsetof(dspx_config, window) == 48,
              "dspx_config layout changed: update _lib.DspxConfig");
static_assert(sizeof(dspx_plan_info) == 32, "dspx_plan_info layout changed: update _lib.DspxPlanInfo");

namespace dspx {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char *get_error() { return g_err; }

template <typename T>
static int upload(const std::vector<T> &h, T **d)
{
    *d = nullptr;
    if (h.empty()) return DSPX_OK;
    DSPX_CUDA_CHECK(cudaMalloc((void **)d, h.size() * sizeof(T)));
    DSPX_CUDA_CHECK(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return DSPX_OK;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard()
    {
        if (ok && prev >= 0) cudaSetDevice(prev);
    }
};

// ---- host pipeline state (pinned staging + device slots) -----------------------
constexpr int PIPE_SLOTS = 3;
struct HostPipe {
    std::mutex mu;
    cudaStream_t stream[PIPE_SLOTS] = {nullptr, nullptr, nullptr};
    void *d_in[PIPE_SLOTS] = {nullptr, nullptr, nullptr};
    void *d_out[PIPE_SLOTS] = {nullptr, nullptr, nullptr};
    void *h_in[PIPE_SLOTS] = {nullptr, nullptr, nullptr};    // pinned staging (pageable callers)
    void *h_out[PIPE_SLOTS] = {nullptr, nullptr, nullptr};
    void *d_f32[PIPE_SLOTS] = {nullptr, nullptr, nullptr};   // float32 clips converted from PCM16
    size_t in_bytes = 0, out_bytes = 0, hin_bytes = 0, hout_bytes = 0, f32_bytes = 0;
    void release()
    {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (d_in[i]) cudaFree(d_in[i]);
            if (d_out[i]) cudaFree(d_out[i]);
            if (h_in[i]) cudaFreeHost(h_in[i]);
            if (h_out[i]) cudaFreeHost(h_out[i]);
            if (d_f32[i]) cudaFree(d_f32[i]);
            d_f32[i] = nullptr;
            if (stream[i]) cudaStreamDestroy(stream[i]);
            d_in[i] = d_out[i] = h_in[i] = h_out[i] = nullptr;
            stream[i] = nullptr;
        }
        in_bytes = out_bytes = hin_bytes = hout_bytes = f32_bytes = 0;
    }
};

static void plan_free_device(dspx_plan *p)
{
    cudaFree(p->d_window);
    cudaFree(p->d_tw);
    cudaFree(p->d_fb_start);
    cudaFree(p->d_fb_cnt);
    cudaFree(p->d_fb_off);
    cudaFree(p->d_fb_w);
    cudaFree(p->d_dct2);
    cudaFree(p->d_bin_filt);
    cudaFree(p->d_bin_wfall);
    cudaFree(p->d_bin_wrise);
    cudaFree(p->d_fast_tables);
    warp8_release(p);
    if (p->host_pipe) {
        auto *hp = static_cast<HostPipe *>(p->host_pipe);
        hp->release();
        delete hp;
        p->host_pipe = nullptr;
    }
}

// ---- launch helpers ----------------------------------------------------------------
static int launch_generic(const dspx_plan *pl, const float *clips, int64_t n_clips, int64_t clip_len,
                          int64_t clip_stride, int64_t T, int take, int pre, float *logmel, float *mfcc,
                          float2 *stft, cudaStream_t st, int nchw = 0)
{
    GenParams gp{};
    gp.clips = clips;
    gp.n_clips = n_clips;
    gp.clip_len = clip_len;
    gp.clip_stride = clip_stride;
    gp.n_frames = T;
    gp.frame_length = pl->cfg.frame_length;
    gp.hop = pl->cfg.hop_length;
    gp.take = take;
    gp.P = pl->P;
    gp.M = pl->M;
    gp.n_bins = pl->n_bins;
    gp.n_stages = pl->n_stages;
    for (int i = 0; i < 16; i++) gp.radix[i] = pl->radix[i];
    gp.n_mels = pl->cfg.n_mels;
    gp.n_mfcc = pl->cfg.n_mfcc;
    int G = 1024 / pl->M;
    if (G < 1) G = 1;
    if (G > 16) G = 16;
    gp.G = G;
    // enough CTAs to fill the machine when the batch is small, whole clips per CTA when it is large
    const int64_t groups = (T + G - 1) / G;
    const int64_t want_ctas = (int64_t)pl->sm_count * 8;
    int64_t splits = n_clips >= want_ctas ? 1 : (want_ctas + n_clips - 1) / n_clips;
    if (splits > groups) splits = groups;
    const int64_t groups_per_cta = (groups + splits - 1) / splits;
    gp.frames_per_cta = (int)(groups_per_cta * G);
    gp.ctas_per_clip = (int)((T + gp.frames_per_cta - 1) / gp.frames_per_cta);
    gp.pre = pre;
    gp.alpha = (float)pl->cfg.pre_emphasis;
    gp.window = pl->d_window;
    gp.tw = pl->d_tw;
    gp.fb_start = pl->d_fb_start;
    gp.fb_cnt = pl->d_fb_cnt;
    gp.fb_off = pl->d_fb_off;
    gp.fb_w = pl->d_fb_w;
    gp.dct2 = pl->d_dct2;
    gp.logmel = logmel;
    gp.lm_ts = nchw ? 1 : pl->cfg.n_mels;
    gp.lm_fs = nchw ? T : 1;
    gp.mfcc = mfcc;
    gp.stft = stft;
    const size_t smem = gen_smem_bytes(G, pl->M, gp.n_mels);
    const int64_t grid = n_clips * gp.ctas_per_clip;
    DSPX_REQUIRE(grid > 0 && grid < (int64_t)2147483647, "batch too large for one launch (%lld CTAs)", (long long)grid);
    DSPX_REQUIRE(smem <= MAX_OPTIN_SMEM, "generic kernel needs %zu bytes of shared memory", smem);
    static std::atomic<unsigned char> optin[64];
    DSPX_CUDA_CHECK(optin_max_smem(feat_generic_kernel, optin, pl->device));
    feat_generic_kernel<<<(unsigned)grid, GEN_THREADS, smem, st>>>(gp);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

// Features of an equal-length batch on the path warp8_select chose (PCM16: int16 rows, peaks per clip or null).
static int launch_features(const dspx_plan *pl, W8Path path, const void *clips, int64_t n_clips, int64_t clip_len,
                           int64_t clip_stride, int64_t T, float *logmel, float *mfcc, cudaStream_t st, int nchw = 0,
                           long long *eacc = nullptr, const int *peaks = nullptr)
{
    const bool pre = pl->cfg.pre_emphasis > 0.0;
    const float *x = static_cast<const float *>(clips);
    if (path == W8_GENERIC)
        return launch_generic(pl, x, n_clips, clip_len, clip_stride, T, pl->take_feat, pre ? 1 : 0, logmel, mfcc, nullptr, st, nchw);
    if (path == W8_X2 || path == W8_X2_AL4)
        return launch_warp8_x2(pl, path == W8_X2_AL4, x, n_clips, clip_stride, T, logmel, mfcc, st, nchw);
    W8Params p = w8_batch_params(pl, clips, n_clips, clip_stride, T, logmel, mfcc, nchw);
    p.eacc = eacc;
    p.peaks = peaks;
    return launch_warp8(pl, path, p, pre, st);
}

static int launch_embed(const float *feats, int64_t n_clips, int64_t T, int C, float *out, cudaStream_t st,
                        const dspx_ragged_clip *rtab = nullptr)
{
    const int cw = C < 128 ? C : 128;
    const int groups = 128 / cw;
    const size_t smem = ((size_t)groups * C + C) * sizeof(double);
    DSPX_REQUIRE(smem <= 48 * 1024, "n_coef %d too large for embed_stats", C);
    DSPX_REQUIRE(n_clips < (int64_t)2147483647, "too many clips for one launch");
    embed_stats_kernel<<<(unsigned)n_clips, 128, smem, st>>>(feats, T, C, out, rtab);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

// embed without mfcc: the fused path -- the kernel accumulates per-clip sums into `eacc` ([n_clips][2][n_mfcc]
// int64, caller-provided scratch) and embed_finalize_kernel writes mean / std; no MFCC tensor exists anywhere.
static int features_device(const dspx_plan *pl, const float *clips, int64_t n_clips, int64_t clip_len,
                           int64_t clip_stride, float *logmel, float *mfcc, float *embed, cudaStream_t st, int nchw = 0,
                           long long *eacc = nullptr)
{
    const int64_t T = dspx_num_frames(pl, clip_len);
    if (T < 0) return DSPX_EINVAL;
    const bool fused = embed && !mfcc;
    const W8Path path = warp8_select(pl, clips, clip_stride, DSPX_DTYPE_F32, false, n_clips, T,
                                     fused ? W8_WANT_EMBED : W8_WANT_FEATURES);
    if (path == W8_UNSUPPORTED) {
        set_error("embeddings without an MFCC buffer need the warp8 kernel (n_fft 512 / 1024 / 2048), frame_length = "
                  "n_fft, an even hop and row stride and 8-byte aligned clips");
        return DSPX_EUNSUPPORTED;
    }
    const int C = pl->cfg.n_mfcc;
    if (fused) DSPX_CUDA_CHECK(cudaMemsetAsync(eacc, 0, (size_t)n_clips * 2 * C * sizeof(long long), st));
    int rc = launch_features(pl, path, clips, n_clips, clip_len, clip_stride, T, logmel, mfcc, st, nchw, fused ? eacc : nullptr);
    if (rc != DSPX_OK) return rc;
    if (fused) {
        const int64_t total = n_clips * C;
        embed_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(eacc, n_clips, T, C, embed);
        DSPX_CUDA_CHECK(cudaGetLastError());
        return DSPX_OK;
    }
    if (embed) rc = launch_embed(mfcc, n_clips, T, C, embed, st);
    return rc;
}

// PCM16 clips on the device -> features, conversion and peak normalisation inside the feature kernel's sample loads.
// peaks_ws: n_clips ints of scratch (only touched when normalize).  warp8 plans only.
static int features_device_pcm16(const dspx_plan *pl, const int16_t *pcm, int64_t n_clips, int64_t clip_len, int64_t pcm_stride,
                                 int normalize, float *logmel, float *mfcc, float *embed, int *peaks_ws, cudaStream_t st)
{
    const int64_t T = dspx_num_frames(pl, clip_len);
    if (T < 0) return DSPX_EINVAL;
    const W8Path path = warp8_select(pl, pcm, pcm_stride, DSPX_DTYPE_PCM16, false, n_clips, T, W8_WANT_FEATURES);
    if (path == W8_UNSUPPORTED) {
        set_error("fused PCM16 ingest needs the warp8 kernel (n_fft 512 / 1024 / 2048) and fewer than 2^31 frame pairs: "
                  "convert with dspx_pcm16_to_float first");
        return DSPX_EUNSUPPORTED;
    }
    DSPX_REQUIRE(!embed || mfcc, "embed_out needs mfcc_out on the PCM16 path");
    DSPX_REQUIRE(n_clips < (int64_t)2147483647, "too many clips for one launch");
    if (normalize) {
        DSPX_REQUIRE(peaks_ws, "peak normalisation needs the workspace");
        pcm16_peak_kernel<<<(unsigned)n_clips, 256, 0, st>>>(pcm, clip_len, pcm_stride, peaks_ws);
        DSPX_CUDA_CHECK(cudaGetLastError());
    }
    int rc = launch_features(pl, path, pcm, n_clips, clip_len, pcm_stride, T, logmel, mfcc, st, 0, nullptr,
                             normalize ? peaks_ws : nullptr);
    if (rc != DSPX_OK) return rc;
    if (embed) rc = launch_embed(mfcc, n_clips, T, pl->cfg.n_mfcc, embed, st);
    return rc;
}

// complex STFT: the warp8 kernel when frame_length == n_fft in {512, 1024, 2048} and the rows are aligned
static int stft_device(const dspx_plan *pl, const float *clips, int64_t n_clips, int64_t clip_len, int64_t clip_stride,
                       int64_t T, int pre, float2 *out, cudaStream_t st)
{
    const W8Path path = warp8_select(pl, clips, clip_stride, DSPX_DTYPE_F32, false, n_clips, T, W8_WANT_STFT);
    if (path == W8_GENERIC)
        return launch_generic(pl, clips, n_clips, clip_len, clip_stride, T, pl->take_stft, pre, nullptr, nullptr, out, st);
    W8Params p = w8_batch_params(pl, clips, n_clips, clip_stride, T, nullptr, nullptr, 0);
    p.stft = out;
    return launch_warp8(pl, path, p, pre != 0, st);
}

// ---- ragged batches (dspx_features_ragged) ------------------------------------------------------------
// Workspace of one call, carved the same way by the size query and the launch (offsets from a 256-byte aligned base):
// the compact first-pair array the ragged kernel searches, PCM16 peaks, fixed-point embedding sums, MFCC scratch for
// embeddings without an MFCC output (when the fused path does not apply), and on plans without a ragged kernel a
// float32 copy of one PCM16 clip at a time.
struct RaggedWs {
    uint32_t *rpairs = nullptr;
    int *peaks = nullptr;
    long long *eacc = nullptr;
    float *mfcc = nullptr;
    float *f32 = nullptr;
};

static W8Path ragged_path(const dspx_plan *pl, int dtype, W8Want want)
{
    return warp8_select(pl, nullptr, 0, dtype, true, 0, 0, want);
}

static size_t ragged_ws_carve(const dspx_plan *pl, const dspx_ragged_clip *tab, int64_t n_clips, int dtype, int normalize,
                              bool want_mfcc, bool want_embed, char *base, RaggedWs *ws)
{
    const bool pcm = dtype == DSPX_DTYPE_PCM16, rk = ragged_path(pl, dtype, W8_WANT_FEATURES) != W8_UNSUPPORTED;
    const bool fused = want_embed && !want_mfcc && ragged_path(pl, dtype, W8_WANT_EMBED) != W8_UNSUPPORTED;
    int64_t total_frames = 0, max_len = 0;
    if (n_clips > 0) total_frames = tab[n_clips - 1].first_frame + tab[n_clips - 1].n_frames;
    for (int64_t i = 0; i < n_clips; i++) max_len = std::max(max_len, tab[i].length);
    const size_t b_pairs = rk ? (size_t)(n_clips + 1) * sizeof(uint32_t) : 0;
    const size_t b_peaks = rk && pcm && normalize ? (size_t)n_clips * sizeof(int) : 0;
    const size_t b_eacc = fused ? (size_t)n_clips * 2 * pl->cfg.n_mfcc * sizeof(long long) : 0;
    const size_t b_mfcc = want_embed && !want_mfcc && !fused ? (size_t)total_frames * pl->cfg.n_mfcc * sizeof(float) : 0;
    const size_t b_f32 = !rk && pcm ? (size_t)max_len * sizeof(float) : 0;
    size_t off = 0;
    auto take = [&](size_t bytes) -> char * {
        char *p = bytes && base ? base + off : nullptr;
        off += align256(bytes);
        return p;
    };
    RaggedWs w;
    w.rpairs = reinterpret_cast<uint32_t *>(take(b_pairs));
    w.peaks = reinterpret_cast<int *>(take(b_peaks));
    w.eacc = reinterpret_cast<long long *>(take(b_eacc));
    w.mfcc = reinterpret_cast<float *>(take(b_mfcc));
    w.f32 = reinterpret_cast<float *>(take(b_f32));
    if (ws) *ws = w;
    return off + 256;
}

// Plans without a ragged kernel: one stream-ordered feature call per clip into its rows of the stacked outputs, the
// embeddings from the stacked MFCCs at the end.  Each clip is computed exactly as a [1, length] call computes it.
static int features_ragged_per_clip(const dspx_plan *pl, const void *samples, int pcm, int normalize,
                                    const dspx_ragged_clip *tab_dev, const dspx_ragged_clip *tab, int64_t n_clips,
                                    float *logmel, float *mfcc, float *embed, const RaggedWs &ws, cudaStream_t st)
{
    float *mf = mfcc ? mfcc : (embed ? ws.mfcc : nullptr);
    for (int64_t i = 0; i < n_clips; i++) {
        const int64_t len = tab[i].length, ff = tab[i].first_frame;
        const float *x = static_cast<const float *>(samples) + tab[i].start;
        if (pcm) {
            pcm16_to_float_kernel<<<1, 256, 0, st>>>(static_cast<const int16_t *>(samples) + tab[i].start, len, len,
                                                     normalize ? 1 : 0, ws.f32, len);
            DSPX_CUDA_CHECK(cudaGetLastError());
            x = ws.f32;
        }
        const int rc = features_device(pl, x, 1, len, len, logmel ? logmel + ff * pl->cfg.n_mels : nullptr,
                                       mf ? mf + ff * pl->cfg.n_mfcc : nullptr, nullptr, st);
        if (rc != DSPX_OK) return rc;
    }
    return embed ? launch_embed(mf, n_clips, 1, pl->cfg.n_mfcc, embed, st, tab_dev) : DSPX_OK;
}

static int features_ragged(const dspx_plan *pl, const void *samples, int dtype, int normalize, const dspx_ragged_clip *tab_dev,
                           const dspx_ragged_clip *tab, int64_t n_clips, float *logmel, float *mfcc, float *embed,
                           char *ws_base, cudaStream_t st)
{
    const int pcm = dtype == DSPX_DTYPE_PCM16 ? 1 : 0;
    RaggedWs ws;
    ragged_ws_carve(pl, tab, n_clips, dtype, normalize, mfcc != nullptr, embed != nullptr, ws_base, &ws);
    const bool fused = ws.eacc != nullptr;                   // embeddings alone, accumulated inside the feature kernel
    const W8Path path = ragged_path(pl, dtype, fused ? W8_WANT_EMBED : W8_WANT_FEATURES);
    if (path == W8_UNSUPPORTED)
        return features_ragged_per_clip(pl, samples, pcm, normalize, tab_dev, tab, n_clips, logmel, mfcc, embed, ws, st);
    const int C = pl->cfg.n_mfcc;
    const uint32_t n_items = (uint32_t)(tab[n_clips - 1].first_pair + (tab[n_clips - 1].n_frames + 1) / 2);
    ragged_pairs_kernel<<<(unsigned)((n_clips + 256) / 256), 256, 0, st>>>(tab_dev, n_clips, ws.rpairs);
    DSPX_CUDA_CHECK(cudaGetLastError());
    if (ws.peaks) {
        pcm16_peak_kernel<<<(unsigned)n_clips, 256, 0, st>>>(static_cast<const int16_t *>(samples), 0, 0, ws.peaks, tab_dev);
        DSPX_CUDA_CHECK(cudaGetLastError());
    }
    if (fused) DSPX_CUDA_CHECK(cudaMemsetAsync(ws.eacc, 0, (size_t)n_clips * 2 * C * sizeof(long long), st));
    float *mf = mfcc ? mfcc : ws.mfcc;                      // ws.mfcc: scratch for embeddings that are not fused, else null
    W8Params p = w8_batch_params(pl, samples, n_clips, 0, 0, logmel, mf, 0);
    p.rtab = tab_dev;
    p.rpairs = ws.rpairs;
    p.n_items = n_items;
    p.eacc = ws.eacc;
    p.peaks = ws.peaks;
    int rc = launch_warp8(pl, path, p, pl->cfg.pre_emphasis > 0.0, st);
    if (rc != DSPX_OK) return rc;
    if (fused) {
        const int64_t total = n_clips * C;
        embed_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(ws.eacc, n_clips, 1, C, embed, tab_dev);
        DSPX_CUDA_CHECK(cudaGetLastError());
        return DSPX_OK;
    }
    return embed ? launch_embed(mf, n_clips, 1, C, embed, st, tab_dev) : DSPX_OK;
}

static int ensure_pipe(dspx_plan *pl, size_t in_bytes, size_t out_bytes, bool stage_in, bool stage_out, HostPipe **out,
                       size_t f32_bytes = 0)
{
    // the HostPipe object itself is created with the plan; its streams and buffers are (re)sized here, with
    // hp->mu held by the caller for the whole pipelined call
    auto *hp = static_cast<HostPipe *>(pl->host_pipe);
    if (!hp) { set_error("plan has no host pipeline state"); return DSPX_EINVAL; }
    for (int i = 0; i < PIPE_SLOTS; i++) {
        if (!hp->stream[i]) DSPX_CUDA_CHECK(cudaStreamCreateWithFlags(&hp->stream[i], cudaStreamNonBlocking));
    }
    if (in_bytes > hp->in_bytes) {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (hp->d_in[i]) cudaFree(hp->d_in[i]);
            hp->d_in[i] = nullptr;
            DSPX_CUDA_CHECK(cudaMalloc(&hp->d_in[i], in_bytes));
        }
        hp->in_bytes = in_bytes;
    }
    if (out_bytes > hp->out_bytes) {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (hp->d_out[i]) cudaFree(hp->d_out[i]);
            hp->d_out[i] = nullptr;
            DSPX_CUDA_CHECK(cudaMalloc(&hp->d_out[i], out_bytes));
        }
        hp->out_bytes = out_bytes;
    }
    if (f32_bytes > hp->f32_bytes) {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (hp->d_f32[i]) cudaFree(hp->d_f32[i]);
            hp->d_f32[i] = nullptr;
            DSPX_CUDA_CHECK(cudaMalloc(&hp->d_f32[i], f32_bytes));
        }
        hp->f32_bytes = f32_bytes;
    }
    if (stage_in && in_bytes > hp->hin_bytes) {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (hp->h_in[i]) cudaFreeHost(hp->h_in[i]);
            hp->h_in[i] = nullptr;
            DSPX_CUDA_CHECK(cudaMallocHost(&hp->h_in[i], in_bytes));
        }
        hp->hin_bytes = in_bytes;
    }
    if (stage_out && out_bytes > hp->hout_bytes) {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (hp->h_out[i]) cudaFreeHost(hp->h_out[i]);
            hp->h_out[i] = nullptr;
            DSPX_CUDA_CHECK(cudaMallocHost(&hp->h_out[i], out_bytes));
        }
        hp->hout_bytes = out_bytes;
    }
    *out = hp;
    return DSPX_OK;
}

// Pageable callers: rows are copied into (or out of) pinned staging by a few host threads -- one thread
// tops out near 8 GB/s, far below what the PCIe link takes.
static void parallel_rows_copy(char *dst, size_t dst_stride, const char *src, size_t src_stride, size_t row_bytes,
                               int64_t rows)
{
    const size_t total = row_bytes * (size_t)rows;
    unsigned hw = std::thread::hardware_concurrency();
    int nt = hw >= 16 ? 8 : (hw >= 8 ? 4 : (hw >= 4 ? 2 : 1));
    if (total < (8u << 20) || rows < nt) nt = 1;
    auto work = [&](int64_t r0, int64_t r1) {
        if (dst_stride == row_bytes && src_stride == row_bytes) {
            memcpy(dst + (size_t)r0 * row_bytes, src + (size_t)r0 * row_bytes, (size_t)(r1 - r0) * row_bytes);
            return;
        }
        for (int64_t r = r0; r < r1; r++) memcpy(dst + (size_t)r * dst_stride, src + (size_t)r * src_stride, row_bytes);
    };
    if (nt == 1) { work(0, rows); return; }
    std::vector<std::thread> pool;
    for (int t = 0; t < nt; t++) {
        const int64_t r0 = rows * t / nt, r1 = rows * (t + 1) / nt;
        if (r1 > r0) pool.emplace_back(work, r0, r1);
    }
    for (auto &th : pool) th.join();
}

static bool is_pinned(const void *p)
{
    if (!p) return true;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// Chunked host pipeline shared by dspx_features_host and dspx_stft_host.
// mode 0: features (logmel/mfcc/embed), mode 1: stft (complex out in `o_stft`).
// elem = 4: float32 clips; elem = 2: PCM16 clips converted (and optionally peak-normalised) on the device.
static int host_pipeline(dspx_plan *pl, int mode, const void *clips_v, int64_t n_clips, int64_t clip_len,
                         int64_t clip_stride, int pre, float *o_logmel, float *o_mfcc, float *o_embed, float *o_stft,
                         int elem = 4, int normalize = 0)
{
    const char *clips = static_cast<const char *>(clips_v);
    const int64_t T = dspx_num_frames(pl, clip_len);
    if (T < 0) return DSPX_EINVAL;
    DSPX_REQUIRE(clips && n_clips >= 0 && clip_stride >= clip_len, "bad clip buffer arguments");
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(pl->device);
    if (!guard.ok) { set_error("cudaSetDevice(%d) failed", pl->device); return DSPX_ECUDA; }
    const size_t clip_bytes = (size_t)clip_len * elem;
    const size_t lm_b = (mode == 0 && o_logmel) ? (size_t)T * pl->cfg.n_mels * 4 : 0;
    // chunk: ~48 MiB of input or ~96 MiB of output, whichever is hit first
    int64_t chunk = std::min<int64_t>(n_clips, (int64_t)((48u << 20) / (clip_bytes ? clip_bytes : 1)));
    if (chunk < 1) chunk = 1;
    // the kernels read a chunk's device copy: rows of clip_len samples in a cudaMalloc'd, so aligned, buffer (the null
    // pointer below)
    const int dtype = elem == 2 ? DSPX_DTYPE_PCM16 : DSPX_DTYPE_F32;
    // embeddings alone: accumulated inside the feature kernel when it can (16 bytes of scratch per coefficient instead
    // of an MFCC tensor); otherwise they are the statistics of the MFCCs that are written anyway
    const bool fused_embed = mode == 0 && o_embed && !o_mfcc &&
                             warp8_select(pl, nullptr, clip_len, dtype, false, chunk, T, W8_WANT_EMBED) != W8_UNSUPPORTED;
    const bool need_mfcc = mode == 0 && (o_mfcc || (o_embed && !fused_embed));
    const size_t mf_b = need_mfcc ? (size_t)T * pl->cfg.n_mfcc * 4 : (fused_embed ? (size_t)pl->cfg.n_mfcc * 16 : 0);
    const size_t em_b = (mode == 0 && o_embed) ? (size_t)2 * pl->cfg.n_mfcc * 4 : 0;
    const size_t st_b = mode == 1 ? (size_t)T * pl->n_bins * 8 : 0;
    const size_t out_per_clip = lm_b + mf_b + em_b + st_b;
    const int64_t chunk_o = (int64_t)((96u << 20) / (out_per_clip ? out_per_clip : 1));
    if (chunk_o < chunk) chunk = chunk_o;
    if (chunk < 1) chunk = 1;
    const bool in_pinned = is_pinned(clips);
    const bool out_pinned = is_pinned(o_logmel) && is_pinned(o_mfcc) && is_pinned(o_embed) && is_pinned(o_stft);
    const size_t off_mf = align256(lm_b * chunk), off_em = off_mf + align256(mf_b * chunk);
    const size_t off_st = off_em + align256(em_b * chunk);
    const size_t out_bytes = off_st + align256(st_b * chunk);
    // One pipelined call at a time per plan: the lock covers the (re)allocation of the staging buffers as well
    // as their use, so concurrent callers sharing a plan queue up here instead of freeing each other's slots.
    HostPipe *hp = static_cast<HostPipe *>(pl->host_pipe);
    DSPX_REQUIRE(hp, "plan has no host pipeline state");
    std::lock_guard<std::mutex> lock(hp->mu);
    // PCM16: the feature kernel converts in its own loads when it can (no float32 copy of the clips); the scratch
    // buffer then only holds one int per clip.  Otherwise pcm16_to_float_kernel converts first and needs the copy.
    const bool fused_pcm = elem == 2 && mode == 0 &&
                           warp8_select(pl, nullptr, clip_len, dtype, false, chunk, T, W8_WANT_FEATURES) != W8_UNSUPPORTED;
    int rc = ensure_pipe(pl, clip_bytes * chunk, out_bytes, !in_pinned, !out_pinned, &hp,
                         elem == 2 ? (fused_pcm ? (size_t)chunk * sizeof(int) : (size_t)clip_len * 4 * chunk) : 0);
    if (rc != DSPX_OK) return rc;
    // "_host" contract: nothing may still be reading the caller's input or writing the caller's output when
    // the call returns, also on the error paths below
    struct Quiesce {
        HostPipe *hp;
        ~Quiesce()
        {
            for (int i = 0; i < PIPE_SLOTS; i++)
                if (hp->stream[i]) cudaStreamSynchronize(hp->stream[i]);
        }
    } quiesce{hp};

    struct Pending { int64_t first = -1, count = 0; } pend[PIPE_SLOTS];
    auto drain = [&](int s) -> int {
        if (pend[s].first < 0) return DSPX_OK;
        DSPX_CUDA_CHECK(cudaStreamSynchronize(hp->stream[s]));
        if (!out_pinned) {
            const int64_t f = pend[s].first, c = pend[s].count;
            const char *h = static_cast<const char *>(hp->h_out[s]);
            if (lm_b) parallel_rows_copy((char *)(o_logmel + (size_t)f * (lm_b / 4)), lm_b, h, lm_b, lm_b, c);
            if (mf_b && o_mfcc) parallel_rows_copy((char *)(o_mfcc + (size_t)f * (mf_b / 4)), mf_b, h + off_mf, mf_b, mf_b, c);
            if (em_b) memcpy(o_embed + (size_t)f * (em_b / 4), h + off_em, em_b * c);
            if (st_b) parallel_rows_copy((char *)(o_stft + (size_t)f * (st_b / 4)), st_b, h + off_st, st_b, st_b, c);
        }
        pend[s].first = -1;
        return DSPX_OK;
    };

    int slot = 0;
    for (int64_t first = 0; first < n_clips; first += chunk, slot = (slot + 1) % PIPE_SLOTS) {
        const int64_t cnt = (n_clips - first) < chunk ? (n_clips - first) : chunk;
        if ((rc = drain(slot)) != DSPX_OK) return rc;
        cudaStream_t st = hp->stream[slot];
        void *d_raw = hp->d_in[slot];
        char *d_o = static_cast<char *>(hp->d_out[slot]);
        const char *src = clips + (size_t)first * clip_stride * elem;
        if (in_pinned) {
            DSPX_CUDA_CHECK(cudaMemcpy2DAsync(d_raw, clip_bytes, src, (size_t)clip_stride * elem, clip_bytes, (size_t)cnt,
                                              cudaMemcpyHostToDevice, st));
        } else {
            char *h = static_cast<char *>(hp->h_in[slot]);
            parallel_rows_copy(h, clip_bytes, src, (size_t)clip_stride * elem, clip_bytes, cnt);
            DSPX_CUDA_CHECK(cudaMemcpyAsync(d_raw, h, clip_bytes * cnt, cudaMemcpyHostToDevice, st));
        }
        float *d_clips = static_cast<float *>(d_raw);
        if (elem == 2 && !fused_pcm) {
            d_clips = static_cast<float *>(hp->d_f32[slot]);
            pcm16_to_float_kernel<<<(unsigned)cnt, 256, 0, st>>>(static_cast<const int16_t *>(d_raw), clip_len, clip_len,
                                                                 normalize, d_clips, clip_len);
            DSPX_CUDA_CHECK(cudaGetLastError());
        }
        float *d_lm = lm_b ? reinterpret_cast<float *>(d_o) : nullptr;
        float *d_mf = mf_b ? reinterpret_cast<float *>(d_o + off_mf) : nullptr;
        float *d_em = em_b ? reinterpret_cast<float *>(d_o + off_em) : nullptr;
        float *d_st = st_b ? reinterpret_cast<float *>(d_o + off_st) : nullptr;
        if (fused_pcm)
            rc = features_device_pcm16(pl, static_cast<const int16_t *>(d_raw), cnt, clip_len, clip_len, normalize, d_lm, d_mf,
                                       d_em, static_cast<int *>(hp->d_f32[slot]), st);
        else if (mode == 0)
            rc = fused_embed ? features_device(pl, d_clips, cnt, clip_len, clip_len, d_lm, nullptr, d_em, st, 0,
                                               reinterpret_cast<long long *>(d_mf))
                             : features_device(pl, d_clips, cnt, clip_len, clip_len, d_lm, d_mf, d_em, st);
        else
            rc = stft_device(pl, d_clips, cnt, clip_len, clip_len, T, pre, reinterpret_cast<float2 *>(d_st), st);
        if (rc != DSPX_OK) return rc;
        char *h_o = out_pinned ? nullptr : static_cast<char *>(hp->h_out[slot]);
        auto d2h = [&](float *user, size_t per, size_t off, const void *dsrc) -> int {
            if (!per || !dsrc) return DSPX_OK;
            void *dst = out_pinned ? (void *)(user + (size_t)first * (per / 4)) : (void *)(h_o + off);
            DSPX_CUDA_CHECK(cudaMemcpyAsync(dst, dsrc, per * cnt, cudaMemcpyDeviceToHost, st));
            return DSPX_OK;
        };
        if ((rc = d2h(o_logmel, lm_b, 0, d_lm)) != DSPX_OK) return rc;
        if (o_mfcc && (rc = d2h(o_mfcc, mf_b, off_mf, d_mf)) != DSPX_OK) return rc;
        if ((rc = d2h(o_embed, em_b, off_em, d_em)) != DSPX_OK) return rc;
        if ((rc = d2h(o_stft, st_b, off_st, d_st)) != DSPX_OK) return rc;
        pend[slot].first = first;
        pend[slot].count = cnt;
    }
    for (int s = 0; s < PIPE_SLOTS; s++)
        if ((rc = drain(s)) != DSPX_OK) return rc;
    return DSPX_OK;
}

}  // namespace dspx

using namespace dspx;

// ======================================================================== C ABI
extern "C" {

const char *dspx_version(void) { return "dspx 0.1 (sm_100a)"; }
const char *dspx_last_error(void) { return get_error(); }

int dspx_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int64_t dspx_next_pow_two(int64_t n) { return n <= 1 ? 1 : next_pow_two(n); }

int dspx_plan_create(const dspx_config *cfg, int device, dspx_plan **out)
{
    DSPX_REQUIRE(cfg && out, "null argument");
    *out = nullptr;
    DSPX_REQUIRE(cfg->frame_length > 0 && cfg->hop_length > 0, "frame_length and hop_length must be positive");
    DSPX_REQUIRE(cfg->sample_rate > 0 && cfg->n_mels > 0 && cfg->n_mfcc > 0, "sample_rate, n_mels, n_mfcc must be positive");
    DSPX_REQUIRE(cfg->n_fft >= 0, "n_fft must be >= 0 (0 = frame_length)");
    DSPX_REQUIRE(cfg->window >= DSPX_WINDOW_HANN && cfg->window <= DSPX_WINDOW_RECT, "Unsupported window: %d", cfg->window);
    const int ndev = dspx_device_count();
    if (ndev <= 0) { set_error("no CUDA device: libdspx has no CPU fallback"); return DSPX_ENODEVICE; }
    DSPX_REQUIRE(device >= 0 && device < ndev, "device %d out of range (%d devices)", device, ndev);

    dspx_plan *p = new (std::nothrow) dspx_plan();
    if (!p) { set_error("out of host memory"); return DSPX_ENOMEM; }
    p->cfg = *cfg;
    p->device = device;
    p->host_pipe = new (std::nothrow) HostPipe();
    if (!p->host_pipe) { set_error("out of host memory"); delete p; return DSPX_ENOMEM; }
    const int nfft_raw = cfg->n_fft > 0 ? cfg->n_fft : cfg->frame_length;
    const int64_t P = next_pow_two(nfft_raw);
    if (P < 16 || P > 8192) {
        set_error("transform length %lld unsupported (power of two in [16, 8192])", (long long)P);
        plan_free_device(p);
        delete p;
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

    build_window(cfg->window, cfg->frame_length, p->host.window);
    const double f_max = cfg->f_max < 0.0 ? (double)cfg->sample_rate / 2.0 : cfg->f_max;
    build_filterbank(cfg->n_mels, p->P, cfg->sample_rate, cfg->f_min, f_max, p->host);
    build_dct2(cfg->n_mfcc, cfg->n_mels, p->host.dct2);

    DeviceGuard guard(device);
    if (!guard.ok) { set_error("cudaSetDevice(%d) failed", device); plan_free_device(p); delete p; return DSPX_ECUDA; }
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { set_error("cudaGetDeviceProperties failed"); plan_free_device(p); delete p; return DSPX_ECUDA; }
    p->sm_count = prop.multiProcessorCount;

    std::vector<float> w32(p->host.window.begin(), p->host.window.end());
    std::vector<float> d32(p->host.dct2.begin(), p->host.dct2.end());
    std::vector<float2> tw(p->P);
    for (int j = 0; j < p->P; j++) {
        const double a = -2.0 * M_PI * (double)j / (double)p->P;
        tw[j] = make_float2((float)std::cos(a), (float)std::sin(a));
    }
    int rc = DSPX_OK;
    if (rc == DSPX_OK) rc = upload(w32, &p->d_window);
    if (rc == DSPX_OK) rc = upload(tw, &p->d_tw);
    if (rc == DSPX_OK) rc = upload(p->host.fb_start, &p->d_fb_start);
    if (rc == DSPX_OK) rc = upload(p->host.fb_cnt, &p->d_fb_cnt);
    if (rc == DSPX_OK) rc = upload(p->host.fb_off, &p->d_fb_off);
    if (rc == DSPX_OK) rc = upload(p->host.fb_w, &p->d_fb_w);
    if (rc == DSPX_OK) rc = upload(d32, &p->d_dct2);
    if (rc == DSPX_OK) rc = upload(p->host.bin_filt, &p->d_bin_filt);
    if (rc == DSPX_OK) rc = upload(p->host.bin_wfall, &p->d_bin_wfall);
    if (rc == DSPX_OK) rc = upload(p->host.bin_wrise, &p->d_bin_wrise);

    p->kernel = DSPX_KERNEL_GENERIC;
    if (rc == DSPX_OK && cfg->kernel != DSPX_KERNEL_GENERIC) {
        const bool ok = warp8_supported(p);
        if (cfg->kernel == DSPX_KERNEL_WARP8 && !ok) {
            set_error("warp8 kernel does not support this configuration");
            rc = DSPX_EUNSUPPORTED;
        } else if (ok) {
            rc = warp8_prepare(p);
            if (rc == DSPX_OK) p->kernel = DSPX_KERNEL_WARP8;
        }
    }
    if (rc != DSPX_OK) {
        plan_free_device(p);
        delete p;
        return rc;
    }
    *out = p;
    return DSPX_OK;
}

int dspx_plan_destroy(dspx_plan *plan)
{
    if (!plan) return DSPX_OK;
    DeviceGuard guard(plan->device);
    plan_free_device(plan);
    delete plan;
    return DSPX_OK;
}

int dspx_plan_get_info(const dspx_plan *plan, dspx_plan_info *out)
{
    DSPX_REQUIRE(plan && out, "null argument");
    out->n_fft_pow2 = plan->P;
    out->n_bins = plan->n_bins;
    out->take_features = plan->take_feat;
    out->take_stft = plan->take_stft;
    out->mel_nnz = (int32_t)plan->host.fb_w.size();
    out->kernel = plan->kernel;
    out->device = plan->device;
    out->sm_count = plan->sm_count;
    return DSPX_OK;
}

int64_t dspx_num_frames(const dspx_plan *plan, int64_t clip_len)
{
    if (!plan) { set_error("null plan"); return DSPX_EINVAL; }
    if (clip_len < plan->cfg.frame_length) {
        set_error("signal of %lld samples is shorter than one frame (%d)", (long long)clip_len, plan->cfg.frame_length);
        return DSPX_EINVAL;
    }
    return 1 + (clip_len - plan->cfg.frame_length) / plan->cfg.hop_length;
}

int dspx_plan_read_table(const dspx_plan *plan, int which, float *out_host, int64_t capacity)
{
    DSPX_REQUIRE(plan && out_host, "null argument");
    DeviceGuard guard(plan->device);
    if (which == 0) {
        DSPX_REQUIRE(capacity >= plan->cfg.frame_length, "capacity too small");
        DSPX_CUDA_CHECK(cudaMemcpy(out_host, plan->d_window, (size_t)plan->cfg.frame_length * 4, cudaMemcpyDeviceToHost));
    } else if (which == 1) {
        // rebuild the dense table from the sparse rows that the kernels actually read
        const int64_t n = (int64_t)plan->cfg.n_mels * plan->n_bins;
        DSPX_REQUIRE(capacity >= n, "capacity too small");
        std::vector<float> w(plan->host.fb_w.size());
        if (!w.empty()) DSPX_CUDA_CHECK(cudaMemcpy(w.data(), plan->d_fb_w, w.size() * 4, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < n; i++) out_host[i] = 0.f;
        for (int m = 0; m < plan->cfg.n_mels; m++)
            for (int q = 0; q < plan->host.fb_cnt[m]; q++)
                out_host[(size_t)m * plan->n_bins + plan->host.fb_start[m] + q] = w[plan->host.fb_off[m] + q];
    } else if (which == 2) {
        const int64_t n = (int64_t)plan->cfg.n_mfcc * plan->cfg.n_mels;
        DSPX_REQUIRE(capacity >= n, "capacity too small");
        DSPX_CUDA_CHECK(cudaMemcpy(out_host, plan->d_dct2, (size_t)n * 4, cudaMemcpyDeviceToHost));
    } else {
        DSPX_REQUIRE(false, "unknown table %d", which);
    }
    return DSPX_OK;
}

int dspx_stft(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len, int64_t clip_stride,
              int pre_emphasis, float *out_dev, void *stream)
{
    DSPX_REQUIRE(plan && clips_dev && out_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && clip_stride >= clip_len, "bad clip buffer arguments");
    const int64_t T = dspx_num_frames(plan, clip_len);
    if (T < 0) return DSPX_EINVAL;
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(plan->device);
    const int pre = (pre_emphasis && plan->cfg.pre_emphasis > 0.0) ? 1 : 0;
    return stft_device(plan, clips_dev, n_clips, clip_len, clip_stride, T, pre, reinterpret_cast<float2 *>(out_dev),
                       static_cast<cudaStream_t>(stream));
}

int dspx_features(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len, int64_t clip_stride,
                  float *logmel_out_dev, float *mfcc_out_dev, float *embed_out_dev, void *stream)
{
    DSPX_REQUIRE(plan && clips_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && clip_stride >= clip_len, "bad clip buffer arguments");
    DSPX_REQUIRE(logmel_out_dev || mfcc_out_dev, "no output requested");
    DSPX_REQUIRE(!embed_out_dev || mfcc_out_dev, "embed_out_dev needs mfcc_out_dev");
    if (dspx_num_frames(plan, clip_len) < 0) return DSPX_EINVAL;
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(plan->device);
    return features_device(plan, clips_dev, n_clips, clip_len, clip_stride, logmel_out_dev, mfcc_out_dev, embed_out_dev,
                           static_cast<cudaStream_t>(stream));
}

size_t dspx_embeddings_workspace(const dspx_plan *plan, int64_t n_clips)
{
    if (!plan || n_clips < 0) return 0;
    return (size_t)n_clips * 2 * plan->cfg.n_mfcc * sizeof(long long) + 256;
}

int dspx_embeddings(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len, int64_t clip_stride,
                    float *embed_out_dev, float *logmel_out_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(plan && clips_dev && embed_out_dev && workspace_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && clip_stride >= clip_len, "bad clip buffer arguments");
    DSPX_REQUIRE(workspace_bytes >= dspx_embeddings_workspace(plan, n_clips), "workspace too small");
    if (dspx_num_frames(plan, clip_len) < 0) return DSPX_EINVAL;
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(plan->device);
    char *ws = static_cast<char *>(workspace_dev);
    ws += (256 - (reinterpret_cast<uintptr_t>(ws) & 255)) & 255;
    return features_device(plan, clips_dev, n_clips, clip_len, clip_stride, logmel_out_dev, nullptr, embed_out_dev,
                           static_cast<cudaStream_t>(stream), 0, reinterpret_cast<long long *>(ws));
}

int dspx_log_mel_nchw(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len,
                      int64_t clip_stride, float *out_dev, void *stream)
{
    DSPX_REQUIRE(plan && clips_dev && out_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && clip_stride >= clip_len, "bad clip buffer arguments");
    if (dspx_num_frames(plan, clip_len) < 0) return DSPX_EINVAL;
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(plan->device);
    return features_device(plan, clips_dev, n_clips, clip_len, clip_stride, out_dev, nullptr, nullptr,
                           static_cast<cudaStream_t>(stream), 1);
}

int dspx_embed_stats(const float *feats_dev, int64_t n_clips, int64_t n_frames, int n_coef, float *out_dev, void *stream)
{
    DSPX_REQUIRE(feats_dev && out_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && n_frames > 0 && n_coef > 0, "bad shape");
    if (n_clips == 0) return DSPX_OK;
    return launch_embed(feats_dev, n_clips, n_frames, n_coef, out_dev, static_cast<cudaStream_t>(stream));
}

int64_t dspx_ragged_layout(const dspx_config *cfg, const int64_t *starts, const int64_t *lengths, int64_t n_clips,
                           int dtype, dspx_ragged_clip *table_out)
{
    DSPX_REQUIRE(cfg && (n_clips == 0 || (starts && lengths && table_out)), "null argument");
    DSPX_REQUIRE(n_clips >= 0, "negative clip count");
    DSPX_REQUIRE(cfg->frame_length > 0 && cfg->hop_length > 0, "frame_length and hop_length must be positive");
    DSPX_REQUIRE(dtype == DSPX_DTYPE_F32 || dtype == DSPX_DTYPE_PCM16, "ragged batches take float32 or PCM16 samples");
    int64_t frames = 0, pairs = 0;
    for (int64_t i = 0; i < n_clips; i++) {
        DSPX_REQUIRE(lengths[i] >= cfg->frame_length, "clip %lld: %lld samples is shorter than one frame (%d)", (long long)i,
                     (long long)lengths[i], cfg->frame_length);
        DSPX_REQUIRE(starts[i] >= 0, "clip %lld: negative start %lld", (long long)i, (long long)starts[i]);
        DSPX_REQUIRE(dtype != DSPX_DTYPE_F32 || !(starts[i] & 1),
                     "clip %lld: float32 clips must start at an even sample (start %lld)", (long long)i, (long long)starts[i]);
        dspx_ragged_clip &r = table_out[i];
        r.start = starts[i];
        r.length = lengths[i];
        r.n_frames = 1 + (lengths[i] - cfg->frame_length) / cfg->hop_length;
        r.first_frame = frames;
        r.first_pair = pairs;
        frames += r.n_frames;
        pairs += (r.n_frames + 1) / 2;
        DSPX_REQUIRE(pairs < (int64_t)0x7fffffff, "ragged batch of 2^31 frame pairs or more (clip %lld)", (long long)i);
    }
    return frames;
}

size_t dspx_features_ragged_workspace(const dspx_plan *plan, const dspx_ragged_clip *table_host, int64_t n_clips,
                                      int dtype, int normalize, int want_logmel, int want_mfcc, int want_embed)
{
    (void)want_logmel;
    if (!plan || n_clips < 0 || (n_clips > 0 && !table_host)) return 0;
    return ragged_ws_carve(plan, table_host, n_clips, dtype, normalize, want_mfcc != 0, want_embed != 0, nullptr, nullptr);
}

int dspx_features_ragged(const dspx_plan *plan, const void *samples_dev, int dtype, int normalize,
                         const dspx_ragged_clip *table_dev, const dspx_ragged_clip *table_host, int64_t n_clips,
                         int64_t total_frames, float *logmel_out_dev, float *mfcc_out_dev, float *embed_out_dev,
                         void *workspace_dev, size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(plan, "null plan");
    DSPX_REQUIRE(dtype == DSPX_DTYPE_F32 || dtype == DSPX_DTYPE_PCM16, "ragged batches take float32 or PCM16 samples");
    DSPX_REQUIRE(n_clips >= 0, "negative clip count");
    if (n_clips == 0) return DSPX_OK;
    DSPX_REQUIRE(samples_dev && table_dev && table_host, "null argument");
    DSPX_REQUIRE(dtype != DSPX_DTYPE_F32 || !(reinterpret_cast<uintptr_t>(samples_dev) & 7),
                 "float32 samples must be 8-byte aligned");
    DSPX_REQUIRE(n_clips < (int64_t)2147483647, "too many clips for one launch");
    const dspx_ragged_clip &last = table_host[n_clips - 1];
    DSPX_REQUIRE(last.first_frame + last.n_frames == total_frames, "total_frames %lld does not match the table (%lld)",
                 (long long)total_frames, (long long)(last.first_frame + last.n_frames));
    DSPX_REQUIRE(last.first_pair + (last.n_frames + 1) / 2 < (int64_t)0x7fffffff, "ragged batch of 2^31 frame pairs or more");
    for (int64_t i = 0; i < n_clips; i++)
        DSPX_REQUIRE(table_host[i].length >= plan->cfg.frame_length, "clip %lld: %lld samples is shorter than one frame (%d)",
                     (long long)i, (long long)table_host[i].length, plan->cfg.frame_length);
    const size_t need = dspx_features_ragged_workspace(plan, table_host, n_clips, dtype, normalize, logmel_out_dev != nullptr,
                                                       mfcc_out_dev != nullptr, embed_out_dev != nullptr);
    DSPX_REQUIRE(workspace_dev && workspace_bytes >= need, "workspace too small (%zu bytes needed)", need);
    if (!logmel_out_dev && !mfcc_out_dev && !embed_out_dev) return DSPX_OK;
    DeviceGuard guard(plan->device);
    char *ws = static_cast<char *>(workspace_dev);
    ws += (256 - (reinterpret_cast<uintptr_t>(ws) & 255)) & 255;
    return features_ragged(plan, samples_dev, dtype, normalize ? 1 : 0, table_dev, table_host, n_clips, logmel_out_dev,
                           mfcc_out_dev, embed_out_dev, ws, static_cast<cudaStream_t>(stream));
}

int dspx_embed_stats_ragged(const float *feats_dev, const dspx_ragged_clip *table_dev, int64_t n_clips, int n_coef,
                            float *out_dev, void *stream)
{
    DSPX_REQUIRE(n_clips >= 0 && n_coef > 0, "bad shape");
    if (n_clips == 0) return DSPX_OK;
    DSPX_REQUIRE(feats_dev && table_dev && out_dev, "null argument");
    return launch_embed(feats_dev, n_clips, 1, n_coef, out_dev, static_cast<cudaStream_t>(stream), table_dev);
}

int dspx_cmvn(float *feats_dev, int64_t n_clips, int64_t n_frames, int n_coef, double eps, void *stream)
{
    DSPX_REQUIRE(feats_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && n_frames > 0 && n_coef > 0 && eps >= 0.0, "bad shape");
    DSPX_REQUIRE(n_clips < (int64_t)2147483647, "too many clips for one launch");
    if (n_clips == 0) return DSPX_OK;
    const int cw = n_coef < 128 ? n_coef : 128;
    const size_t smem = ((size_t)(128 / cw) * n_coef + 2 * (size_t)n_coef) * sizeof(double);
    DSPX_REQUIRE(smem <= 48 * 1024, "n_coef %d too large for cmvn", n_coef);
    cmvn_kernel<<<(unsigned)n_clips, 128, smem, static_cast<cudaStream_t>(stream)>>>(feats_dev, n_frames, n_coef, eps);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

int dspx_features_host(const dspx_plan *plan, const float *clips_host, int64_t n_clips, int64_t clip_len,
                       int64_t clip_stride, float *logmel_out_host, float *mfcc_out_host, float *embed_out_host)
{
    DSPX_REQUIRE(plan, "null plan");
    DSPX_REQUIRE(logmel_out_host || mfcc_out_host || embed_out_host, "no output requested");
    return host_pipeline(const_cast<dspx_plan *>(plan), 0, clips_host, n_clips, clip_len, clip_stride, 0,
                         logmel_out_host, mfcc_out_host, embed_out_host, nullptr);
}

int dspx_pcm16_to_float(const int16_t *pcm_dev, int64_t n_clips, int64_t clip_len, int64_t pcm_stride, int normalize,
                        float *out_dev, int64_t out_stride, void *stream)
{
    DSPX_REQUIRE(pcm_dev && out_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && clip_len > 0 && pcm_stride >= clip_len && out_stride >= clip_len, "bad clip buffer arguments");
    DSPX_REQUIRE(n_clips < (int64_t)2147483647, "too many clips for one launch");
    if (n_clips == 0) return DSPX_OK;
    pcm16_to_float_kernel<<<(unsigned)n_clips, 256, 0, static_cast<cudaStream_t>(stream)>>>(pcm_dev, clip_len, pcm_stride,
                                                                                            normalize ? 1 : 0, out_dev, out_stride);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

size_t dspx_features_pcm16_workspace(int64_t n_clips) { return n_clips > 0 ? (size_t)n_clips * sizeof(int) + 256 : 256; }

int dspx_features_pcm16(const dspx_plan *plan, const int16_t *pcm_dev, int64_t n_clips, int64_t clip_len, int64_t pcm_stride,
                        int normalize, float *logmel_out_dev, float *mfcc_out_dev, float *embed_out_dev, void *workspace_dev,
                        size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(plan && pcm_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && clip_len > 0 && pcm_stride >= clip_len, "bad clip buffer arguments");
    DSPX_REQUIRE(logmel_out_dev || mfcc_out_dev, "no output requested");
    DSPX_REQUIRE(!normalize || (workspace_dev && workspace_bytes >= dspx_features_pcm16_workspace(n_clips)), "workspace too small");
    if (dspx_num_frames(plan, clip_len) < 0) return DSPX_EINVAL;
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(plan->device);
    char *ws = static_cast<char *>(workspace_dev);
    if (ws) ws += (256 - (reinterpret_cast<uintptr_t>(ws) & 255)) & 255;
    return features_device_pcm16(plan, pcm_dev, n_clips, clip_len, pcm_stride, normalize ? 1 : 0, logmel_out_dev, mfcc_out_dev,
                                 embed_out_dev, reinterpret_cast<int *>(ws), static_cast<cudaStream_t>(stream));
}

int dspx_features_host_pcm16(const dspx_plan *plan, const int16_t *pcm_host, int64_t n_clips, int64_t clip_len,
                             int64_t pcm_stride, int normalize, float *logmel_out_host, float *mfcc_out_host,
                             float *embed_out_host)
{
    DSPX_REQUIRE(plan, "null plan");
    DSPX_REQUIRE(logmel_out_host || mfcc_out_host || embed_out_host, "no output requested");
    return host_pipeline(const_cast<dspx_plan *>(plan), 0, pcm_host, n_clips, clip_len, pcm_stride, 0, logmel_out_host,
                         mfcc_out_host, embed_out_host, nullptr, 2, normalize ? 1 : 0);
}

int dspx_stft_host(const dspx_plan *plan, const float *clips_host, int64_t n_clips, int64_t clip_len, int64_t clip_stride,
                   int pre_emphasis, float *out_host)
{
    DSPX_REQUIRE(plan && out_host, "null argument");
    const int pre = (pre_emphasis && plan->cfg.pre_emphasis > 0.0) ? 1 : 0;
    return host_pipeline(const_cast<dspx_plan *>(plan), 1, clips_host, n_clips, clip_len, clip_stride, pre, nullptr,
                         nullptr, nullptr, out_host);
}

int dspx_fft_c2c(const float *in_dev, int64_t batch, int64_t n_in, int64_t n, int inverse, float *out_dev,
                 float *work_dev, void *stream)
{
    DSPX_REQUIRE(in_dev && out_dev, "null argument");
    DSPX_REQUIRE(batch >= 0 && n_in >= 0 && n >= 1, "bad fft shape");
    if (batch == 0) return DSPX_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t P = next_pow_two(n);
    const int64_t n_valid = n_in < n ? n_in : n;
    const float2 *in = reinterpret_cast<const float2 *>(in_dev);
    float2 *out = reinterpret_cast<float2 *>(out_dev);
    float2 *work = reinterpret_cast<float2 *>(work_dev);
    if (P == 1) {
        fft_copy1_kernel<<<(unsigned)((batch + 255) / 256), 256, 0, st>>>(in, out, batch, n_in, n_valid);
        DSPX_CUDA_CHECK(cudaGetLastError());
        return DSPX_OK;
    }
    int radix[64], ns_count = 0;
    for (int64_t m = P; m > 1;) {
        if (m % 4 == 0) { radix[ns_count++] = 4; m /= 4; }
        else { radix[ns_count++] = 2; m /= 2; }
    }
    DSPX_REQUIRE(ns_count == 1 || work_dev, "work_dev required for transforms longer than 4");
    int64_t ns = 1;
    const float2 *src = in;
    for (int s = 0; s < ns_count; s++) {
        FftStage fs{};
        fs.in = src;
        fs.out = ((ns_count - 1 - s) % 2 == 0) ? out : work;
        fs.batch = batch;
        fs.in_stride = s == 0 ? n_in : P;
        fs.n_valid = n_valid;
        fs.P = P;
        fs.ns = ns;
        fs.R = radix[s];
        fs.inverse = inverse ? 1 : 0;
        fs.first = s == 0;
        fs.last = s == ns_count - 1;
        const int64_t total = batch * (P / fs.R);
        int64_t blocks = (total + 255) / 256;
        if (blocks > 148 * 32) blocks = 148 * 32;
        fft_stage_kernel<<<(unsigned)blocks, 256, 0, st>>>(fs);
        DSPX_CUDA_CHECK(cudaGetLastError());
        src = fs.out;
        ns *= fs.R;
    }
    return DSPX_OK;
}

// Tuning / test knobs of the ranking path, read from the environment once per process (never in the launch
// path): DSPX_TOPK = tc | f32 | f64 forces a kernel, DSPX_TOPK_SPLITS fixes the database split count.
struct TopkKnobs {
    const char *force;
    bool f64;
    long long splits;
};
static const TopkKnobs &topk_knobs()
{
    static const TopkKnobs k = [] {
        TopkKnobs t{};
        t.force = getenv("DSPX_TOPK");
        t.f64 = getenv("DSPX_TOPK_F64") != nullptr;
        const char *e = getenv("DSPX_TOPK_SPLITS");
        t.splits = e ? atoll(e) : 0;
        return t;
    }();
    return k;
}

static int topk_splits(int64_t nq, int64_t ndb, int sm_count)
{
    const int64_t qtiles = (nq + TK_QPC - 1) / TK_QPC;
    int64_t s = (2 * (int64_t)sm_count + qtiles - 1) / qtiles;
    const int64_t max_by_rows = (ndb + 4 * TK_ROWS - 1) / (4 * TK_ROWS);       // at least 4 tiles per split
    if (s > max_by_rows) s = max_by_rows;
    if (s > TK_MAX_SPLITS) s = TK_MAX_SPLITS;
    if (s < 1) s = 1;
    return (int)s;
}

size_t dspx_cosine_topk_workspace(int64_t nq, int64_t ndb, int dim, int k)
{
    if (nq < 0 || ndb < 0 || dim <= 0 || k <= 0) return 0;
    size_t b = align256((size_t)nq * dim * 8) + align256((size_t)ndb * dim * 8);
    b += align256((size_t)nq * TK_MAX_SPLITS * k * 8) + align256((size_t)nq * TK_MAX_SPLITS * k * 4);
    // float copies for the filter kernels: 32 floats per row covers both layouts (dim <= 32 there)
    b += align256((size_t)((nq + TC_QT - 1) / TC_QT) * TC_QT * TC_KPAD * 4);
    b += align256((size_t)((ndb + TK_ROWS - 1) / TK_ROWS) * TK_ROWS * TC_KPAD * 4);
    b += align256((size_t)nq * 8);                                                // thresholds shared between splits
    b += align256((size_t)((nq + TC_QT - 1) / TC_QT) * TK_MAX_SPLITS * 4);      // per (query tile, split): lists written
    return b + 1024;
}

int dspx_cosine_topk(const void *q_dev, int64_t nq, const void *db_dev, int64_t ndb, int dim, int dtype, int k,
                     int32_t *idx_out_dev, double *score_out_dev, void *workspace_dev, size_t workspace_bytes,
                     void *stream)
{
    DSPX_REQUIRE(q_dev && db_dev && idx_out_dev && workspace_dev, "null argument");
    DSPX_REQUIRE(nq >= 0 && ndb >= 1 && dim >= 1, "bad shape");
    DSPX_REQUIRE(k >= 1 && k <= DSPX_MAX_K && k <= ndb, "k must be in [1, min(%d, ndb)]", DSPX_MAX_K);
    DSPX_REQUIRE(dtype == DSPX_DTYPE_F32 || dtype == DSPX_DTYPE_F64, "bad dtype");
    DSPX_REQUIRE(ndb < (int64_t)2147483647, "database too large for int32 indices");
    DSPX_REQUIRE(workspace_bytes >= dspx_cosine_topk_workspace(nq, ndb, dim, k), "workspace too small");
    if (nq == 0) return DSPX_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int dev = 0, sm = 148;
    DSPX_CUDA_CHECK(cudaGetDevice(&dev));
    DSPX_CUDA_CHECK(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev));
    char *ws = static_cast<char *>(workspace_dev);
    double *qn = reinterpret_cast<double *>(ws);
    ws += align256((size_t)nq * dim * 8);
    double *dbn = reinterpret_cast<double *>(ws);
    ws += align256((size_t)ndb * dim * 8);
    double *pscore = reinterpret_cast<double *>(ws);
    ws += align256((size_t)nq * TK_MAX_SPLITS * k * 8);
    int32_t *pidx = reinterpret_cast<int32_t *>(ws);
    ws += align256((size_t)nq * TK_MAX_SPLITS * k * 4);
    float *qf_t = reinterpret_cast<float *>(ws);
    const size_t qf_bytes = (size_t)((nq + TC_QT - 1) / TC_QT) * TC_QT * TC_KPAD * 4;
    ws += align256(qf_bytes);
    float *dbf_t = reinterpret_cast<float *>(ws);
    const size_t dbf_bytes = (size_t)((ndb + TK_ROWS - 1) / TK_ROWS) * TK_ROWS * TC_KPAD * 4;
    ws += align256(dbf_bytes);
    unsigned long long *shared_thr = reinterpret_cast<unsigned long long *>(ws);
    ws += align256((size_t)nq * 8);
    int *split_done = reinterpret_cast<int *>(ws);
    // Filter kernels (single-chunk dimensions, lists that fit beside the tiles), all with exact float64 re-scoring:
    // tensor-core (split fp16) filter, else packed-FP32 filter, else the all-float64 kernel.  DSPX_TOPK = tc | f32 | f64 forces one.
    const TopkKnobs &knobs = topk_knobs();
    const char *force = knobs.force;
    const bool want_f64 = knobs.f64 || (force && !strcmp(force, "f64"));
    const bool tc_ok = dim <= 32 && k <= TC_MAX_K;
    const bool f32_ok = dim <= 32 && topk_f32_smem_bytes(dim, k, dim == 26 ? 26 : 32) <= 200 * 1024;
    const bool use_tc = !want_f64 && tc_ok && !(force && !strcmp(force, "f32") && f32_ok);
    const bool prefilter = !want_f64 && !use_tc && f32_ok;

    if (use_tc) {
        // fp16 operand images (128 bytes per row, same size as the float copies of the other filter); the kernel writes the
        // zero padding too (columns >= dim, rows up to the tile multiple): no memset pass
        const int64_t nq_pad = (nq + TC_QT - 1) / TC_QT * TC_QT, ndb_pad = (ndb + TK_ROWS - 1) / TK_ROWS * TK_ROWS;
        const unsigned gq = (unsigned)((nq_pad + NR_ROWS - 1) / NR_ROWS), gd = (unsigned)((ndb_pad + NR_ROWS - 1) / NR_ROWS);
        if (dtype == DSPX_DTYPE_F32) {
            normalize_rows_split16_kernel<float><<<gq, 128, 0, st>>>((const float *)q_dev, nq, nq_pad, dim, qn, (unsigned char *)qf_t);
            normalize_rows_split16_kernel<float><<<gd, 128, 0, st>>>((const float *)db_dev, ndb, ndb_pad, dim, dbn, (unsigned char *)dbf_t);
        } else {
            normalize_rows_split16_kernel<double><<<gq, 128, 0, st>>>((const double *)q_dev, nq, nq_pad, dim, qn, (unsigned char *)qf_t);
            normalize_rows_split16_kernel<double><<<gd, 128, 0, st>>>((const double *)db_dev, ndb, ndb_pad, dim, dbn, (unsigned char *)dbf_t);
        }
    } else
    if (prefilter) {
        DSPX_CUDA_CHECK(cudaMemsetAsync(qf_t, 0, qf_bytes, st));              // zero padding of the last tiles
        DSPX_CUDA_CHECK(cudaMemsetAsync(dbf_t, 0, dbf_bytes, st));
        if (dtype == DSPX_DTYPE_F32) {
            normalize_rows_tiled_kernel<float><<<(unsigned)((nq + 127) / 128), 128, 0, st>>>((const float *)q_dev, nq, dim, qn, qf_t, TKF_QPC);
            normalize_rows_tiled_kernel<float><<<(unsigned)((ndb + 127) / 128), 128, 0, st>>>((const float *)db_dev, ndb, dim, dbn, dbf_t, TK_ROWS);
        } else {
            normalize_rows_tiled_kernel<double><<<(unsigned)((nq + 127) / 128), 128, 0, st>>>((const double *)q_dev, nq, dim, qn, qf_t, TKF_QPC);
            normalize_rows_tiled_kernel<double><<<(unsigned)((ndb + 127) / 128), 128, 0, st>>>((const double *)db_dev, ndb, dim, dbn, dbf_t, TK_ROWS);
        }
    } else if (dtype == DSPX_DTYPE_F32) {
        normalize_rows_kernel<float><<<(unsigned)((nq + 127) / 128), 128, 0, st>>>((const float *)q_dev, nq, dim, qn);
        normalize_rows_kernel<float><<<(unsigned)((ndb + 127) / 128), 128, 0, st>>>((const float *)db_dev, ndb, dim, dbn);
    } else {
        normalize_rows_kernel<double><<<(unsigned)((nq + 127) / 128), 128, 0, st>>>((const double *)q_dev, nq, dim, qn);
        normalize_rows_kernel<double><<<(unsigned)((ndb + 127) / 128), 128, 0, st>>>((const double *)db_dev, ndb, dim, dbn);
    }
    DSPX_CUDA_CHECK(cudaGetLastError());

    TopkParams tp{};
    tp.qn = qn;
    tp.dbn = dbn;
    tp.nq = nq;
    tp.ndb = ndb;
    tp.dim = dim;
    tp.k = k;
    tp.n_splits = topk_splits(nq, ndb, sm);
    int64_t rps = (ndb + tp.n_splits - 1) / tp.n_splits;
    rps = (rps + TK_ROWS - 1) / TK_ROWS * TK_ROWS;
    tp.rows_per_split = rps;
    tp.n_splits = (int)((ndb + rps - 1) / rps);
    tp.idx_out = tp.n_splits == 1 ? idx_out_dev : pidx;
    tp.score_out = tp.n_splits == 1 ? score_out_dev : pscore;
    dim3 grid((unsigned)((nq + TK_QPC - 1) / TK_QPC), (unsigned)tp.n_splits);
    if (use_tc || prefilter) {
        // one CTA per SM: pick the split count whose grid fills whole waves (every extra split also restarts
        // the running lists, which costs insertions -- the per-split penalty)
        const int64_t qtiles = use_tc ? (nq + TC_QT - 1) / TC_QT : (nq + TKF_QPC - 1) / TKF_QPC;
        int64_t max_sp = (ndb + 8 * TK_ROWS - 1) / (8 * TK_ROWS);
        if (max_sp > 16) max_sp = 16;
        if (max_sp < 1) max_sp = 1;
        int64_t sp = 1;
        double best = 1e30;
        for (int64_t c = 1; c <= max_sp; c++) {
            const double waves = (double)((qtiles * c + sm - 1) / sm);
            const double cost = waves / (double)c * (1.0 + 0.02 * (double)c);
            if (cost < best - 1e-12) { best = cost; sp = c; }
        }
        if (knobs.splits >= 1 && knobs.splits <= TK_MAX_SPLITS) sp = knobs.splits;      // tuning knob
        int64_t rows = (ndb + sp - 1) / sp;
        rows = (rows + TK_ROWS - 1) / TK_ROWS * TK_ROWS;
        tp.rows_per_split = rows;
        tp.n_splits = (int)((ndb + rows - 1) / rows);
        tp.idx_out = tp.n_splits == 1 ? idx_out_dev : pidx;
        tp.score_out = tp.n_splits == 1 ? score_out_dev : pscore;
        if (use_tc) {
            TopkTcParams cp{};
            cp.base = tp;
            cp.qx = reinterpret_cast<const unsigned char *>(qf_t);
            cp.dbx = reinterpret_cast<const unsigned char *>(dbf_t);
            cp.shared_thr = tp.n_splits > 1 ? shared_thr : nullptr;
            cp.done = tp.n_splits > 1 ? split_done : nullptr;
            if (cp.done) DSPX_CUDA_CHECK(cudaMemsetAsync(split_done, 0, (size_t)qtiles * tp.n_splits * 4, st));
#ifdef DSPX_TC_PROFILE                  // profiling builds only: DSPX_EXPERIMENT_KEEP_THR=1 keeps the thresholds of the previous call (steady-state per-role cycles)
            if (cp.shared_thr && !getenv("DSPX_EXPERIMENT_KEEP_THR"))
#else
            if (cp.shared_thr)
#endif
                DSPX_CUDA_CHECK(cudaMemsetAsync(shared_thr, 0, (size_t)nq * 8, st));
            dim3 cgrid((unsigned)qtiles, (unsigned)tp.n_splits);
            const size_t smem = topk_tc_smem_bytes(k);
            if (dim == 26) {
                { static std::atomic<unsigned char> optin[64]; DSPX_CUDA_CHECK(optin_max_smem(cosine_topk_tc_kernel<26>, optin, dev)); }
                cosine_topk_tc_kernel<26><<<cgrid, TC_THREADS, smem, st>>>(cp);
            } else {
                { static std::atomic<unsigned char> optin[64]; DSPX_CUDA_CHECK(optin_max_smem(cosine_topk_tc_kernel<0>, optin, dev)); }
                cosine_topk_tc_kernel<0><<<cgrid, TC_THREADS, smem, st>>>(cp);
            }
        } else {
        TopkF32Params fp{};
        fp.base = tp;
        fp.qf_t = qf_t;
        fp.dbf_t = dbf_t;
        fp.eps = 4e-6f + (float)dim * 1.2e-7f;         // > 2 * 2^-24 * (dim + 2): bound on |s32 - s64| for unit vectors
        dim3 fgrid((unsigned)qtiles, (unsigned)tp.n_splits);
        if (dim == 26) {
            const size_t smem = topk_f32_smem_bytes(dim, k, 26);
            { static std::atomic<unsigned char> optin[64]; DSPX_CUDA_CHECK(optin_max_smem(cosine_topk_f32_kernel<26>, optin, dev)); }
            cosine_topk_f32_kernel<26><<<fgrid, TKF_WARPS * 32, smem, st>>>(fp);
        } else {
            const size_t smem = topk_f32_smem_bytes(dim, k, 32);
            { static std::atomic<unsigned char> optin[64]; DSPX_CUDA_CHECK(optin_max_smem(cosine_topk_f32_kernel<32>, optin, dev)); }
            cosine_topk_f32_kernel<32><<<fgrid, TKF_WARPS * 32, smem, st>>>(fp);
        }
        }
    } else if (dim == 26) {                            // MFCC embeddings: 2 x 13, the whole vector in one chunk
        const size_t smem = topk_smem_bytes(dim, k, 26);
        { static std::atomic<unsigned char> optin[64]; DSPX_CUDA_CHECK(optin_max_smem(cosine_topk_kernel<26>, optin, dev)); }
        cosine_topk_kernel<26><<<grid, TK_WARPS * 32, smem, st>>>(tp);
    } else {
        const size_t smem = topk_smem_bytes(dim, k, 32);
        { static std::atomic<unsigned char> optin[64]; DSPX_CUDA_CHECK(optin_max_smem(cosine_topk_kernel<32>, optin, dev)); }
        cosine_topk_kernel<32><<<grid, TK_WARPS * 32, smem, st>>>(tp);
    }
    DSPX_CUDA_CHECK(cudaGetLastError());
    if (tp.n_splits > 1) {
        topk_merge_kernel<<<(unsigned)((nq + 3) / 4), 128, 0, st>>>(pidx, pscore, nq, tp.n_splits, k, idx_out_dev, score_out_dev);
        DSPX_CUDA_CHECK(cudaGetLastError());
    }
    return DSPX_OK;
}

#ifdef DSPX_TC_PROFILE
extern "C" int dspx_debug_tc_trace(long long *out)       // [32][18], see retrieval_tc.cuh
{
    return cudaMemcpyFromSymbol(out, dspx::tc_trace, 32 * 18 * sizeof(long long)) == cudaSuccess ? 0 : -1;
}
extern "C" int dspx_debug_tc_prof(long long *out16)
{
    return cudaMemcpyFromSymbol(out16, dspx::tc_prof, 16 * sizeof(long long)) == cudaSuccess ? 0 : -1;
}
#endif

int dspx_cosine_matrix(const void *q_dev, int64_t nq, const void *db_dev, int64_t ndb, int dim, int dtype,
                       double *sims_out_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(q_dev && db_dev && sims_out_dev && workspace_dev, "null argument");
    DSPX_REQUIRE(nq >= 0 && ndb >= 0 && dim >= 1, "bad shape");
    DSPX_REQUIRE(nq <= 65535, "at most 65535 query rows per call");
    DSPX_REQUIRE(dtype == DSPX_DTYPE_F32 || dtype == DSPX_DTYPE_F64, "bad dtype");
    DSPX_REQUIRE(workspace_bytes >= dspx_cosine_topk_workspace(nq, ndb, dim, 1), "workspace too small");
    if (nq == 0 || ndb == 0) return DSPX_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char *ws = static_cast<char *>(workspace_dev);
    double *qn = reinterpret_cast<double *>(ws);
    double *dbn = reinterpret_cast<double *>(ws + align256((size_t)nq * dim * 8));
    if (dtype == DSPX_DTYPE_F32) {
        normalize_rows_kernel<float><<<(unsigned)((nq + 127) / 128), 128, 0, st>>>((const float *)q_dev, nq, dim, qn);
        normalize_rows_kernel<float><<<(unsigned)((ndb + 127) / 128), 128, 0, st>>>((const float *)db_dev, ndb, dim, dbn);
    } else {
        normalize_rows_kernel<double><<<(unsigned)((nq + 127) / 128), 128, 0, st>>>((const double *)q_dev, nq, dim, qn);
        normalize_rows_kernel<double><<<(unsigned)((ndb + 127) / 128), 128, 0, st>>>((const double *)db_dev, ndb, dim, dbn);
    }
    dim3 grid((unsigned)((ndb + 255) / 256), (unsigned)nq);
    cosine_matrix_kernel<<<grid, 256, 0, st>>>(qn, dbn, nq, ndb, dim, sims_out_dev);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

int dspx_dct2(const float *x_dev, int64_t rows, int n, int n_mfcc, float *out_dev, void *stream)
{
    DSPX_REQUIRE(x_dev && out_dev, "null argument");
    DSPX_REQUIRE(rows >= 0 && n >= 1 && n_mfcc >= 1, "bad shape");
    if (rows == 0) return DSPX_OK;
    const int64_t total = rows * n_mfcc;
    dct2_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x_dev, rows, n, n_mfcc, out_dev);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

int dspx_hits_at_k(const int32_t *topk_idx_dev, int64_t nq, int k_stride, int k, const int32_t *targets_db_dev,
                   const int32_t *targets_q_dev, long long *hits_dev, void *stream)
{
    DSPX_REQUIRE(topk_idx_dev && targets_db_dev && targets_q_dev && hits_dev, "null argument");
    DSPX_REQUIRE(nq >= 0 && k >= 1 && k <= k_stride, "bad shape");
    if (nq == 0) return DSPX_OK;
    hits_at_k_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        topk_idx_dev, nq, k_stride, k, targets_db_dev, targets_q_dev, reinterpret_cast<unsigned long long *>(hits_dev));
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

}  // extern "C"
