// dspx.cu -- C ABI of libdspx.so (include/dspx.h): plan management, kernel
// launches and the host-buffer pipeline.  All numerical work is in the .cuh
// kernels included below, and what a plan and a call run is chosen in the host
// headers (feat_select.cuh, retrieval_select.cuh); this file validates
// arguments and launches what they choose.
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
#include "feat_select.cuh"
#include "fft_generic.cuh"
#include "retrieval.cuh"
#include "retrieval_f32.cuh"
#include "retrieval_tc.cuh"
#include "retrieval_select.cuh"
#include "ingest.cuh"
#include "resample.cuh"
#include "decode.cuh"
#include "flac.cuh"

// the ctypes binding (dsp_final_b200/_lib.py) mirrors these layouts; tests assert the same numbers
static_assert(sizeof(dspx_config) == 56 && offsetof(dspx_config, f_min) == 24 && offsetof(dspx_config, window) == 48,
              "dspx_config layout changed: update _lib.DspxConfig");
static_assert(sizeof(dspx_plan_info) == 32, "dspx_plan_info layout changed: update _lib.DspxPlanInfo");
static_assert(sizeof(dspx_decode_clip) == 40 && offsetof(dspx_decode_clip, out_start) == 24,
              "dspx_decode_clip layout changed: update batch.py");
static_assert(sizeof(dspx_flac_file) == 80 && offsetof(dspx_flac_file, sample_rate) == 64,
              "dspx_flac_file layout changed: update batch.py");
static_assert(sizeof(dspx_flac_frame) == 48 && offsetof(dspx_flac_frame, in_bytes) == 24,
              "dspx_flac_frame layout changed: update batch.py");

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
    void *d_ws[PIPE_SLOTS] = {nullptr, nullptr, nullptr};    // scratch of the feature call (feat_ws_carve)
    size_t in_bytes = 0, out_bytes = 0, hin_bytes = 0, hout_bytes = 0, ws_bytes = 0;
    void release()
    {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (d_in[i]) cudaFree(d_in[i]);
            if (d_out[i]) cudaFree(d_out[i]);
            if (h_in[i]) cudaFreeHost(h_in[i]);
            if (h_out[i]) cudaFreeHost(h_out[i]);
            if (d_ws[i]) cudaFree(d_ws[i]);
            d_ws[i] = nullptr;
            if (stream[i]) cudaStreamDestroy(stream[i]);
            d_in[i] = d_out[i] = h_in[i] = h_out[i] = nullptr;
            stream[i] = nullptr;
        }
        in_bytes = out_bytes = hin_bytes = hout_bytes = ws_bytes = 0;
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

// ---- feature calls (dspx_features, dspx_embeddings, dspx_log_mel_nchw, dspx_features_pcm16, dspx_features_ragged and
// the host pipeline): feat_steps (feat_select.cuh) chooses the steps, run_features enqueues them ---------------------
struct FeatOut {
    float *logmel, *mfcc, *embed;
    int nchw;                 // log-mel as [B, 1, n_mels, T]
};

static int run_features(const dspx_plan *pl, const FeatBatch &b, const FeatSteps &s, const FeatOut &o, const FeatWs &ws,
                        cudaStream_t st)
{
    const int C = pl->cfg.n_mfcc;
    const int64_t n = b.n_clips;
    float *mf = o.mfcc ? o.mfcc : ws.mfcc;
    if (s.per_clip) {
        // one stream-ordered call per clip into its rows of the stacked outputs, each computed exactly as a [1, length]
        // call computes it; the embeddings from the stacked MFCCs at the end
        const size_t elem = b.dtype == DSPX_DTYPE_PCM16 ? sizeof(int16_t) : sizeof(float);
        for (int64_t i = 0; i < n; i++) {
            const dspx_ragged_clip &c = b.tab[i];
            const FeatBatch row{static_cast<const char *>(b.samples) + c.start * elem, b.dtype, b.normalize, 1, c.length,
                                c.length, nullptr, nullptr};
            const FeatOut ro{o.logmel ? o.logmel + c.first_frame * pl->cfg.n_mels : nullptr,
                             mf ? mf + c.first_frame * C : nullptr, nullptr, 0};
            const int rc = run_features(pl, row, feat_steps(pl, row, mf != nullptr, false), ro, ws, st);
            if (rc != DSPX_OK) return rc;
        }
        return o.embed ? launch_embed(mf, n, 1, C, o.embed, st, b.tab_dev) : DSPX_OK;
    }
    const bool ragged = b.tab != nullptr, pre = pl->cfg.pre_emphasis > 0.0;
    if (ragged) {
        ragged_pairs_kernel<<<(unsigned)((n + 256) / 256), 256, 0, st>>>(b.tab_dev, n, ws.rpairs);
        DSPX_CUDA_CHECK(cudaGetLastError());
    }
    const void *x = b.samples;
    int64_t stride = b.stride;
    if (s.peaks) {
        pcm16_peak_kernel<<<(unsigned)n, 256, 0, st>>>(static_cast<const int16_t *>(b.samples), b.clip_len, b.stride, ws.peaks,
                                                       b.tab_dev);
        DSPX_CUDA_CHECK(cudaGetLastError());
    } else if (s.convert) {
        pcm16_to_float_kernel<<<(unsigned)n, 256, 0, st>>>(static_cast<const int16_t *>(b.samples), b.clip_len, b.stride,
                                                           b.normalize, ws.f32, b.clip_len);
        DSPX_CUDA_CHECK(cudaGetLastError());
        x = ws.f32;
        stride = b.clip_len;
    }
    if (s.fused) DSPX_CUDA_CHECK(cudaMemsetAsync(ws.eacc, 0, (size_t)n * 2 * C * sizeof(long long), st));
    const float *xf = static_cast<const float *>(x);
    int rc;
    if (s.path == W8_GENERIC) {
        rc = launch_generic(pl, xf, n, b.clip_len, stride, s.T, pl->take_feat, pre ? 1 : 0, o.logmel, mf, nullptr, st, o.nchw);
    } else if (s.path == W8_X2 || s.path == W8_X2_AL4) {
        rc = launch_warp8_x2(pl, s.path == W8_X2_AL4, xf, n, stride, s.T, o.logmel, mf, st, o.nchw);
    } else {
        W8Params p = w8_batch_params(pl, x, n, stride, ragged ? 0 : s.T, o.logmel, mf, o.nchw);
        if (ragged) {
            p.rtab = b.tab_dev;
            p.rpairs = ws.rpairs;
            p.n_items = (uint32_t)(b.tab[n - 1].first_pair + (b.tab[n - 1].n_frames + 1) / 2);
        }
        p.eacc = ws.eacc;
        p.peaks = ws.peaks;
        rc = launch_warp8(pl, s.path, p, pre, st);
    }
    if (rc != DSPX_OK) return rc;
    const int64_t frames = ragged ? 1 : s.T;          // a ragged batch takes each clip's frames from its table
    if (s.fused) {
        embed_finalize_kernel<<<(unsigned)((n * C + 255) / 256), 256, 0, st>>>(ws.eacc, n, frames, C, o.embed, b.tab_dev);
        DSPX_CUDA_CHECK(cudaGetLastError());
        return DSPX_OK;
    }
    return o.embed ? launch_embed(mf, n, frames, C, o.embed, st, b.tab_dev) : DSPX_OK;
}

static int ensure_pipe(dspx_plan *pl, size_t in_bytes, size_t out_bytes, size_t ws_bytes, bool stage_in, bool stage_out,
                       HostPipe **out)
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
    if (ws_bytes > hp->ws_bytes) {
        for (int i = 0; i < PIPE_SLOTS; i++) {
            if (hp->d_ws[i]) cudaFree(hp->d_ws[i]);
            hp->d_ws[i] = nullptr;
            DSPX_CUDA_CHECK(cudaMalloc(&hp->d_ws[i], ws_bytes));
        }
        hp->ws_bytes = ws_bytes;
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
    // the kernels read a chunk's device copy: rows of clip_len samples at the start of a cudaMalloc'd, so aligned,
    // buffer.  The steps do not depend on the chunk's clip count: 48 MiB of input hold fewer than 2^31 frames, and a
    // chunk of one clip stays one.
    const FeatBatch batch{nullptr, elem == 2 ? DSPX_DTYPE_PCM16 : DSPX_DTYPE_F32, normalize, chunk, clip_len, clip_len,
                          nullptr, nullptr};
    const FeatSteps steps = mode == 0 ? feat_steps(pl, batch, o_mfcc != nullptr, o_embed != nullptr) : FeatSteps{};
    const size_t mf_b = o_mfcc ? (size_t)T * pl->cfg.n_mfcc * 4 : 0;
    const size_t em_b = (mode == 0 && o_embed) ? (size_t)2 * pl->cfg.n_mfcc * 4 : 0;
    const size_t st_b = mode == 1 ? (size_t)T * pl->n_bins * 8 : 0;
    // the chunk counts an MFCC tensor for embeddings that do not fuse and 16 bytes per coefficient for fused sums
    const size_t scratch_b = steps.mfcc_scratch ? (size_t)T * pl->cfg.n_mfcc * 4 : (steps.fused ? (size_t)pl->cfg.n_mfcc * 16 : 0);
    const size_t out_per_clip = lm_b + mf_b + scratch_b + em_b + st_b;
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
    FeatBatch sized = batch;
    sized.n_clips = chunk;
    const size_t ws_bytes = mode == 0 ? feat_ws_carve(pl, sized, steps, nullptr, nullptr) : 0;
    int rc = ensure_pipe(pl, clip_bytes * chunk, out_bytes, ws_bytes, !in_pinned, !out_pinned, &hp);
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
            if (mf_b) parallel_rows_copy((char *)(o_mfcc + (size_t)f * (mf_b / 4)), mf_b, h + off_mf, mf_b, mf_b, c);
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
        float *d_lm = lm_b ? reinterpret_cast<float *>(d_o) : nullptr;
        float *d_mf = mf_b ? reinterpret_cast<float *>(d_o + off_mf) : nullptr;
        float *d_em = em_b ? reinterpret_cast<float *>(d_o + off_em) : nullptr;
        float *d_st = st_b ? reinterpret_cast<float *>(d_o + off_st) : nullptr;
        if (mode == 0) {
            FeatBatch b = batch;
            b.samples = d_raw;
            b.n_clips = cnt;
            FeatWs ws;
            feat_ws_carve(pl, b, steps, static_cast<char *>(hp->d_ws[slot]), &ws);
            rc = run_features(pl, b, steps, FeatOut{d_lm, d_mf, d_em, 0}, ws, st);
        } else {
            rc = stft_device(pl, static_cast<const float *>(d_raw), cnt, clip_len, clip_len, T, pre,
                             reinterpret_cast<float2 *>(d_st), st);
        }
        if (rc != DSPX_OK) return rc;
        char *h_o = out_pinned ? nullptr : static_cast<char *>(hp->h_out[slot]);
        auto d2h = [&](float *user, size_t per, size_t off, const void *dsrc) -> int {
            if (!per || !dsrc) return DSPX_OK;
            void *dst = out_pinned ? (void *)(user + (size_t)first * (per / 4)) : (void *)(h_o + off);
            DSPX_CUDA_CHECK(cudaMemcpyAsync(dst, dsrc, per * cnt, cudaMemcpyDeviceToHost, st));
            return DSPX_OK;
        };
        if ((rc = d2h(o_logmel, lm_b, 0, d_lm)) != DSPX_OK) return rc;
        if ((rc = d2h(o_mfcc, mf_b, off_mf, d_mf)) != DSPX_OK) return rc;
        if ((rc = d2h(o_embed, em_b, off_em, d_em)) != DSPX_OK) return rc;
        if ((rc = d2h(o_stft, st_b, off_st, d_st)) != DSPX_OK) return rc;
        pend[slot].first = first;
        pend[slot].count = cnt;
    }
    for (int s = 0; s < PIPE_SLOTS; s++)
        if ((rc = drain(s)) != DSPX_OK) return rc;
    return DSPX_OK;
}

// ---- ranking (dspx_cosine_topk, dspx_cosine_matrix) ------------------------------

// The kernel, launch and workspace layout of a call come from topk_select and topk_ws_carve (retrieval_select.cuh).

// Normalised float64 rows of x into out64, plus the operand image that kernel `kern` reads, in tiles of `tile` rows: the
// fp16 split of the tensor-core filter (including its zero padding), the float copy of the FP32 filter, none for TOPK_F64.
template <typename T>
static void launch_normalize(TopkKernel kern, const T *x, int64_t n, int dim, int tile, double *out64, float *img,
                             cudaStream_t st)
{
    if (kern == TOPK_TC) {
        const int64_t n_pad = (n + tile - 1) / tile * tile;
        normalize_rows_split16_kernel<T><<<(unsigned)((n_pad + NR_ROWS - 1) / NR_ROWS), 128, 0, st>>>(
            x, n, n_pad, dim, out64, reinterpret_cast<unsigned char *>(img));
    } else if (kern == TOPK_F32) {
        normalize_rows_tiled_kernel<T><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(x, n, dim, out64, img, tile);
    } else {
        normalize_rows_kernel<T><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(x, n, dim, out64);
    }
}

static void normalize_rows(TopkKernel kern, const void *x, int dtype, int64_t n, int dim, int tile, double *out64,
                           float *img, cudaStream_t st)
{
    if (dtype == DSPX_DTYPE_F32)
        launch_normalize(kern, static_cast<const float *>(x), n, dim, tile, out64, img, st);
    else
        launch_normalize(kern, static_cast<const double *>(x), n, dim, tile, out64, img, st);
}

// each kernel instantiation has its own opt-in flags
template <auto Kernel, class Params>
static int topk_launch(const TopkLaunch &L, const Params &p, int device, cudaStream_t st)
{
    static std::atomic<unsigned char> optin[64];
    DSPX_CUDA_CHECK(optin_max_smem(Kernel, optin, device));
    Kernel<<<L.grid, L.threads, L.smem, st>>>(p);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

// ---- resampling (resample.cuh) --------------------------------------------------

// One batch: zero the per-clip peaks, resample (or copy, for up == down == 1), then divide by the peaks.  Grids are
// split every 65535 clips (grid.y).  max_out: output length of the longest clip.
static int resample_launch(const dspx_resampler *rs, RsBatch b, int64_t n_clips, int64_t max_out, int normalize,
                           unsigned *peaks, cudaStream_t st)
{
    static std::atomic<unsigned char> optin[64];
    const RsGeom &g = rs->g;
    const int64_t tiles = rs->identity ? 0 : rs_tiles(g, max_out);
    DSPX_REQUIRE(tiles < (int64_t)0x7fffffff, "clip too long for one launch");
    if (!rs->identity && g.smem > 48 * 1024) DSPX_CUDA_CHECK(optin_max_smem(resample_poly_kernel, optin, rs->device));
    if (normalize) DSPX_CUDA_CHECK(cudaMemsetAsync(peaks, 0, (size_t)n_clips * sizeof(unsigned), st));
    const int64_t elem_blocks = std::min<int64_t>(rs_ceil_div(max_out, 256), 4096);
    for (int64_t c0 = 0; c0 < n_clips; c0 += 65535) {
        const unsigned nc = (unsigned)std::min<int64_t>(n_clips - c0, 65535);
        RsBatch bc = b;
        if (b.rtab) {
            bc.rtab = b.rtab + c0;
        } else {
            bc.in = static_cast<const char *>(b.in) + (size_t)(c0 * b.in_stride) * (b.pcm ? sizeof(int16_t) : sizeof(float));
            bc.out = b.out + c0 * b.out_stride;
        }
        unsigned *pk = normalize ? peaks + c0 : nullptr;
        if (rs->identity)
            resample_copy_kernel<<<dim3((unsigned)elem_blocks, nc), 256, 0, st>>>(g, bc, pk);
        else
            resample_poly_kernel<<<dim3((unsigned)tiles, nc), RS_THREADS, g.smem, st>>>(g, bc, rs->d_tab, pk);
        DSPX_CUDA_CHECK(cudaGetLastError());
        if (normalize) {
            resample_normalize_kernel<<<dim3((unsigned)elem_blocks, nc), 256, 0, st>>>(g, bc, pk);
            DSPX_CUDA_CHECK(cudaGetLastError());
        }
    }
    return DSPX_OK;
}

// ---- WAV decoding (decode.cuh) ---------------------------------------------------

// A decode table row as dspx_decode_layout writes it; returns an error message or nullptr.
static const char *decode_row_error(const dspx_decode_clip &r)
{
    if (dec_bytes(r.dtype) == 0) return "unknown dtype";
    if (r.channels < 1 || r.channels > DSPX_MAX_CHANNELS) return "channels outside 1 .. 32";
    if (r.n_frames < 1 || r.n_frames > DEC_MAX_LEN) return "n_frames outside 1 .. 2^40";
    if (r.in_offset < 0 || r.in_offset % 16) return "in_offset negative or not a multiple of 16";
    return nullptr;
}

// One launch per pass, split every 65535 clips (grid.y): decode (and fold the peaks), then, when normalising, the
// divide pass.
static int decode_launch(const void *in, const dspx_decode_clip *tab, int64_t n_clips, int64_t max_tiles, int normalize,
                         float *out, unsigned *peaks, cudaStream_t st)
{
    if (normalize) DSPX_CUDA_CHECK(cudaMemsetAsync(peaks, 0, (size_t)n_clips * sizeof(unsigned), st));
    const int passes[2] = {normalize ? DEC_PEAK : DEC_STORE, DEC_NORM};
    for (int p = 0; p < (normalize ? 2 : 1); p++)
        for (int64_t c0 = 0; c0 < n_clips; c0 += 65535) {
            const unsigned nc = (unsigned)std::min<int64_t>(n_clips - c0, 65535);
            wav_decode_kernel<<<dim3((unsigned)max_tiles, nc), DEC_THREADS, DEC_SMEM, st>>>(
                static_cast<const unsigned char *>(in), tab + c0, out, normalize ? peaks + c0 : nullptr, passes[p]);
            DSPX_CUDA_CHECK(cudaGetLastError());
        }
    return DSPX_OK;
}

// ---- FLAC decoding (flac.cuh) ---------------------------------------------------

// The workspace: a peak per file, then the frames' integers (ws_offset is relative to the latter).
static size_t flac_peaks_bytes(int64_t n_files) { return align256((size_t)std::max<int64_t>(n_files, 1) * sizeof(unsigned)); }

static int flac_launch(const void *in, const dspx_flac_file *files, const dspx_flac_frame *frames, int64_t n_frames,
                       int64_t n_files, int normalize, float *out, int32_t *status, char *ws, cudaStream_t st)
{
    unsigned *peaks = reinterpret_cast<unsigned *>(ws);
    char *samples = ws + flac_peaks_bytes(n_files);
    if (normalize) DSPX_CUDA_CHECK(cudaMemsetAsync(peaks, 0, (size_t)n_files * sizeof(unsigned), st));
    flac_frame_kernel<<<(unsigned)((n_frames + FL_THREADS - 1) / FL_THREADS), FL_THREADS, 0, st>>>(
        static_cast<const unsigned char *>(in), files, frames, n_frames, samples, status);
    DSPX_CUDA_CHECK(cudaGetLastError());
    const int passes[2] = {normalize ? FL_PEAK : FL_STORE, FL_NORM};
    for (int p = 0; p < (normalize ? 2 : 1); p++)
        for (int64_t f0 = 0; f0 < n_frames; f0 += 0x7fffffff) {
            const unsigned nf = (unsigned)std::min<int64_t>(n_frames - f0, 0x7fffffff);
            flac_mix_kernel<<<nf, FL_MIX_THREADS, 0, st>>>(files, frames + f0, samples, status + f0, out, peaks, passes[p]);
            DSPX_CUDA_CHECK(cudaGetLastError());
        }
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
    p->device = device;
    p->host_pipe = new (std::nothrow) HostPipe();
    if (!p->host_pipe) { set_error("out of host memory"); delete p; return DSPX_ENOMEM; }
    int rc = plan_derive(cfg, p);
    if (rc != DSPX_OK) {
        plan_free_device(p);
        delete p;
        return rc;
    }

    DeviceGuard guard(device);
    if (!guard.ok) { set_error("cudaSetDevice(%d) failed", device); plan_free_device(p); delete p; return DSPX_ECUDA; }
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { set_error("cudaGetDeviceProperties failed"); plan_free_device(p); delete p; return DSPX_ECUDA; }
    p->sm_count = prop.multiProcessorCount;

    rc = upload(p->host.window32, &p->d_window);
    if (rc == DSPX_OK) rc = upload(p->host.tw, &p->d_tw);
    if (rc == DSPX_OK) rc = upload(p->host.fb_start, &p->d_fb_start);
    if (rc == DSPX_OK) rc = upload(p->host.fb_cnt, &p->d_fb_cnt);
    if (rc == DSPX_OK) rc = upload(p->host.fb_off, &p->d_fb_off);
    if (rc == DSPX_OK) rc = upload(p->host.fb_w, &p->d_fb_w);
    if (rc == DSPX_OK) rc = upload(p->host.dct2_32, &p->d_dct2);
    if (rc == DSPX_OK) rc = upload(p->host.bin_filt, &p->d_bin_filt);
    if (rc == DSPX_OK) rc = upload(p->host.bin_wfall, &p->d_bin_wfall);
    if (rc == DSPX_OK) rc = upload(p->host.bin_wrise, &p->d_bin_wrise);
    if (rc == DSPX_OK && p->kernel == DSPX_KERNEL_WARP8) rc = warp8_prepare(p);
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
    const FeatBatch b{clips_dev, DSPX_DTYPE_F32, 0, n_clips, clip_len, clip_stride, nullptr, nullptr};
    return run_features(plan, b, feat_steps(plan, b, mfcc_out_dev != nullptr, embed_out_dev != nullptr),
                        FeatOut{logmel_out_dev, mfcc_out_dev, embed_out_dev, 0}, FeatWs{}, static_cast<cudaStream_t>(stream));
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
    const FeatBatch b{clips_dev, DSPX_DTYPE_F32, 0, n_clips, clip_len, clip_stride, nullptr, nullptr};
    const FeatSteps s = feat_steps(plan, b, false, true);
    if (!s.fused) {
        set_error("embeddings without an MFCC buffer need the warp8 kernel (n_fft 512 / 1024 / 2048), frame_length = "
                  "n_fft, an even hop and row stride, 8-byte aligned clips and at most %lld frames per clip",
                  (long long)w8_embed_max_frames(plan->cfg.n_mels));
        return DSPX_EUNSUPPORTED;
    }
    FeatWs ws;
    feat_ws_carve(plan, b, s, ws_align(workspace_dev), &ws);
    return run_features(plan, b, s, FeatOut{logmel_out_dev, nullptr, embed_out_dev, 0}, ws, static_cast<cudaStream_t>(stream));
}

int dspx_log_mel_nchw(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len,
                      int64_t clip_stride, float *out_dev, void *stream)
{
    DSPX_REQUIRE(plan && clips_dev && out_dev, "null argument");
    DSPX_REQUIRE(n_clips >= 0 && clip_stride >= clip_len, "bad clip buffer arguments");
    if (dspx_num_frames(plan, clip_len) < 0) return DSPX_EINVAL;
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(plan->device);
    const FeatBatch b{clips_dev, DSPX_DTYPE_F32, 0, n_clips, clip_len, clip_stride, nullptr, nullptr};
    return run_features(plan, b, feat_steps(plan, b, false, false), FeatOut{out_dev, nullptr, nullptr, 1}, FeatWs{},
                        static_cast<cudaStream_t>(stream));
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
    const FeatBatch b{nullptr, dtype, normalize ? 1 : 0, n_clips, 0, 0, table_host, nullptr};
    return feat_ws_carve(plan, b, feat_steps(plan, b, want_mfcc != 0, want_embed != 0), nullptr, nullptr);
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
    const FeatBatch b{samples_dev, dtype, normalize ? 1 : 0, n_clips, 0, 0, table_host, table_dev};
    const FeatSteps s = feat_steps(plan, b, mfcc_out_dev != nullptr, embed_out_dev != nullptr);
    const size_t need = feat_ws_carve(plan, b, s, nullptr, nullptr);
    DSPX_REQUIRE(workspace_dev && workspace_bytes >= need, "workspace too small (%zu bytes needed)", need);
    if (!logmel_out_dev && !mfcc_out_dev && !embed_out_dev) return DSPX_OK;
    DeviceGuard guard(plan->device);
    FeatWs ws;
    feat_ws_carve(plan, b, s, ws_align(workspace_dev), &ws);
    return run_features(plan, b, s, FeatOut{logmel_out_dev, mfcc_out_dev, embed_out_dev, 0}, ws,
                        static_cast<cudaStream_t>(stream));
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
    const FeatBatch b{pcm_dev, DSPX_DTYPE_PCM16, normalize ? 1 : 0, n_clips, clip_len, pcm_stride, nullptr, nullptr};
    const FeatSteps s = feat_steps(plan, b, mfcc_out_dev != nullptr, embed_out_dev != nullptr);
    if (s.convert) {
        set_error("fused PCM16 ingest needs the warp8 kernel (n_fft 512 / 1024 / 2048) and fewer than 2^31 frame pairs: "
                  "convert with dspx_pcm16_to_float first");
        return DSPX_EUNSUPPORTED;
    }
    DSPX_REQUIRE(!embed_out_dev || mfcc_out_dev, "embed_out needs mfcc_out on the PCM16 path");
    DSPX_REQUIRE(n_clips < (int64_t)2147483647, "too many clips for one launch");
    FeatWs ws;
    feat_ws_carve(plan, b, s, ws_align(workspace_dev), &ws);
    return run_features(plan, b, s, FeatOut{logmel_out_dev, mfcc_out_dev, embed_out_dev, 0}, ws,
                        static_cast<cudaStream_t>(stream));
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

size_t dspx_cosine_topk_workspace(int64_t nq, int64_t ndb, int dim, int k)
{
    if (nq < 0 || ndb < 0 || dim <= 0 || k <= 0) return 0;
    return topk_ws_carve(nq, ndb, dim, k, nullptr, nullptr);
}

int dspx_cosine_topk(const void *q_dev, int64_t nq, const void *db_dev, int64_t ndb, int dim, int dtype, int k,
                     int32_t *idx_out_dev, double *score_out_dev, void *workspace_dev, size_t workspace_bytes,
                     void *stream)
{
    DSPX_REQUIRE(db_dev && workspace_dev && (nq == 0 || (q_dev && idx_out_dev)), "null argument");
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
    const TopkLaunch L = topk_select(nq, ndb, dim, k, sm);
    TopkWs ws;
    topk_ws_carve(nq, ndb, dim, k, static_cast<char *>(workspace_dev), &ws);
    if (L.kernel == TOPK_F32) {                        // zero padding of the last tiles (the fp16 split writes its own)
        DSPX_CUDA_CHECK(cudaMemsetAsync(ws.qf, 0, ws.qf_bytes, st));
        DSPX_CUDA_CHECK(cudaMemsetAsync(ws.dbf, 0, ws.dbf_bytes, st));
    }
    normalize_rows(L.kernel, q_dev, dtype, nq, dim, L.kernel == TOPK_TC ? TC_QT : TKF_QPC, ws.qn, ws.qf, st);
    normalize_rows(L.kernel, db_dev, dtype, ndb, dim, TK_ROWS, ws.dbn, ws.dbf, st);
    DSPX_CUDA_CHECK(cudaGetLastError());

    TopkParams tp{};
    tp.qn = ws.qn;
    tp.dbn = ws.dbn;
    tp.nq = nq;
    tp.ndb = ndb;
    tp.dim = dim;
    tp.k = k;
    tp.n_splits = L.n_splits;
    tp.rows_per_split = L.rows_per_split;
    tp.idx_out = L.n_splits == 1 ? idx_out_dev : ws.pidx;
    tp.score_out = L.n_splits == 1 ? score_out_dev : ws.pscore;
    int rc;
    if (L.kernel == TOPK_TC) {
        TopkTcParams cp{};
        cp.base = tp;
        cp.qx = reinterpret_cast<const unsigned char *>(ws.qf);
        cp.dbx = reinterpret_cast<const unsigned char *>(ws.dbf);
        if (L.n_splits > 1) {
            cp.shared_thr = ws.shared_thr;
            cp.done = ws.split_done;
            DSPX_CUDA_CHECK(cudaMemsetAsync(ws.split_done, 0, (size_t)L.grid.x * L.n_splits * 4, st));
#ifdef DSPX_TC_PROFILE                  // profiling builds only: DSPX_EXPERIMENT_KEEP_THR=1 keeps the thresholds of the previous call (steady-state per-role cycles)
            if (!getenv("DSPX_EXPERIMENT_KEEP_THR"))
#endif
                DSPX_CUDA_CHECK(cudaMemsetAsync(ws.shared_thr, 0, (size_t)nq * 8, st));
        }
        rc = L.cw == 26 ? topk_launch<cosine_topk_tc_kernel<26>>(L, cp, dev, st)
                        : topk_launch<cosine_topk_tc_kernel<0>>(L, cp, dev, st);
    } else if (L.kernel == TOPK_F32) {
        TopkF32Params fp{};
        fp.base = tp;
        fp.qf_t = ws.qf;
        fp.dbf_t = ws.dbf;
        fp.eps = 4e-6f + (float)dim * 1.2e-7f;         // > 2 * 2^-24 * (dim + 2): bound on |s32 - s64| for unit vectors
        rc = L.cw == 26 ? topk_launch<cosine_topk_f32_kernel<26>>(L, fp, dev, st)
                        : topk_launch<cosine_topk_f32_kernel<32>>(L, fp, dev, st);
    } else {
        rc = L.cw == 26 ? topk_launch<cosine_topk_kernel<26>>(L, tp, dev, st)
                        : topk_launch<cosine_topk_kernel<32>>(L, tp, dev, st);
    }
    if (rc != DSPX_OK) return rc;
    if (L.n_splits > 1) {
        topk_merge_kernel<<<(unsigned)((nq + 3) / 4), 128, 0, st>>>(ws.pidx, ws.pscore, nq, L.n_splits, k, idx_out_dev, score_out_dev);
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
    DSPX_REQUIRE(workspace_dev && (nq == 0 || ndb == 0 || (q_dev && db_dev && sims_out_dev)), "null argument");
    DSPX_REQUIRE(nq >= 0 && ndb >= 0 && dim >= 1, "bad shape");
    DSPX_REQUIRE(nq <= 65535, "at most 65535 query rows per call");
    DSPX_REQUIRE(dtype == DSPX_DTYPE_F32 || dtype == DSPX_DTYPE_F64, "bad dtype");
    DSPX_REQUIRE(workspace_bytes >= dspx_cosine_topk_workspace(nq, ndb, dim, 1), "workspace too small");
    if (nq == 0 || ndb == 0) return DSPX_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    TopkWs ws;
    topk_ws_carve(nq, ndb, dim, 1, static_cast<char *>(workspace_dev), &ws);
    normalize_rows(TOPK_F64, q_dev, dtype, nq, dim, 0, ws.qn, nullptr, st);
    normalize_rows(TOPK_F64, db_dev, dtype, ndb, dim, 0, ws.dbn, nullptr, st);
    dim3 grid((unsigned)((ndb + 255) / 256), (unsigned)nq);
    cosine_matrix_kernel<<<grid, 256, 0, st>>>(ws.qn, ws.dbn, nq, ndb, dim, sims_out_dev);
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

// ---- resampling ----

int dspx_resampler_create(int64_t up, int64_t down, const float *window_host, int64_t n_window, int device,
                          dspx_resampler **out)
{
    DSPX_REQUIRE(out, "null argument");
    *out = nullptr;
    DSPX_REQUIRE(up >= 1 && down >= 1, "up and down must be >= 1 (got %lld, %lld)", (long long)up, (long long)down);
    int64_t a = up, b = down;
    while (b) { const int64_t r = a % b; a = b; b = r; }
    up /= a;
    down /= a;
    DSPX_REQUIRE(up <= RS_MAX_FACTOR && down <= RS_MAX_FACTOR, "reduced ratio %lld/%lld: factors above 2^20 are not supported",
                 (long long)up, (long long)down);
    const bool identity = up == 1 && down == 1;
    DSPX_REQUIRE(identity || (window_host && n_window >= 1), "a filter window is required");
    const int ndev = dspx_device_count();
    if (ndev <= 0) { set_error("no CUDA device: libdspx has no CPU fallback"); return DSPX_ENODEVICE; }
    DSPX_REQUIRE(device >= 0 && device < ndev, "device %d out of range (%d devices)", device, ndev);
    dspx_resampler *rs = new (std::nothrow) dspx_resampler();
    if (!rs) { set_error("out of host memory"); return DSPX_ENOMEM; }
    rs->identity = identity;
    rs->device = device;
    rs->g.up = up;
    rs->g.down = down;
    if (!identity) {
        std::vector<float> tab;
        int P = 0;
        int64_t remove = 0;
        if (!rs_build_table(up, down, window_host, n_window, tab, &P, &remove)) {
            delete rs;
            set_error("window of %lld taps is too short for up = %lld (need n_window - (n_window - 1) / 2 >= up)",
                      (long long)n_window, (long long)up);
            return DSPX_EINVAL;
        }
        if (!rs_geometry(up, down, P, remove, MAX_OPTIN_SMEM, &rs->g)) {
            delete rs;
            set_error("ratio %lld/%lld needs %d taps per phase: too many for one tile in shared memory", (long long)up,
                      (long long)down, P);
            return DSPX_EINVAL;
        }
        DeviceGuard guard(device);
        if (!guard.ok) { delete rs; set_error("cudaSetDevice(%d) failed", device); return DSPX_ECUDA; }
        const int rc = upload(tab, &rs->d_tab);
        if (rc != DSPX_OK) { cudaFree(rs->d_tab); delete rs; return rc; }
    }
    *out = rs;
    return DSPX_OK;
}

int dspx_resampler_destroy(dspx_resampler *rs)
{
    if (!rs) return DSPX_OK;
    DeviceGuard guard(rs->device);
    cudaFree(rs->d_tab);
    delete rs;
    return DSPX_OK;
}

int64_t dspx_resample_len(const dspx_resampler *rs, int64_t n_in)
{
    DSPX_REQUIRE(rs, "null resampler");
    DSPX_REQUIRE(n_in >= 0 && n_in <= ((int64_t)1 << 40), "input length %lld out of range", (long long)n_in);
    return rs_out_len(n_in, rs->g.up, rs->g.down);
}

size_t dspx_resample_workspace(int64_t n_clips) { return n_clips > 0 ? (size_t)n_clips * sizeof(unsigned) + 256 : 256; }

int dspx_resample(const dspx_resampler *rs, const void *in_dev, int dtype, int64_t n_clips, int64_t n_in, int64_t in_stride,
                  int normalize, float *out_dev, int64_t out_stride, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(rs && in_dev && out_dev, "null argument");
    DSPX_REQUIRE(dtype == DSPX_DTYPE_F32 || dtype == DSPX_DTYPE_PCM16, "resampling takes float32 or PCM16 samples");
    DSPX_REQUIRE(n_clips >= 0 && n_in >= 1 && n_in <= ((int64_t)1 << 40) && in_stride >= n_in, "bad input buffer arguments");
    const int64_t n_out = rs_out_len(n_in, rs->g.up, rs->g.down);
    DSPX_REQUIRE(out_stride >= n_out, "out_stride %lld is shorter than the output (%lld)", (long long)out_stride, (long long)n_out);
    DSPX_REQUIRE(!normalize || (workspace_dev && workspace_bytes >= dspx_resample_workspace(n_clips)), "workspace too small");
    if (n_clips == 0) return DSPX_OK;
    DeviceGuard guard(rs->device);
    const RsBatch b{in_dev, dtype == DSPX_DTYPE_PCM16, n_in, in_stride, out_dev, out_stride, nullptr};
    return resample_launch(rs, b, n_clips, n_out, normalize ? 1 : 0, reinterpret_cast<unsigned *>(ws_align(workspace_dev)),
                           static_cast<cudaStream_t>(stream));
}

int64_t dspx_resample_layout(int64_t up, int64_t down, const int64_t *in_starts, const int64_t *in_lengths, int64_t n_clips,
                             dspx_resample_clip *table_out)
{
    DSPX_REQUIRE(n_clips == 0 || (in_starts && in_lengths && table_out), "null argument");
    DSPX_REQUIRE(n_clips >= 0, "negative clip count");
    DSPX_REQUIRE(up >= 1 && down >= 1, "up and down must be >= 1 (got %lld, %lld)", (long long)up, (long long)down);
    int64_t a = up, b = down;
    while (b) { const int64_t r = a % b; a = b; b = r; }
    up /= a;
    down /= a;
    int64_t at = 0;
    for (int64_t i = 0; i < n_clips; i++) {
        DSPX_REQUIRE(in_lengths[i] >= 1 && in_lengths[i] <= ((int64_t)1 << 40), "clip %lld: length %lld out of range",
                     (long long)i, (long long)in_lengths[i]);
        DSPX_REQUIRE(in_starts[i] >= 0, "clip %lld: negative start %lld", (long long)i, (long long)in_starts[i]);
        dspx_resample_clip &r = table_out[i];
        r.in_start = in_starts[i];
        r.in_length = in_lengths[i];
        r.out_start = at;
        r.out_length = rs_out_len(in_lengths[i], up, down);
        at += (r.out_length + 3) & ~(int64_t)3;      // RAGGED_ALIGN: the packed output is a valid ragged feature batch
    }
    return n_clips ? table_out[n_clips - 1].out_start + table_out[n_clips - 1].out_length : 0;
}

int dspx_resample_ragged(const dspx_resampler *rs, const void *in_dev, int dtype, int normalize,
                         const dspx_resample_clip *table_dev, const dspx_resample_clip *table_host, int64_t n_clips,
                         float *out_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(rs, "null resampler");
    DSPX_REQUIRE(dtype == DSPX_DTYPE_F32 || dtype == DSPX_DTYPE_PCM16, "resampling takes float32 or PCM16 samples");
    DSPX_REQUIRE(n_clips >= 0, "negative clip count");
    if (n_clips == 0) return DSPX_OK;
    DSPX_REQUIRE(in_dev && out_dev && table_dev && table_host, "null argument");
    DSPX_REQUIRE(!normalize || (workspace_dev && workspace_bytes >= dspx_resample_workspace(n_clips)), "workspace too small");
    int64_t max_out = 0;
    for (int64_t i = 0; i < n_clips; i++) {
        const dspx_resample_clip &r = table_host[i];
        DSPX_REQUIRE(r.in_start >= 0 && r.in_length >= 1 && r.in_length <= ((int64_t)1 << 40) && r.out_start >= 0,
                     "clip %lld: bad table row", (long long)i);
        DSPX_REQUIRE(r.out_length == rs_out_len(r.in_length, rs->g.up, rs->g.down),
                     "clip %lld: output length %lld does not match this ratio (%lld)", (long long)i, (long long)r.out_length,
                     (long long)rs_out_len(r.in_length, rs->g.up, rs->g.down));
        max_out = std::max(max_out, r.out_length);
    }
    DeviceGuard guard(rs->device);
    const RsBatch b{in_dev, dtype == DSPX_DTYPE_PCM16, 0, 0, out_dev, 0, table_dev};
    return resample_launch(rs, b, n_clips, max_out, normalize ? 1 : 0, reinterpret_cast<unsigned *>(ws_align(workspace_dev)),
                           static_cast<cudaStream_t>(stream));
}

// ---- WAV decoding ----

int64_t dspx_decode_layout(const int64_t *in_offsets, const int64_t *n_frames, const int32_t *channels, const int32_t *dtypes,
                           int64_t n_clips, dspx_decode_clip *table_out)
{
    DSPX_REQUIRE(n_clips >= 0, "negative clip count");
    DSPX_REQUIRE(n_clips == 0 || (in_offsets && n_frames && channels && dtypes && table_out), "null argument");
    int64_t at = 0;
    for (int64_t i = 0; i < n_clips; i++) {
        const dspx_decode_clip r{in_offsets[i], n_frames[i], channels[i], dtypes[i], at, n_frames[i]};
        const char *bad = decode_row_error(r);
        DSPX_REQUIRE(!bad, "clip %lld: %s (in_offset %lld, n_frames %lld, channels %d, dtype %d)", (long long)i, bad,
                     (long long)r.in_offset, (long long)r.n_frames, (int)r.channels, (int)r.dtype);
        table_out[i] = r;
        at += (r.out_length + 3) & ~(int64_t)3;      // RAGGED_ALIGN: the packed output is a valid ragged batch
    }
    return n_clips ? table_out[n_clips - 1].out_start + table_out[n_clips - 1].out_length : 0;
}

size_t dspx_decode_workspace(int64_t n_clips) { return n_clips > 0 ? (size_t)n_clips * sizeof(unsigned) + 256 : 256; }

int dspx_decode_ragged(const void *in_dev, const dspx_decode_clip *table_dev, const dspx_decode_clip *table_host,
                       int64_t n_clips, int normalize, float *out_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(n_clips >= 0, "negative clip count");
    if (n_clips == 0) return DSPX_OK;
    DSPX_REQUIRE(in_dev && out_dev && table_dev && table_host, "null argument");
    DSPX_REQUIRE(reinterpret_cast<uintptr_t>(in_dev) % 16 == 0 && reinterpret_cast<uintptr_t>(out_dev) % 16 == 0,
                 "in_dev and out_dev must be 16-byte aligned");
    DSPX_REQUIRE(!normalize || (workspace_dev && workspace_bytes >= dspx_decode_workspace(n_clips)), "workspace too small");
    int64_t max_tiles = 0;
    for (int64_t i = 0; i < n_clips; i++) {
        const dspx_decode_clip &r = table_host[i];
        const char *bad = decode_row_error(r);
        DSPX_REQUIRE(!bad, "clip %lld: bad table row: %s", (long long)i, bad);
        DSPX_REQUIRE(r.out_start >= 0 && r.out_start % 4 == 0 && r.out_length == r.n_frames,
                     "clip %lld: out_start must be a non-negative multiple of 4 and out_length equal n_frames", (long long)i);
        max_tiles = std::max(max_tiles, dec_tiles(r));
    }
    DSPX_REQUIRE(max_tiles < (int64_t)0x7fffffff, "clip too long for one launch");
    return decode_launch(in_dev, table_dev, n_clips, max_tiles, normalize ? 1 : 0, out_dev,
                         reinterpret_cast<unsigned *>(ws_align(workspace_dev)), static_cast<cudaStream_t>(stream));
}

// ---- FLAC decoding ----

int64_t dspx_flac_layout(const void *const *files_host, const int64_t *sizes, const int64_t *in_offsets, int64_t n_files,
                         dspx_flac_file *files_out, dspx_flac_frame *frames_out, int64_t frames_capacity,
                         int64_t *n_frames_out)
{
    DSPX_REQUIRE(n_files >= 0 && frames_capacity >= 0, "negative file count or capacity");
    DSPX_REQUIRE(n_files == 0 || (files_host && sizes && in_offsets && n_frames_out), "null argument");
    DSPX_REQUIRE(frames_out || frames_capacity == 0, "frames_out is NULL with a non-zero capacity");
    int64_t at = 0, end = 0, nf = 0, ws = 0;
    FlFile f;
    for (int64_t i = 0; i < n_files; i++) {
        DSPX_REQUIRE(files_host[i] && sizes[i] >= 0, "file %lld: no bytes or a negative size", (long long)i);
        DSPX_REQUIRE(in_offsets[i] >= 0 && in_offsets[i] % 16 == 0, "file %lld: in_offset negative or not a multiple of 16",
                     (long long)i);
        int64_t where = 0;
        const char *bad = fl_parse_file(static_cast<const unsigned char *>(files_host[i]), sizes[i], f, &where);
        DSPX_REQUIRE(!bad, "file %lld: byte %lld: %s", (long long)i, (long long)where, bad);
        if (files_out)
            files_out[i] = dspx_flac_file{in_offsets[i], sizes[i], at, f.samples, nf, (int64_t)f.frames.size(), ws,
                                          f.ws_bytes, f.si.rate, f.si.channels, f.si.bps, 0};
        for (size_t j = 0; j < f.frames.size() && nf + (int64_t)j < frames_capacity; j++) {
            frames_out[nf + (int64_t)j] = f.frames[j];
            frames_out[nf + (int64_t)j].file = (int32_t)i;
        }
        nf += (int64_t)f.frames.size();
        ws += f.ws_bytes;
        end = at + f.samples;
        at += (f.samples + 3) & ~(int64_t)3;      // RAGGED_ALIGN: the packed output is a valid ragged batch
    }
    if (n_frames_out) *n_frames_out = nf;
    return end;
}

size_t dspx_flac_workspace(const dspx_flac_file *files_host, int64_t n_files)
{
    size_t samples = 0;
    for (int64_t i = 0; files_host && i < n_files; i++)
        samples = std::max(samples, (size_t)(files_host[i].ws_start + files_host[i].ws_bytes));
    return 256 + flac_peaks_bytes(n_files) + samples;
}

int dspx_flac_decode(const void *in_dev, const dspx_flac_file *files_dev, const dspx_flac_file *files_host, int64_t n_files,
                     const dspx_flac_frame *frames_dev, const dspx_flac_frame *frames_host, int64_t n_frames, int normalize,
                     float *out_dev, int32_t *status_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    DSPX_REQUIRE(n_files >= 0 && n_frames >= 0, "negative file or frame count");
    if (n_frames == 0) return DSPX_OK;
    DSPX_REQUIRE(in_dev && files_dev && files_host && frames_dev && frames_host && out_dev && status_dev && workspace_dev,
                 "null argument");
    DSPX_REQUIRE(reinterpret_cast<uintptr_t>(in_dev) % 16 == 0 && reinterpret_cast<uintptr_t>(out_dev) % 16 == 0,
                 "in_dev and out_dev must be 16-byte aligned");
    for (int64_t i = 0; i < n_files; i++) {
        const dspx_flac_file &r = files_host[i];
        DSPX_REQUIRE(r.channels >= 1 && r.channels <= DSPX_FLAC_MAX_CHANNELS && r.bps >= 4 && r.bps <= 32 &&
                         r.in_offset >= 0 && r.in_offset % 16 == 0 && r.in_bytes >= 0 && r.out_start >= 0 &&
                         r.out_start % 4 == 0 && r.out_length >= 0 && r.ws_start >= 0 && r.ws_start % 16 == 0 &&
                         r.ws_bytes >= 0,
                     "file %lld: bad table row", (long long)i);
    }
    const size_t need = dspx_flac_workspace(files_host, n_files);
    DSPX_REQUIRE(workspace_bytes >= need, "workspace too small (%zu bytes, need %zu)", workspace_bytes, need);
    for (int64_t f = 0; f < n_frames; f++) {
        const dspx_flac_frame &fr = frames_host[f];
        DSPX_REQUIRE(fr.file >= 0 && fr.file < n_files, "frame %lld: file outside the table", (long long)f);
        const dspx_flac_file &r = files_host[fr.file];
        DSPX_REQUIRE(fr.assignment >= 0 && fr.assignment <= 10 && fl_channels(fr.assignment) == r.channels &&
                         fr.block_size >= 1 && fr.block_size <= FL_MAX_BLOCK && fr.header_bytes >= 6 &&
                         fr.in_bytes >= fr.header_bytes + 2 && fr.in_offset >= 0 &&
                         fr.in_offset + fr.in_bytes <= r.in_bytes && fr.out_start >= 0 &&
                         fr.out_start + fr.block_size <= r.out_length && fr.ws_offset >= 0 && fr.ws_offset % 16 == 0 &&
                         fr.ws_offset + fl_ws_bytes(r.bps, fr.assignment, fr.block_size) <= r.ws_bytes,
                     "frame %lld: bad table row", (long long)f);
    }
    return flac_launch(in_dev, files_dev, frames_dev, n_frames, n_files, normalize ? 1 : 0, out_dev, status_dev,
                       ws_align(workspace_dev), static_cast<cudaStream_t>(stream));
}

}  // extern "C"
