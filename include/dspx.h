/*
 * dspx.h -- C ABI of libdspx.so: the B200 (sm_100a) replacement for the
 * reference's src/dsp -> MFCC-retrieval hot path (Audiofool934/dsp-final).
 *
 * The reference is pure Python and has no FFI layer (SURVEY.md section 8b); its
 * boundary for this path is the import surface of src/dsp plus
 * src/retrieval/retrieval.py.  Each entry point below names the reference
 * interface it stands in for (paths relative to the reference checkout).
 * The Python host side (dsp_final_b200/) binds these with ctypes and keeps
 * the reference's call signatures; INTEGRATION.md shows the reference-side shim.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - return 0 on success, a negative DSPX_E* code otherwise; never throws.
 *     dspx_last_error() returns a thread-local message for the last failure.
 *     A call that returns DSPX_EUNSUPPORTED has enqueued nothing, so the
 *     caller may fall back to another entry point on the same buffers.
 *   - "_dev" pointers are device memory owned by the caller; all device work is
 *     enqueued on the caller's stream (cudaStream_t passed as void*), with no
 *     hidden synchronisation and no allocation in the launch path.
 *   - "_host" entry points take host memory, run their own pinned staging and
 *     copy/compute overlap, and return after the results are in the host
 *     buffers.
 *   - the plan owns device constant tables (window, twiddles, sparse mel
 *     filterbank, DCT basis); it is immutable after creation and may be shared
 *     between threads.
 *   - there is no CPU fallback: without a CUDA device every compute entry
 *     point fails with DSPX_ENODEVICE.
 */
#ifndef DSPX_H
#define DSPX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSPX_OK 0
#define DSPX_EINVAL (-1)      /* bad argument (the Python side raises ValueError) */
#define DSPX_ENOMEM (-2)
#define DSPX_ECUDA (-3)       /* a CUDA runtime call failed; see dspx_last_error() */
#define DSPX_ENODEVICE (-4)
#define DSPX_EUNSUPPORTED (-5)

#define DSPX_WINDOW_HANN 0
#define DSPX_WINDOW_HAMMING 1
#define DSPX_WINDOW_RECT 2

#define DSPX_DTYPE_F32 0
#define DSPX_DTYPE_F64 1

/* kernel selection for dspx_features (dspx_plan_info.kernel reports the pick) */
#define DSPX_KERNEL_AUTO 0
#define DSPX_KERNEL_GENERIC 1  /* any power-of-two n_fft in [16, 8192] */
#define DSPX_KERNEL_WARP8 2    /* warp-autonomous packed-f32x2 kernel: frame_length = n_fft in {512, 1024, 2048} */

/* Field-for-field image of the reference MfccConfig dataclass, src/dsp/mfcc.py:10-21. */
typedef struct dspx_config {
    int32_t sample_rate;
    int32_t frame_length;
    int32_t hop_length;
    int32_t n_fft;          /* 0 = None -> frame_length (mfcc.py:89) */
    int32_t n_mels;
    int32_t n_mfcc;
    double f_min;
    double f_max;           /* < 0 = None -> sample_rate / 2 (mfcc.py:39-40) */
    double pre_emphasis;    /* <= 0 disables (mfcc.py:87) */
    int32_t window;         /* DSPX_WINDOW_* (src/dsp/stft.py:12-24) */
    int32_t kernel;         /* DSPX_KERNEL_*; 0 = auto */
} dspx_config;

typedef struct dspx_plan dspx_plan;

typedef struct dspx_plan_info {
    int32_t n_fft_pow2;     /* transform length: next power of two (fft.py:38-42, mfcc.py:91) */
    int32_t n_bins;         /* n_fft_pow2 / 2 + 1 */
    int32_t take_features;  /* samples of each frame that enter the FFT on the MFCC path */
    int32_t take_stft;      /* same for the plain stft() entry (fft.py:32-33 truncation) */
    int32_t mel_nnz;        /* non-zeros of the mel filterbank */
    int32_t kernel;         /* DSPX_KERNEL_* actually used by dspx_features */
    int32_t device;
    int32_t sm_count;
} dspx_plan_info;

const char *dspx_version(void);
const char *dspx_last_error(void);
int dspx_device_count(void);

/* ---- plan: MfccConfig + the lru-cached tables of stft.py:12, mfcc.py:61,79 ---- */
int dspx_plan_create(const dspx_config *cfg, int device, dspx_plan **out);
int dspx_plan_destroy(dspx_plan *plan);
int dspx_plan_get_info(const dspx_plan *plan, dspx_plan_info *out);
/* n_frames = 1 + (clip_len - frame_length) / hop_length (stft.py:33); DSPX_EINVAL when
 * clip_len < frame_length (the reference reads out of bounds there; we refuse). */
int64_t dspx_num_frames(const dspx_plan *plan, int64_t clip_len);
/* copy a constant table back to the host (tests): which = 0 window [frame_length] f32,
 * 1 dense mel filterbank [n_mels, n_bins] f32, 2 DCT basis x2 [n_mfcc, n_mels] f32 */
int dspx_plan_read_table(const dspx_plan *plan, int which, float *out_host, int64_t capacity);

/* ---- stft(signal, frame_length, hop_length, window, n_fft)  src/dsp/stft.py:43-56 ----
 * clips_dev [n_clips][clip_stride] f32, first clip_len samples of each row used.
 * out_dev [n_clips, n_frames, n_bins] interleaved complex64.  pre_emphasis: 0 for the
 * reference stft() (which has none), 1 to see the spectrum the MFCC path uses. */
int dspx_stft(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len,
              int64_t clip_stride, int pre_emphasis, float *out_dev, void *stream);

/* ---- log_mel_spectrogram / mfcc / clip embedding, fused ----
 * src/dsp/mfcc.py:86-109 and src/retrieval/retrieval.py:19-23,38-41.
 * Any of the three outputs may be NULL; embed_out_dev needs mfcc_out_dev.
 * logmel [n_clips, n_frames, n_mels] f32; mfcc [n_clips, n_frames, n_mfcc] f32;
 * embed [n_clips, 2*n_mfcc] f32 = concat(mean_t, std_t (ddof 0)). */
int dspx_features(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len,
                  int64_t clip_stride, float *logmel_out_dev, float *mfcc_out_dev,
                  float *embed_out_dev, void *stream);

/* Clip embeddings alone (compute_embeddings, src/retrieval/retrieval.py:26-43, without keeping the MFCCs):
 * the feature kernel adds every frame's coefficients and their squares to per-clip fixed-point accumulators in
 * workspace_dev (order-independent, so results are reproducible) and a finalize step writes
 * embed [n_clips, 2*n_mfcc] f32.  No MFCC tensor is written or read.  logmel_out_dev may be NULL.
 * Runs when the plan uses the warp8 kernel, frame_length equals the transform length (n_fft_pow2) and that is 512,
 * 1024 or 2048, hop_length and clip_stride are even, clips_dev is 8-byte aligned and n_clips * ceil(n_frames / 2)
 * < 2^31.  Otherwise DSPX_EUNSUPPORTED: use dspx_features with an MFCC buffer. */
size_t dspx_embeddings_workspace(const dspx_plan *plan, int64_t n_clips);
int dspx_embeddings(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len,
                    int64_t clip_stride, float *embed_out_dev, float *logmel_out_dev, void *workspace_dev,
                    size_t workspace_bytes, void *stream);

/* log-mel written directly in the CNN input layout [n_clips, 1, n_mels, n_frames] that
 * LogMelTransform / train_cnn build with feat.T[None] (src/train/transforms.py:16-18,
 * scripts/models/train_cnn.py:46-47): same values as dspx_features' log-mel, transposed in the
 * store epilogue (SURVEY 8f row f3). */
int dspx_log_mel_nchw(const dspx_plan *plan, const float *clips_dev, int64_t n_clips, int64_t clip_len,
                      int64_t clip_stride, float *out_dev, void *stream);

/* dct_type_2(x, n_mfcc), src/dsp/mfcc.py:73-83, for callers that hold their own log-mel
 * rows (scripts/tools/plot_dsp_viz.py): x [rows, n] f32 -> out [rows, n_mfcc] f32,
 * out[r,k] = 2 * sum_j x[r,j] cos(pi/n (j+0.5) k). */
int dspx_dct2(const float *x_dev, int64_t rows, int n, int n_mfcc, float *out_dev, void *stream);

/* mean / population-std over frames of any [n_clips, n_frames, n_coef] f32 feature
 * tensor (retrieval.py:38-41 on cached features). out [n_clips, 2*n_coef] f32. */
int dspx_embed_stats(const float *feats_dev, int64_t n_clips, int64_t n_frames, int n_coef,
                     float *out_dev, void *stream);

/* Optional CMVN epilogue (BASELINE.json north_star "a log/CMVN epilogue"; the reference applies none after
 * mfcc.py:102-109, so callers opt in): in place over [n_clips, n_frames, n_coef] f32 features,
 * y = (x - mean_t) / (std_t + eps) per clip and coefficient, population std, statistics in float64. */
int dspx_cmvn(float *feats_dev, int64_t n_clips, int64_t n_frames, int n_coef, double eps, void *stream);

/* Host-buffer twins of the two calls above (what FeatureCache.compute_feature,
 * src/features/cache.py:65-74, and a batched precompute need): pinned staging,
 * chunked H2D / kernel / D2H overlap inside; synchronous. */
int dspx_features_host(const dspx_plan *plan, const float *clips_host, int64_t n_clips,
                       int64_t clip_len, int64_t clip_stride, float *logmel_out_host,
                       float *mfcc_out_host, float *embed_out_host);
int dspx_stft_host(const dspx_plan *plan, const float *clips_host, int64_t n_clips,
                   int64_t clip_len, int64_t clip_stride, int pre_emphasis, float *out_host);

/* ---- PCM16 ingest: load_audio + normalize_audio, src/utils/audio.py:19-38 (SURVEY 8f row f2) ----
 * x = int16 / 32768 (what soundfile returns for dtype="float32"), then x / max|x| when normalize
 * != 0 and the clip is not all zero -- the correctly rounded float32 quotient, i.e. bit-identical
 * to NumPy.  The _host form ships int16 over PCIe (half the bytes of float32 clips). */
int dspx_pcm16_to_float(const int16_t *pcm_dev, int64_t n_clips, int64_t clip_len, int64_t pcm_stride,
                        int normalize, float *out_dev, int64_t out_stride, void *stream);
/* Device-pointer form with the conversion FUSED into the feature kernel's sample loads: no float32 copy of the clips
 * exists.  Runs when the plan uses the warp8 kernel with a transform length (n_fft_pow2) of 512, 1024 or 2048 and
 * n_clips * ceil(n_frames / 2) < 2^31; otherwise DSPX_EUNSUPPORTED: convert with dspx_pcm16_to_float first.  q = s * (1/m), one fma refinement -- the
 * correctly rounded s / m for every |s| <= m <= 32768 (checked exhaustively), i.e. the same samples as above.
 * workspace_dev (dspx_features_pcm16_workspace bytes) holds one peak per clip; unused when normalize == 0. */
size_t dspx_features_pcm16_workspace(int64_t n_clips);
int dspx_features_pcm16(const dspx_plan *plan, const int16_t *pcm_dev, int64_t n_clips, int64_t clip_len,
                        int64_t pcm_stride, int normalize, float *logmel_out_dev, float *mfcc_out_dev,
                        float *embed_out_dev, void *workspace_dev, size_t workspace_bytes, void *stream);
int dspx_features_host_pcm16(const dspx_plan *plan, const int16_t *pcm_host, int64_t n_clips,
                             int64_t clip_len, int64_t pcm_stride, int normalize,
                             float *logmel_out_host, float *mfcc_out_host, float *embed_out_host);

/* ---- ragged batches: clips of different lengths in one call ----
 * The clips lie back to back in one flat buffer of float32 or int16 samples.  dspx_ragged_layout (host only, no
 * device needed) validates their starts and lengths and fills one table row per clip; the outputs are the per-clip
 * outputs of dspx_features stacked along the frame axis: logmel [total_frames, n_mels], mfcc [total_frames, n_mfcc],
 * embed [n_clips, 2*n_mfcc]; clip i owns rows first_frame .. first_frame + n_frames - 1.  Every clip gets exactly
 * the values dspx_features / dspx_features_pcm16 give it alone (pre-emphasis restarts at its sample 0). */
#define DSPX_DTYPE_PCM16 2
typedef struct dspx_ragged_clip {
    int64_t start;        /* first sample of the clip in the flat buffer (samples of the buffer's type) */
    int64_t length;       /* samples */
    int64_t n_frames;     /* 1 + (length - frame_length) / hop_length */
    int64_t first_frame;  /* row of its first frame in the [total_frames, ...] outputs */
    int64_t first_pair;   /* exclusive prefix sum of (n_frames + 1) / 2 */
} dspx_ragged_clip;
/* Returns total_frames (>= 0), or DSPX_EINVAL naming the first clip shorter than frame_length, a float32 clip that
 * starts at an odd sample, a negative start, or a batch of 2^31 frame pairs or more.  dtype: DSPX_DTYPE_F32 or
 * DSPX_DTYPE_PCM16. */
int64_t dspx_ragged_layout(const dspx_config *cfg, const int64_t *starts, const int64_t *lengths, int64_t n_clips,
                           int dtype, dspx_ragged_clip *table_out);
/* Device scratch for one dspx_features_ragged call with these outputs requested (flags 0 / 1). */
size_t dspx_features_ragged_workspace(const dspx_plan *plan, const dspx_ragged_clip *table_host, int64_t n_clips,
                                      int dtype, int normalize, int want_logmel, int want_mfcc, int want_embed);
/* samples_dev: the flat buffer (float32: 8-byte aligned), dtype DSPX_DTYPE_F32 or DSPX_DTYPE_PCM16 (normalize as in
 * dspx_features_pcm16).  table_dev and table_host hold the same dspx_ragged_layout table, on the device and on the
 * host.  Any of the three outputs may be NULL.  Warp8 plans with n_fft 512 / 1024 / 2048 run one launch for the
 * whole batch (with embed alone on aligned float32 frames, the fused embeddings of dspx_embeddings).  Plans without
 * a ragged kernel (the generic kernel, n_fft 4096) loop over the clips on the host and enqueue one feature call per
 * clip: correct, but as slow as one call per clip. */
int dspx_features_ragged(const dspx_plan *plan, const void *samples_dev, int dtype, int normalize,
                         const dspx_ragged_clip *table_dev, const dspx_ragged_clip *table_host, int64_t n_clips,
                         int64_t total_frames, float *logmel_out_dev, float *mfcc_out_dev, float *embed_out_dev,
                         void *workspace_dev, size_t workspace_bytes, void *stream);
/* dspx_embed_stats over stacked features: feats [total_frames, n_coef], clip i = rows first_frame .. + n_frames;
 * out [n_clips, 2*n_coef].  Same per-clip summation order as dspx_embed_stats. */
int dspx_embed_stats_ragged(const float *feats_dev, const dspx_ragged_clip *table_dev, int64_t n_clips, int n_coef,
                            float *out_dev, void *stream);

/* ---- fft / ifft / rfft  src/dsp/fft.py:27-77 ----
 * in_dev [batch, n_in] interleaved complex64; the first min(n_in, n) samples are used,
 * zero-padded to P = next_pow2(n).  out_dev and work_dev each hold [batch, P] complex64.
 * inverse != 0 gives conj(fft(conj x)) / P. */
int64_t dspx_next_pow_two(int64_t n);
int dspx_fft_c2c(const float *in_dev, int64_t batch, int64_t n_in, int64_t n, int inverse,
                 float *out_dev, float *work_dev, void *stream);

/* ---- cosine_similarity + argsort(-sims)[:, :k]  src/retrieval/retrieval.py:46-49,65 ----
 * q [nq, dim], db [ndb, dim] of dtype DSPX_DTYPE_*.  Scores are float64, rows scaled by
 * 1/(||row|| + 1e-10); idx_out [nq, k] int32 in descending score order, ties broken by
 * the lower database index (np.argsort(..., kind="stable")).  score_out may be NULL.
 * workspace_dev must hold dspx_cosine_topk_workspace() bytes.  k <= DSPX_MAX_K. */
#define DSPX_MAX_K 128
size_t dspx_cosine_topk_workspace(int64_t nq, int64_t ndb, int dim, int k);
int dspx_cosine_topk(const void *q_dev, int64_t nq, const void *db_dev, int64_t ndb, int dim,
                     int dtype, int k, int32_t *idx_out_dev, double *score_out_dev,
                     void *workspace_dev, size_t workspace_bytes, void *stream);

/* The dense matrix itself (cosine_similarity, retrieval.py:46-49), float64 [nq, ndb];
 * same scores, bit for bit, as the ones dspx_cosine_topk ranks.  Same workspace. */
int dspx_cosine_matrix(const void *q_dev, int64_t nq, const void *db_dev, int64_t ndb, int dim,
                       int dtype, double *sims_out_dev, void *workspace_dev, size_t workspace_bytes,
                       void *stream);

/* hit@k of evaluate_retrieval (retrieval.py:66-70): adds, for the first k of every row of
 * topk_idx [nq, k_stride], one hit when any retrieved DB target equals the query target.
 * hits_dev is a device int64 the caller zeroed. */
int dspx_hits_at_k(const int32_t *topk_idx_dev, int64_t nq, int k_stride, int k,
                   const int32_t *targets_db_dev, const int32_t *targets_q_dev,
                   long long *hits_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DSPX_H */
