// emu.cu -- TEST-ONLY host replay of the kernels' phase functions.
//
// The feature kernels are written as __host__ __device__ "phase" functions over a
// flat item index, separated by barriers.  This file replays those same functions
// on the CPU, one item after another, so that the index arithmetic, table layouts
// and numerics of the CUDA source can be checked against the oracle in the dev
// container (which has nvcc but no GPU).  It is built into libdspx_emu.so, which
// only tests/ load; libdspx.so (the product) contains none of this and has no CPU
// path.
#include <vector>

#define DSPX_EMU                     // no launchers, so no feature-kernel instantiations: only their phase functions run here
#include "dspx_internal.cuh"
#include "tables.cuh"
#include "feat_generic.cuh"
#include "feat_warp8.cuh"
#include "feat_warp8_x2.cuh"

namespace dspx {
void set_error(const char *, ...) {}
const char *get_error() { return ""; }
}  // namespace dspx

using namespace dspx;

struct EmuTables {
    HostTables t;
    std::vector<float> window, dct2;
    std::vector<float2> tw;
    int P = 0, M = 0, n_bins = 0, take_feat = 0, take_stft = 0, n_stages = 0;
    int radix[16] = {0};
};

static int emu_build(const dspx_config *cfg, EmuTables &e)
{
    const int nfft_raw = cfg->n_fft > 0 ? cfg->n_fft : cfg->frame_length;
    e.P = (int)next_pow_two(nfft_raw);
    if (e.P < 16 || e.P > 8192) return DSPX_EUNSUPPORTED;
    e.M = e.P / 2;
    e.n_bins = e.M + 1;
    e.take_feat = cfg->frame_length < e.P ? cfg->frame_length : e.P;
    e.take_stft = cfg->frame_length < nfft_raw ? cfg->frame_length : nfft_raw;
    int m = e.M;
    while (m > 1) {
        if (m % 4 == 0) { e.radix[e.n_stages++] = 4; m /= 4; }
        else { e.radix[e.n_stages++] = 2; m /= 2; }
    }
    if (!build_window(cfg->window, cfg->frame_length, e.t.window)) return DSPX_EINVAL;
    const double f_max = cfg->f_max < 0.0 ? cfg->sample_rate / 2.0 : cfg->f_max;
    build_filterbank(cfg->n_mels, e.P, cfg->sample_rate, cfg->f_min, f_max, e.t);
    build_dct2(cfg->n_mfcc, cfg->n_mels, e.t.dct2);
    e.window.assign(e.t.window.begin(), e.t.window.end());
    e.dct2.assign(e.t.dct2.begin(), e.t.dct2.end());
    e.tw.resize(e.P);
    for (int j = 0; j < e.P; j++) {
        const double a = -2.0 * M_PI * (double)j / (double)e.P;
        e.tw[j] = make_float2((float)std::cos(a), (float)std::sin(a));
    }
    return DSPX_OK;
}

extern "C" {

// Replays feat_generic_kernel.  stft_out != NULL selects the complex-spectrum mode.
int emu_features_generic(const dspx_config *cfg, const float *clips, int64_t n_clips, int64_t clip_len,
                         int64_t clip_stride, int stft_mode, int stft_pre, float *logmel, float *mfcc, float *stft_out,
                         int frames_per_cta_override)
{
    EmuTables e;
    int rc = emu_build(cfg, e);
    if (rc != DSPX_OK) return rc;
    if (clip_len < cfg->frame_length) return DSPX_EINVAL;
    const int64_t T = 1 + (clip_len - cfg->frame_length) / cfg->hop_length;
    GenParams p{};
    p.clips = clips;
    p.n_clips = n_clips;
    p.clip_len = clip_len;
    p.clip_stride = clip_stride;
    p.n_frames = T;
    p.frame_length = cfg->frame_length;
    p.hop = cfg->hop_length;
    p.take = stft_mode ? e.take_stft : e.take_feat;
    p.P = e.P;
    p.M = e.M;
    p.n_bins = e.n_bins;
    p.n_stages = e.n_stages;
    for (int i = 0; i < 16; i++) p.radix[i] = e.radix[i];
    p.n_mels = cfg->n_mels;
    p.n_mfcc = cfg->n_mfcc;
    int G = 1024 / e.M;
    if (G < 1) G = 1;
    if (G > 16) G = 16;
    p.G = G;
    const int64_t groups = (T + G - 1) / G;
    int64_t gpc = frames_per_cta_override > 0 ? (frames_per_cta_override + G - 1) / G : groups;
    p.frames_per_cta = (int)(gpc * G);
    p.ctas_per_clip = (int)((T + p.frames_per_cta - 1) / p.frames_per_cta);
    p.pre = stft_mode ? (stft_pre && cfg->pre_emphasis > 0.0) : (cfg->pre_emphasis > 0.0);
    p.alpha = (float)cfg->pre_emphasis;
    p.window = e.window.data();
    p.tw = e.tw.data();
    p.fb_start = e.t.fb_start.data();
    p.fb_cnt = e.t.fb_cnt.data();
    p.fb_off = e.t.fb_off.data();
    p.fb_w = e.t.fb_w.data();
    p.dct2 = e.dct2.data();
    p.logmel = logmel;
    p.lm_ts = p.n_mels;
    p.lm_fs = 1;
    p.mfcc = mfcc;
    p.stft = stft_mode ? reinterpret_cast<float2 *>(stft_out) : nullptr;

    std::vector<unsigned char> smem(gen_smem_bytes(G, p.M, p.n_mels));
    const GenSmem sm = gen_carve(smem.data(), G, p.M, p.n_mels);
    for (int64_t blk = 0; blk < n_clips * p.ctas_per_clip; blk++) {
        const int64_t clip_idx = blk / p.ctas_per_clip, chunk = blk - clip_idx * p.ctas_per_clip;
        const float *clip = clips + clip_idx * clip_stride;
        const int64_t t_begin = chunk * p.frames_per_cta;
        int64_t t_end = t_begin + p.frames_per_cta;
        if (t_end > T) t_end = T;
        for (int64_t t0 = t_begin; t0 < t_end; t0 += G) {
            for (int i = 0; i < G * p.M; i++) gen_phase_load(p, sm, clip, t0, i);
            float2 *in = sm.a, *out = sm.b;
            int ns = 1;
            for (int s = 0; s < p.n_stages; s++) {
                for (int i = 0; i < G * (p.M / p.radix[s]); i++) gen_phase_stage(p, in, out, s, ns, i);
                ns *= p.radix[s];
                float2 *tmp = in; in = out; out = tmp;
            }
            float *pw = reinterpret_cast<float *>(out);
            for (int i = 0; i < G * (p.M / 2 + 1); i++) gen_phase_post(p, in, pw, clip_idx, t0, i);
            if (!p.stft) {
                for (int i = 0; i < G * p.n_mels * GEN_MEL_PARTS; i++) gen_phase_melpart(p, pw, sm.part, i);
                for (int i = 0; i < G * p.n_mels; i++) gen_phase_logmel(p, sm.part, sm.lm, clip_idx, t0, i);
                if (p.mfcc)
                    for (int i = 0; i < G * p.n_mfcc; i++) gen_phase_dct(p, sm.lm, clip_idx, t0, i);
            }
        }
    }
    return DSPX_OK;
}

// Modelled shared-memory wavefronts of the table-driven accesses of feat_warp8_kernel (the model w8_wavefronts64 /
// the quarter-warp rule for 128-bit loads; profiles/r02_warp8_layout.md compares it with ncu's per-instruction counts):
// out = {power stores, their minimum, run-piece sum stores, their minimum, filter-sum loads, their minimum, rounds,
//        bins that share a tile slot with another bin (must be 0)}
int emu_warp8_layout(const dspx_config *cfg, int32_t *out)
{
    EmuTables e;
    int rc = emu_build(cfg, e);
    if (rc != DSPX_OK) return rc;
    dspx_plan pl;
    pl.cfg = *cfg;
    pl.P = e.P;
    pl.M = e.M;
    pl.n_bins = e.n_bins;
    pl.host = e.t;
    if (!warp8_supported(&pl)) return DSPX_EUNSUPPORTED;
    std::vector<float> blob;
    W8Tables tb{};
    warp8_build_tables(&pl, blob, tb);
    if (tb.x2) return DSPX_EUNSUPPORTED;
    const int units = tb.r1 >= 8 ? tb.r1 / 8 : 1, active = tb.r1 >= 8 ? 32 : 16, M = 64 * tb.r1, J = 8 * tb.r1;
    const int32_t *ppos = reinterpret_cast<const int32_t *>(blob.data() + tb.ppos);
    const int dump = W8_CSTRIDE * tb.n_slots + 8;
    int pw = 0, pw_min = 0;
    std::vector<int> owner(dump + 1, -1);
    int shared_slots = 0;
    for (int w = 0; w < units; w++)
        for (int m = 0; m < 9; m++)
            for (int s = 0; s < 2; s++) {
                int a[32], n = 0;
                for (int l = 0; l < 32; l++) {
                    const bool on = l < active && (m < 8 || l + 32 * w == 0);
                    a[l] = on ? ppos[((w * 9 + m) * 32 + l) * 2 + s] : -1;
                    n += on;
                    if (on && a[l] != dump) {
                        const int k0 = w8_bin(J, l + 32 * w, m), k = s ? M - k0 : k0;
                        if (owner[a[l]] >= 0 && owner[a[l]] != k) shared_slots++;
                        owner[a[l]] = k;
                    }
                }
                pw += w8_wavefronts64(a);
                pw_min += (n > 16) ? 2 : (n > 0 ? 1 : 0);
            }
    const int32_t *cflag = reinterpret_cast<const int32_t *>(blob.data() + tb.cflag);
    int sw = 0, sw_min = 0;
    for (int r = 0; r < tb.rounds; r++)
        for (int s = 0; s < 2; s++) {
            int a[32], lo = 0, hi = 0;
            for (int l = 0; l < 32; l++) {
                const int fl = cflag[w8_flag_index(l * tb.rounds + r, l, tb.rounds)];
                a[l] = (fl & 2) ? (s ? (int)((unsigned)fl >> 20) : ((fl >> 8) & 0xfff)) : -1;
                if (a[l] >= 0) (l < 16 ? lo : hi)++;
            }
            sw += w8_wavefronts64(a);
            sw_min += (lo > 0) + (hi > 0);
        }
    const int32_t *fd = reinterpret_cast<const int32_t *>(blob.data() + tb.fdesc);
    const int psh = tb.cw_lanes == 16 ? 1 : 0, n_slots = tb.lm_part << psh;
    int fl_wf = 0, fl_min = 0;
    for (int base = 0; base < n_slots; base += 32)
        for (int i = 0; i < 3; i++)
            for (int q = 0; q < 4; q++) {                                   // 128-bit loads: a quarter-warp per wavefront
                int units16[8], cnt[8] = {0}, worst = 0;
                for (int l = 0; l < 8; l++) {
                    const int f = base + 8 * q + l;
                    units16[l] = fd[2 * (f < cfg->n_mels ? f : 0)] / 2 + i;
                    bool dup = false;
                    for (int o = 0; o < l; o++) dup = dup || units16[o] == units16[l];
                    if (!dup) worst = std::max(worst, ++cnt[units16[l] & 7]);
                }
                fl_wf += worst;
                fl_min += 1;
            }
    out[0] = pw; out[1] = pw_min; out[2] = sw; out[3] = sw_min; out[4] = fl_wf; out[5] = fl_min; out[6] = tb.rounds; out[7] = shared_slots;
    return DSPX_OK;
}

// Replays feat_warp8_kernel: one "warp" at a time, each phase run for lanes 0..31 in turn
// (a __syncwarp() separates the phases on the device).  rtab != NULL replays the RAGGED variant over a
// dspx_ragged_layout table (clip_len and clip_stride unused).
static int emu_warp8(const dspx_config *cfg, const float *clips, int64_t n_clips, int64_t clip_len,
                     int64_t clip_stride, float *logmel, float *mfcc, float *stft_out, int stft_pre,
                     const dspx_ragged_clip *rtab)
{
    EmuTables e;
    int rc = emu_build(cfg, e);
    if (rc != DSPX_OK) return rc;
    dspx_plan pl;
    pl.cfg = *cfg;
    pl.P = e.P;
    pl.M = e.M;
    pl.n_bins = e.n_bins;
    pl.host = e.t;
    pl.take_stft = e.take_stft;
    pl.kernel = DSPX_KERNEL_WARP8;
    if (!warp8_supported(&pl) || (!rtab && clip_len < cfg->frame_length)) return DSPX_EUNSUPPORTED;
    const int64_t T = rtab ? 0 : 1 + (clip_len - cfg->frame_length) / cfg->hop_length;
    // the variant the library would launch
    const W8Path path = warp8_select(&pl, clips, clip_stride, DSPX_DTYPE_F32, rtab != nullptr, n_clips, T,
                                     stft_out ? W8_WANT_STFT : W8_WANT_FEATURES);
    if (path == W8_GENERIC || path == W8_UNSUPPORTED) return DSPX_EUNSUPPORTED;
    const bool u4 = path == W8_U4, share = path == W8_SHARE;
    std::vector<float> blob;
    W8Tables tb{};
    warp8_build_tables(&pl, blob, tb);
    W8Params p{};
    p.clips = clips;
    p.n_clips = n_clips;
    p.clip_stride = clip_stride;
    p.n_frames = T;
    p.pairs_per_clip = (uint32_t)((T + 1) / 2);
    p.n_items = (uint32_t)(n_clips * p.pairs_per_clip);
    std::vector<uint32_t> rpairs;
    if (rtab) {
        for (int64_t i = 0; i < n_clips; i++) rpairs.push_back((uint32_t)rtab[i].first_pair);
        rpairs.push_back(n_clips ? (uint32_t)(rtab[n_clips - 1].first_pair + (rtab[n_clips - 1].n_frames + 1) / 2) : 0);
        p.rtab = rtab;
        p.rpairs = rpairs.data();
        p.n_items = rpairs.back();
    }
    p.hop = cfg->hop_length;
    p.n_mels = cfg->n_mels;
    p.n_mfcc = cfg->n_mfcc;
    p.alpha = (float)cfg->pre_emphasis;
    p.tb = tb;
    p.tables = blob.data();
    p.logmel = logmel;
    p.mfcc = mfcc;
    p.lm_ts = p.n_mels;
    p.lm_fs = 1;
    p.stft = reinterpret_cast<float2 *>(stft_out);
    const bool pre = stft_out ? (stft_pre && cfg->pre_emphasis > 0.0) : (cfg->pre_emphasis > 0.0);
    std::vector<float> warp_smem(w8_warp_floats(tb, p.n_mels) + 4, 0.f);
    W8Ctx c;
    // 16-byte align the warp tile like the device carve-up does
    float *ws = warp_smem.data();
    while (reinterpret_cast<uintptr_t>(ws) & 15) ws++;
    w8_carve(blob.data(), ws, tb, p.n_mels, c);
    c.alpha = p.alpha;
    c.win_a = cfg->window == DSPX_WINDOW_HANN ? 0.25f : (cfg->window == DSPX_WINDOW_HAMMING ? 0.27f : 0.5f);
    c.win_b = cfg->window == DSPX_WINDOW_HANN ? -0.25f : (cfg->window == DSPX_WINDOW_HAMMING ? -0.23f : 0.f);
    c.n_mels = p.n_mels;
    c.n_mfcc = p.n_mfcc;
    c.rounds = tb.rounds;
    c.cw_lanes = tb.cw_lanes;
    c.dct_row = tb.dct_row;
    c.lm_part = tb.lm_part;
    c.take = cfg->frame_length < e.P ? cfg->frame_length : e.P;
    const int r1 = tb.r1;
    const int units = r1 >= 8 ? r1 / 8 : 1;
    if (tb.x2) {
        // n_fft 4096 (feat_warp8_x2.cuh): one frame per item, the same phase order as feat_warp8_x2_kernel
        p.pairs_per_clip = (uint32_t)T;
        p.n_items = (uint32_t)(n_clips * T);
        const bool al4 = path == W8_X2_AL4;
        std::vector<W8Power4> pw4(32 * 2);
        for (uint32_t item = 0; item < p.n_items; item++) {
            w8x2_set_item(p, c, item);
            for (int lane = 0; lane < 32; lane++) {
                if (pre) { if (al4) w8x2_pass1<true, true>(c, lane); else w8x2_pass1<true, false>(c, lane); }
                else { if (al4) w8x2_pass1<false, true>(c, lane); else w8x2_pass1<false, false>(c, lane); }
            }
            for (int lane = 0; lane < 32; lane++) w8_pass2<16>(c, lane);
            for (int lane = 0; lane < 32; lane++)
                for (int w = 0; w < 2; w++) w8x2_pass3(c, lane, w, pw4[lane * 2 + w]);
            for (int lane = 0; lane < 32; lane++)
                for (int w = 0; w < 2; w++) w8x2_store_power(c, lane, w, pw4[lane * 2 + w]);
            for (int lane = 0; lane < 32; lane++) w8x2_mel_chunks(c, lane);
            for (int lane = 0; lane < 32; lane++) w8_logmel(c, lane);
            if (c.mfccA) {
                for (int c0 = 0; c0 < c.n_mfcc; c0 += c.cw_lanes) {
                    float2 acc[32];
                    for (int lane = 0; lane < 32; lane++) acc[lane] = w8_dct_partial(c, lane, c0);
                    for (int lane = 0; lane < 32; lane++) {
                        float2 t = acc[lane];
                        if (c.cw_lanes == 16) { t.x += acc[lane ^ 16].x; t.y += acc[lane ^ 16].y; }
                        w8_dct_store(c, lane, c0, t);
                    }
                }
            }
        }
        return DSPX_OK;
    }
    std::vector<W8Power> pw(32 * 2);
    // the device kernel computes window / twiddles on the feature path and loads them in STFT mode: replay the same
#define W8_P1(R, PRE_, SH_) do { if (p.stft) w8_pass1<R, PRE_, SH_, false>(c, lane); else if (u4) w8_pass1<R, PRE_, false, false, true>(c, lane); else w8_pass1<R, PRE_, SH_, true>(c, lane); } while (0)
    for (uint32_t item = 0; item < p.n_items; item++) {
        if (rtab) w8_set_item<false, true>(p, c, item);
        else w8_set_item(p, c, item);
        for (int lane = 0; lane < 32; lane++) {
            if (r1 == 4 && share) { if (pre) W8_P1(4, true, true); else W8_P1(4, false, true); }
            else if (r1 == 4) { if (pre) W8_P1(4, true, false); else W8_P1(4, false, false); }
            else if (r1 == 8 && share) { if (pre) W8_P1(8, true, true); else W8_P1(8, false, true); }
            else if (r1 == 8) { if (pre) W8_P1(8, true, false); else W8_P1(8, false, false); }
            else if (u4) { if (pre) w8_pass1<16, true, false, false, true>(c, lane); else w8_pass1<16, false, false, false, true>(c, lane); }
            else { if (pre) w8_pass1<16, true, false, false>(c, lane); else w8_pass1<16, false, false, false>(c, lane); }
        }
        for (int lane = 0; lane < 32; lane++) {
            if (r1 == 4) w8_pass2<4>(c, lane);
            else if (r1 == 8) w8_pass2<8>(c, lane);
            else w8_pass2<16>(c, lane);
        }
        if (p.stft) {
            for (int lane = 0; lane < 32; lane++)
                for (int w = 0; w < units; w++) {
                    if (r1 == 4) w8_pass3_stft<4>(c, lane, w);
                    else if (r1 == 8) w8_pass3_stft<8>(c, lane, w);
                    else w8_pass3_stft<16>(c, lane, w);
                }
            continue;
        }
        for (int lane = 0; lane < 32; lane++)
            for (int w = 0; w < units; w++) {
                if (r1 == 4) w8_pass3<4>(c, lane, w, pw[lane * 2 + w]);
                else if (r1 == 8) w8_pass3<8>(c, lane, w, pw[lane * 2 + w]);
                else w8_pass3<16>(c, lane, w, pw[lane * 2 + w]);
            }
        for (int lane = 0; lane < 32; lane++)
            for (int w = 0; w < units; w++) {
                if (r1 == 4) w8_store_power<4>(c, lane, w, pw[lane * 2 + w]);
                else if (r1 == 8) w8_store_power<8>(c, lane, w, pw[lane * 2 + w]);
                else w8_store_power<16>(c, lane, w, pw[lane * 2 + w]);
            }
        for (int lane = 0; lane < 32; lane++) w8_mel_chunks(c, lane);
        for (int lane = 0; lane < 32; lane++) w8_logmel(c, lane);
        if (c.mfccA || c.eacc) {
            for (int c0 = 0; c0 < c.n_mfcc; c0 += c.cw_lanes) {
                float2 acc[32];
                for (int lane = 0; lane < 32; lane++) acc[lane] = w8_dct_partial(c, lane, c0);
                for (int lane = 0; lane < 32; lane++) {
                    float2 t = acc[lane];
                    if (c.cw_lanes == 16) { t.x += acc[lane ^ 16].x; t.y += acc[lane ^ 16].y; }    // the device's shuffle
                    w8_dct_store(c, lane, c0, t);
                }
            }
        }
    }
    return DSPX_OK;
}

int emu_features_warp8(const dspx_config *cfg, const float *clips, int64_t n_clips, int64_t clip_len,
                       int64_t clip_stride, float *logmel, float *mfcc, float *stft_out, int stft_pre)
{
    return emu_warp8(cfg, clips, n_clips, clip_len, clip_stride, logmel, mfcc, stft_out, stft_pre, nullptr);
}

// The RAGGED variant over a flat float32 buffer and a dspx_ragged_layout table: outputs [total_frames, ...].
int emu_features_warp8_ragged(const dspx_config *cfg, const float *samples, const dspx_ragged_clip *table, int64_t n_clips,
                              float *logmel, float *mfcc)
{
    return emu_warp8(cfg, samples, n_clips, 0, 0, logmel, mfcc, nullptr, 0, table);
}

// Exhaustive check of the fused PCM16 normalisation (w8_pcm_to_float): for every peak m in [1, 32768] and every sample
// |s| <= m, the value the feature kernel feeds to the transform must equal NumPy's float32 (s / 32768) / (m / 32768).
// Returns the number of mismatches (0 expected) and the number of pairs through *total.
long long emu_pcm16_quotient_mismatches(long long *total)
{
    long long bad = 0, n = 0;
#pragma omp parallel for reduction(+ : bad, n) schedule(dynamic, 64)
    for (int m = 1; m <= 32768; m++) {
        const float fm = (float)m, r = 1.0f / fm, peak = fm * (1.0f / 32768.0f);
        for (int s = -m; s <= m; s++) {
            if (s > 32767) continue;
            const float ref = ((float)s * (1.0f / 32768.0f)) / peak;
            if (dspx::w8_pcm_to_float(s, fm, r) != ref) bad++;
            n++;
        }
    }
    if (total) *total = n;
    return bad;
}

}  // extern "C"
