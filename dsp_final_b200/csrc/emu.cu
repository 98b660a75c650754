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
#include "resample.cuh"
#include "decode.cuh"
#include "flac.cuh"
#include "retrieval_select.cuh"
#include "feat_select.cuh"

namespace dspx {
void set_error(const char *, ...) {}
const char *get_error() { return ""; }
}  // namespace dspx

using namespace dspx;

// A plan as dspx_plan_create derives it (plan_derive), without the device uploads
struct EmuPlan : dspx_plan {
    ~EmuPlan() { warp8_release(this); }
};

// The warp8 tables of a configuration, also where they do not fit in shared memory (the plan then uses the generic kernel)
static int emu_warp8_tables(const dspx_config *cfg, std::vector<float> &blob, W8Tables &tb)
{
    dspx_config gc = *cfg;
    gc.kernel = DSPX_KERNEL_GENERIC;
    EmuPlan pl;
    const int rc = plan_derive(&gc, &pl);
    if (rc != DSPX_OK) return rc;
    if (!warp8_supported(&pl)) return DSPX_EUNSUPPORTED;
    warp8_build_tables(&pl, blob, tb);
    return DSPX_OK;
}

extern "C" {

// Replays feat_generic_kernel.  stft_out != NULL selects the complex-spectrum mode.
int emu_features_generic(const dspx_config *cfg, const float *clips, int64_t n_clips, int64_t clip_len,
                         int64_t clip_stride, int stft_mode, int stft_pre, float *logmel, float *mfcc, float *stft_out,
                         int frames_per_cta_override)
{
    dspx_config gc = *cfg;
    gc.kernel = DSPX_KERNEL_GENERIC;
    EmuPlan pl;
    int rc = plan_derive(&gc, &pl);
    if (rc != DSPX_OK) return rc;
    const HostTables &h = pl.host;
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
    p.take = stft_mode ? pl.take_stft : pl.take_feat;
    p.P = pl.P;
    p.M = pl.M;
    p.n_bins = pl.n_bins;
    p.n_stages = pl.n_stages;
    for (int i = 0; i < 16; i++) p.radix[i] = pl.radix[i];
    p.n_mels = cfg->n_mels;
    p.n_mfcc = cfg->n_mfcc;
    int G = 1024 / pl.M;
    if (G < 1) G = 1;
    if (G > 16) G = 16;
    p.G = G;
    const int64_t groups = (T + G - 1) / G;
    int64_t gpc = frames_per_cta_override > 0 ? (frames_per_cta_override + G - 1) / G : groups;
    p.frames_per_cta = (int)(gpc * G);
    p.ctas_per_clip = (int)((T + p.frames_per_cta - 1) / p.frames_per_cta);
    p.pre = stft_mode ? (stft_pre && cfg->pre_emphasis > 0.0) : (cfg->pre_emphasis > 0.0);
    p.alpha = (float)cfg->pre_emphasis;
    p.window = h.window32.data();
    p.tw = h.tw.data();
    p.fb_start = h.fb_start.data();
    p.fb_cnt = h.fb_cnt.data();
    p.fb_off = h.fb_off.data();
    p.fb_w = h.fb_w.data();
    p.dct2 = h.dct2_32.data();
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
    std::vector<float> blob;
    W8Tables tb{};
    const int rc = emu_warp8_tables(cfg, blob, tb);
    if (rc != DSPX_OK) return rc;
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

// The CTA shapes a plan of feat_warp8_kernel can launch (warp8_shapes): out = {table bytes, shared memory of the 8-,
// 20-, 12- and 10-warp configurations (0 where one does not fit), 8-warp CTAs per SM, first-pass radix, x2 (n_fft 4096)}
int emu_warp8_shapes(const dspx_config *cfg, int64_t *out)
{
    std::vector<float> blob;
    W8Tables tb{};
    const int rc = emu_warp8_tables(cfg, blob, tb);
    if (rc != DSPX_OK) return rc;
    const W8Shapes s = warp8_shapes(tb, cfg->n_mels);
    out[0] = (int64_t)tb.total * 4; out[1] = s.smem; out[2] = s.smem_wide; out[3] = s.smem_mid; out[4] = s.smem_r16;
    out[5] = s.ctas_per_sm; out[6] = tb.r1; out[7] = tb.x2;
    return DSPX_OK;
}

// Replays feat_warp8_kernel: one "warp" at a time, each phase run for lanes 0..31 in turn
// (a __syncwarp() separates the phases on the device).  rtab != NULL replays the RAGGED variant over a
// dspx_ragged_layout table (clip_len and clip_stride unused).
static int emu_warp8(const dspx_config *cfg, const float *clips, int64_t n_clips, int64_t clip_len,
                     int64_t clip_stride, float *logmel, float *mfcc, float *stft_out, int stft_pre,
                     const dspx_ragged_clip *rtab)
{
    EmuPlan pl;
    if (plan_derive(cfg, &pl) != DSPX_OK || pl.kernel != DSPX_KERNEL_WARP8 || (!rtab && clip_len < cfg->frame_length))
        return DSPX_EUNSUPPORTED;
    const int64_t T = rtab ? 0 : 1 + (clip_len - cfg->frame_length) / cfg->hop_length;
    // the variant the library would launch
    const W8Path path = warp8_select(&pl, clips, clip_stride, DSPX_DTYPE_F32, rtab != nullptr, n_clips, T,
                                     stft_out ? W8_WANT_STFT : W8_WANT_FEATURES);
    if (path == W8_GENERIC || path == W8_UNSUPPORTED) return DSPX_EUNSUPPORTED;
    const bool u4 = path == W8_U4, share = path == W8_SHARE;
    W8PlanData &pd = *static_cast<W8PlanData *>(pl.fast_host);
    const W8Tables &tb = pd.tb;
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
    p.tables = pd.blob.data();
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
    w8_carve(pd.blob.data(), ws, tb, p.n_mels, c);
    c.alpha = p.alpha;
    c.win_a = cfg->window == DSPX_WINDOW_HANN ? 0.25f : (cfg->window == DSPX_WINDOW_HAMMING ? 0.27f : 0.5f);
    c.win_b = cfg->window == DSPX_WINDOW_HANN ? -0.25f : (cfg->window == DSPX_WINDOW_HAMMING ? -0.23f : 0.f);
    c.n_mels = p.n_mels;
    c.n_mfcc = p.n_mfcc;
    c.rounds = tb.rounds;
    c.cw_lanes = tb.cw_lanes;
    c.dct_row = tb.dct_row;
    c.lm_part = tb.lm_part;
    c.take = pl.take_feat;
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

static int emu_resampler(int64_t up, int64_t down, const float *window, int64_t n_window, RsGeom &g, std::vector<float> &tab,
                         bool &identity)
{
    if (up < 1 || down < 1) return DSPX_EINVAL;
    int64_t a = up, b = down;
    while (b) { const int64_t r = a % b; a = b; b = r; }
    up /= a;
    down /= a;
    identity = up == 1 && down == 1;
    g.up = up;
    g.down = down;
    if (identity) return DSPX_OK;
    int P = 0;
    int64_t remove = 0;
    if (!rs_build_table(up, down, window, n_window, tab, &P, &remove)) return DSPX_EINVAL;
    if (!rs_geometry(up, down, P, remove, MAX_OPTIN_SMEM, &g)) return DSPX_EINVAL;
    return DSPX_OK;
}

// Tile geometry of a ratio: out[0..7] = P, S, NR, W, RS, smem bytes, U, remove.
int emu_resample_shape(int64_t up, int64_t down, const float *window, int64_t n_window, int64_t *out)
{
    RsGeom g;
    std::vector<float> tab;
    bool identity = false;
    const int rc = emu_resampler(up, down, window, n_window, g, tab, identity);
    if (rc != DSPX_OK) return rc;
    const int64_t v[8] = {g.P, g.S, g.NR, g.W, g.RS, (int64_t)g.smem, g.U, g.remove};
    for (int i = 0; i < 8; i++) out[i] = v[i];
    return DSPX_OK;
}

// Replays resample_poly_kernel (or resample_copy_kernel) and resample_normalize_kernel through the kernel's tile
// decomposition: each tile's inputs and table rows are staged (rs_stage_row, rs_stage_phase) into a buffer of exactly the
// kernel's dynamic shared-memory size, then every (work item, lane) runs rs_group.  table != NULL: ragged batch (n_in, in_stride, out_stride unused).
int emu_resample(int64_t up, int64_t down, const float *window, int64_t n_window, const void *in, int dtype, int64_t n_clips,
                 int64_t n_in, int64_t in_stride, int normalize, float *out, int64_t out_stride, const dspx_resample_clip *table)
{
    RsGeom g;
    std::vector<float> tab;
    bool identity = false;
    const int rc = emu_resampler(up, down, window, n_window, g, tab, identity);
    if (rc != DSPX_OK) return rc;
    if (dtype != DSPX_DTYPE_F32 && dtype != DSPX_DTYPE_PCM16) return DSPX_EINVAL;
    const RsBatch b{in, dtype == DSPX_DTYPE_PCM16, n_in, in_stride, out, out_stride, table};
    for (int64_t clip = 0; clip < n_clips; clip++) {
        const RsClip c = rs_clip(b, g, clip);
        unsigned peak = 0;
        if (identity) {
            for (int64_t i = 0; i < c.n_out; i++) {
                c.out[i] = rs_load(c.in, b.pcm, i);
                peak = std::max(peak, rs_abs_bits(c.out[i]));
            }
        } else {
            const int64_t tiles = rs_tiles(g, c.n_out);
            for (int64_t tile = 0; tile < tiles; tile++) {
                const RsTile t = rs_tile(g, tile);
                std::vector<float> smem(g.smem / sizeof(float));
                float *ts = smem.data() + (int64_t)g.NR * g.RS;
                for (int r = 0; r < g.NR; r++) rs_stage_row(g, t, c, b.pcm, r, smem.data() + (int64_t)r * g.RS, 0, 1);
                for (int s = 0; s < t.S; s++) rs_stage_phase(g, t, tab.data(), s, ts + (int64_t)s * g.P, 0, 1);
                for (int item = 0; item < rs_items(g, t); item++)
                    for (int lane = 0; lane < 32; lane++) peak = std::max(peak, rs_group(g, t, c, smem.data(), ts, item, lane));
            }
        }
        if (normalize)
            for (int64_t i = 0; i < c.n_out; i++) c.out[i] = rs_normalize(c.out[i], peak);
    }
    return DSPX_OK;
}

// Replays wav_decode_kernel through the kernel's tile decomposition: each tile's input bytes are staged (dec_stage) into
// a buffer of exactly the kernel's dynamic shared-memory size, decoded frame by frame (dec_frames) into the output
// staging part of that buffer and stored (dec_store); with normalize, the peak pass over every tile of the batch
// comes first, as on the device.  table: a dspx_decode_layout table; in / out as for dspx_decode_ragged.
int emu_decode(const void *in, const dspx_decode_clip *table, int64_t n_clips, int normalize, float *out)
{
    for (int64_t i = 0; i < n_clips; i++)
        if (dec_bytes(table[i].dtype) == 0 || table[i].channels < 1 || table[i].channels > DSPX_MAX_CHANNELS ||
            table[i].n_frames < 1 || table[i].in_offset % 16 || table[i].out_start % 4)
            return DSPX_EINVAL;
    const unsigned char *src = static_cast<const unsigned char *>(in);
    std::vector<unsigned> peaks(n_clips, 0u);
    const int passes[2] = {normalize ? DEC_PEAK : DEC_STORE, DEC_NORM};
    for (int p = 0; p < (normalize ? 2 : 1); p++)
        for (int64_t i = 0; i < n_clips; i++) {
            const dspx_decode_clip &r = table[i];
            const DecWork w = dec_work(r, passes[p]);
            for (int64_t tile = 0; tile < dec_tiles(r); tile++) {
                const DecTile t = dec_tile(r, src, out, tile);
                if (w.divide) {
                    dec_divide(t, peaks[i], 0, 1);
                    continue;
                }
                std::vector<unsigned char> smem(DEC_SMEM);
                unsigned char *xs = smem.data();
                float *ys = reinterpret_cast<float *>(xs + DEC_IN_BYTES);
                dec_stage(t, xs, 0, 1);
                const unsigned pk = dec_frames(r, t, xs, ys, w.store, w.normalize, peaks[i], 0, 1);
                if (w.peak) peaks[i] = std::max(peaks[i], pk);
                if (w.store) dec_store(t, ys, 0, 1);
            }
        }
    return DSPX_OK;
}

// Replays flac_frame_kernel and flac_mix_kernel frame by frame: fl_frame decodes each frame into a heap buffer of
// exactly its integers' size (block_size x channels x 4 or 8 bytes) with a coefficient scratch of the kernel's size,
// then fl_mix_frame writes its outputs; with normalize, fl_divide runs after every frame's peak is folded, as on the
// device.  Tables from dspx_flac_layout; in / out / status as for dspx_flac_decode.
int emu_flac_decode(const void *in, const dspx_flac_file *files, int64_t n_files, const dspx_flac_frame *frames,
                    int64_t n_frames, int normalize, float *out, int32_t *status)
{
    for (int64_t f = 0; f < n_frames; f++)
        if (frames[f].file < 0 || frames[f].file >= n_files || frames[f].assignment < 0 || frames[f].assignment > 10 ||
            frames[f].block_size < 1 || frames[f].block_size > FL_MAX_BLOCK)
            return DSPX_EINVAL;
    uint16_t table[256];
    for (int i = 0; i < 256; i++) table[i] = fl_crc16_entry(i);
    const unsigned char *src = static_cast<const unsigned char *>(in);
    std::vector<std::vector<char>> samples(n_frames);
    for (int64_t f = 0; f < n_frames; f++) {
        const dspx_flac_frame &fr = frames[f];
        const int bps = files[fr.file].bps;
        samples[f].resize((size_t)fr.block_size * fl_channels(fr.assignment) * (fl_wide(bps) ? 8 : 4));
        std::vector<int32_t> coef(FL_MAX_ORDER + 1);
        status[f] = fl_frame(src + files[fr.file].in_offset, fr, bps, samples[f].data(), coef.data(), table);
    }
    std::vector<unsigned> peaks(n_files, 0u);
    for (int64_t f = 0; f < n_frames; f++)
        if (!status[f]) {
            const dspx_flac_frame &fr = frames[f];
            const dspx_flac_file &file = files[fr.file];
            peaks[fr.file] = std::max(peaks[fr.file],
                                      fl_mix_frame(fr, file.bps, samples[f].data(), out + file.out_start, false, 0u, 0, 1));
        }
    if (normalize)
        for (int64_t f = 0; f < n_frames; f++)
            if (!status[f]) fl_divide(frames[f], out + files[frames[f].file].out_start, peaks[frames[f].file], 0, 1);
    return DSPX_OK;
}

// The launch of a dspx_cosine_topk call (topk_select): out = {kernel (0 tensor-core filter, 1 FP32 filter, 2 float64),
// template argument, grid.x, grid.y, threads, dynamic shared memory, n_splits, rows_per_split}
int emu_topk_select(int64_t nq, int64_t ndb, int dim, int k, int sm_count, int64_t *out)
{
    if (nq < 0 || ndb < 1 || dim < 1 || k < 1 || sm_count < 1) return DSPX_EINVAL;
    const TopkLaunch L = topk_select(nq, ndb, dim, k, sm_count);
    const int64_t v[8] = {(int64_t)L.kernel, L.cw, L.grid.x, L.grid.y, L.threads, (int64_t)L.smem, L.n_splits, L.rows_per_split};
    for (int i = 0; i < 8; i++) out[i] = v[i];
    return DSPX_OK;
}

// The ranking workspace (topk_ws_carve): out = {offset, extent} of qn, dbn, pscore, pidx, qf, dbf, shared_thr and
// split_done, then the total (dspx_cosine_topk_workspace).  A region's extent runs to the next region's offset.
int emu_topk_workspace(int64_t nq, int64_t ndb, int dim, int k, int64_t *out)
{
    if (nq < 0 || ndb < 0 || dim < 1 || k < 1) return DSPX_EINVAL;
    char *const base = reinterpret_cast<char *>((uintptr_t)1 << 44);   // never dereferenced: only offsets are read
    TopkWs w;
    const size_t total = topk_ws_carve(nq, ndb, dim, k, base, &w);
    const char *p[9] = {(char *)w.qn, (char *)w.dbn, (char *)w.pscore, (char *)w.pidx, (char *)w.qf, (char *)w.dbf,
                        (char *)w.shared_thr, (char *)w.split_done, base + (total - 1024)};
    for (int i = 0; i < 8; i++) {
        out[2 * i] = p[i] - base;
        out[2 * i + 1] = p[i + 1] - p[i];
    }
    out[16] = (int64_t)total;
    return DSPX_OK;
}

// A plan as dspx_plan_create derives it; *kernel: the DSPX_KERNEL_* it runs
int emu_plan_create(const dspx_config *cfg, int *kernel, dspx_plan **out)
{
    EmuPlan *pl = new EmuPlan();
    const int rc = plan_derive(cfg, pl);
    if (rc != DSPX_OK) { delete pl; return rc; }
    *kernel = pl->kernel;
    *out = pl;
    return DSPX_OK;
}

void emu_plan_destroy(dspx_plan *pl) { delete static_cast<EmuPlan *>(pl); }

static FeatBatch emu_batch(const void *samples, int dtype, int normalize, int64_t n_clips, int64_t clip_len, int64_t stride,
                           const dspx_ragged_clip *table)
{
    return table ? FeatBatch{samples, dtype, normalize, n_clips, 0, 0, table, nullptr}
                 : FeatBatch{samples, dtype, normalize, n_clips, clip_len, stride, nullptr, nullptr};
}

// The steps of a feature call (feat_steps): out = {path (W8Path), convert, peaks, fused, mfcc_scratch, per_clip, T}.
// samples is only compared for alignment; table != NULL: a ragged batch (clip_len and stride unused).
int emu_feat_steps(const dspx_plan *pl, const void *samples, int dtype, int normalize, int64_t n_clips, int64_t clip_len,
                   int64_t stride, const dspx_ragged_clip *table, int want_mfcc, int want_embed, int64_t *out)
{
    const FeatSteps s = feat_steps(pl, emu_batch(samples, dtype, normalize, n_clips, clip_len, stride, table), want_mfcc != 0,
                                   want_embed != 0);
    const int64_t v[7] = {s.path, s.convert, s.peaks, s.fused, s.mfcc_scratch, s.per_clip, s.T};
    for (int i = 0; i < 7; i++) out[i] = v[i];
    return DSPX_OK;
}

// The workspace of that call (feat_ws_carve) in a buffer that starts base_offset bytes past a 256-byte boundary, moved
// up to the next one as the entry points do (ws_align): out = offsets from the buffer's start of rpairs, peaks, eacc,
// mfcc and f32 (-1 where a step needs none), then the carve's size (dspx_features_ragged_workspace).
int emu_feat_workspace(const dspx_plan *pl, const void *samples, int dtype, int normalize, int64_t n_clips, int64_t clip_len,
                       int64_t stride, const dspx_ragged_clip *table, int want_mfcc, int want_embed, int64_t base_offset,
                       int64_t *out)
{
    if (base_offset < 0) return DSPX_EINVAL;
    const FeatBatch b = emu_batch(samples, dtype, normalize, n_clips, clip_len, stride, table);
    const FeatSteps s = feat_steps(pl, b, want_mfcc != 0, want_embed != 0);
    char *const buf = reinterpret_cast<char *>(((uintptr_t)1 << 44) + base_offset);   // never dereferenced
    FeatWs w;
    const size_t total = feat_ws_carve(pl, b, s, ws_align(buf), &w);
    const char *p[5] = {(char *)w.rpairs, (char *)w.peaks, (char *)w.eacc, (char *)w.mfcc, (char *)w.f32};
    for (int i = 0; i < 5; i++) out[i] = p[i] ? p[i] - buf : -1;
    out[5] = (int64_t)total;
    return DSPX_OK;
}

}  // extern "C"
