// feat_warp8.cuh -- the headline kernel: warp-autonomous, radix-8, packed-f32x2 fused
// pre-emphasis -> frame -> window -> FFT -> |X|^2 -> mel -> log -> DCT for frame_length =
// n_fft = 1024 (the configuration BASELINE.json quotes its metric on).
//
// Reference ops replaced: src/dsp/mfcc.py:86-109 (log_mel_spectrogram, mfcc) with everything
// they call: stft.py:27-56 (framing, window), fft.py:27-77 (rfft), mfcc.py:32-83 (mel, DCT).
//
// Design (DESIGN.md "warp8 kernel" has the long form):
//  * One WARP owns two consecutive frames of a clip at a time and never synchronises with any
//    other warp: no __syncthreads in the main loop, only __syncwarp between FFT passes.
//  * The two frames ride in the two halves of Blackwell's packed FP32 instructions (FFMA2 /
//    FADD2 / FMUL2, sm_100+): every arithmetic instruction, shared-memory access and address
//    computation serves both frames; twiddles enter as scalar-broadcast operands.
//  * 1024 real samples are packed into a 512-point complex FFT = 8 x 8 x 8: three in-register
//    radix-8 passes, two exchanges through an 8 KB per-warp shared-memory tile addressed with an
//    XOR swizzle (128-bit accesses, conflict-free in all three access patterns).
//  * The last pass is laid out so that lane u holds bins k = u (mod 64) AND their mirror
//    images 512-k, so the packed-real split and |X|^2 need no further exchange.
//  * Samples are read straight from global memory (coalesced 8-byte loads of 256-byte rows; the
//    50% frame overlap is served by L1/L2), pre-emphasised with rounded mul + rounded sub exactly
//    like NumPy's float32 evaluation, and windowed in registers.
//  * mel projection = balanced (filter, part) work items over the power spectrum in shared
//    memory; log; DCT from a shared-memory table; features stored straight to HBM.
//
// The per-lane work between two __syncwarp()s is written as __host__ __device__ "lane phase"
// functions so that csrc/emu.cu can replay the exact same source on the CPU (tests only).
#pragma once

#include <algorithm>

#include "dspx_internal.cuh"

namespace dspx {

constexpr int W8_WARPS = 8;               // warps per CTA, two CTAs per SM (128 registers per thread)
#ifndef DSPX_W8_WIDE
#define DSPX_W8_WIDE 20
#endif
constexpr int W8_WARPS_WIDE = DSPX_W8_WIDE;
#ifndef DSPX_W8_R16
#define DSPX_W8_R16 10
#endif
constexpr int W8_WARPS_MID = 12;         // tables and tiles too large for 20 warps (128 mels): one 12-warp CTA instead of one of 8
constexpr int W8_WARPS_R16 = DSPX_W8_R16;           // n_fft 2048: one CTA per SM with as many 16 KB tiles as fit beside the tables         // or one 20-warp CTA per SM (<= 102 registers): more warps in flight to
                                          // cover the shared-memory pipe; +6 % on the feature path, worse for STFT mode



// ---- packed two-frame arithmetic (x = frame A, y = frame B) ------------------------------
#if defined(__CUDA_ARCH__)
DSPX_HD float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
DSPX_HD float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
DSPX_HD float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
DSPX_HD float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
#else
DSPX_HD float2 add2(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
DSPX_HD float2 sub2(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
DSPX_HD float2 mul2(float2 a, float2 b) { return make_float2(a.x * b.x, a.y * b.y); }
DSPX_HD float2 fma2(float2 a, float2 b, float2 c) { return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
#endif
DSPX_HD float2 bc2(float s) { return make_float2(s, s); }
DSPX_HD float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }

// (re, im) *= (c + i s) for both frames; c, s scalar
DSPX_HD void cmul2(float2 &re, float2 &im, float c, float s)
{
    const float2 cc = bc2(c), ss = bc2(s);
    const float2 r = fma2(neg2(im), ss, mul2(re, cc));
    im = fma2(im, cc, mul2(re, ss));
    re = r;
}

// 8-point forward DFT in registers (decimation in frequency), natural order in and out.
// 52 packed adds + 4 packed muls.
DSPX_HD void dft8(float2 (&re)[8], float2 (&im)[8])
{
    const float h = 0.70710678118654752440f;
    float2 ar[8], ai[8];
#pragma unroll
    for (int n = 0; n < 4; n++) {
        ar[n] = add2(re[n], re[n + 4]);
        ai[n] = add2(im[n], im[n + 4]);
        ar[n + 4] = sub2(re[n], re[n + 4]);
        ai[n + 4] = sub2(im[n], im[n + 4]);
    }
    // odd branch twiddles: a5 *= (1 - i)/sqrt2, a6 *= -i, a7 *= (-1 - i)/sqrt2
    {
        const float2 r5 = add2(ar[5], ai[5]), i5 = sub2(ai[5], ar[5]);
        ar[5] = mul2(r5, bc2(h));
        ai[5] = mul2(i5, bc2(h));
        const float2 r6 = ai[6], i6 = neg2(ar[6]);
        ar[6] = r6;
        ai[6] = i6;
        const float2 r7 = sub2(ai[7], ar[7]), i7 = add2(ar[7], ai[7]);
        ar[7] = mul2(r7, bc2(h));
        ai[7] = mul2(i7, bc2(-h));
    }
#pragma unroll
    for (int o = 0; o < 2; o++) {          // o = 0: even outputs from a0..a3, o = 1: odd from a4..a7
        const int b = 4 * o;
        const float2 s02r = add2(ar[b], ar[b + 2]), s02i = add2(ai[b], ai[b + 2]);
        const float2 d02r = sub2(ar[b], ar[b + 2]), d02i = sub2(ai[b], ai[b + 2]);
        const float2 s13r = add2(ar[b + 1], ar[b + 3]), s13i = add2(ai[b + 1], ai[b + 3]);
        const float2 d13r = sub2(ai[b + 1], ai[b + 3]);                 // (c1 - c3) * (-i)
        const float2 d13i = sub2(ar[b + 3], ar[b + 1]);
        re[o] = add2(s02r, s13r);
        im[o] = add2(s02i, s13i);
        re[o + 2] = add2(d02r, d13r);
        im[o + 2] = add2(d02i, d13i);
        re[o + 4] = sub2(s02r, s13r);
        im[o + 4] = sub2(s02i, s13i);
        re[o + 6] = sub2(d02r, d13r);
        im[o + 6] = sub2(d02i, d13i);
    }
}

// 4-point forward DFT (8 packed adds)
DSPX_HD void dft4(float2 (&re)[4], float2 (&im)[4])
{
    const float2 s02r = add2(re[0], re[2]), s02i = add2(im[0], im[2]);
    const float2 d02r = sub2(re[0], re[2]), d02i = sub2(im[0], im[2]);
    const float2 s13r = add2(re[1], re[3]), s13i = add2(im[1], im[3]);
    const float2 d13r = sub2(im[1], im[3]), d13i = sub2(re[3], re[1]);      // (v1 - v3) * (-i)
    re[0] = add2(s02r, s13r); im[0] = add2(s02i, s13i);
    re[1] = add2(d02r, d13r); im[1] = add2(d02i, d13i);
    re[2] = sub2(s02r, s13r); im[2] = sub2(s02i, s13i);
    re[3] = sub2(d02r, d13r); im[3] = sub2(d02i, d13i);
}

// 16-point forward DFT = 4 x 4: DFT-4 over n2 (n = n1 + 4 n2), twiddle W16^(n1 k2), DFT-4 over n1;
// output X[k2 + 4 k1].  Natural order in and out.
DSPX_HD void dft16(float2 (&re)[16], float2 (&im)[16])
{
    const float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f, h = 0.70710678118654752440f;
    float2 yr[4][4], yi[4][4];                       // [n1][k2]
#pragma unroll
    for (int n1 = 0; n1 < 4; n1++) {
        float2 tr[4] = {re[n1], re[n1 + 4], re[n1 + 8], re[n1 + 12]};
        float2 ti[4] = {im[n1], im[n1 + 4], im[n1 + 8], im[n1 + 12]};
        dft4(tr, ti);
#pragma unroll
        for (int k2 = 0; k2 < 4; k2++) { yr[n1][k2] = tr[k2]; yi[n1][k2] = ti[k2]; }
    }
    // twiddles W16^(n1 k2) = exp(-2 pi i n1 k2 / 16): (cos, -sin)
    cmul2(yr[1][1], yi[1][1], c1, -s1);              // W^1
    cmul2(yr[1][2], yi[1][2], h, -h);                // W^2
    cmul2(yr[1][3], yi[1][3], s1, -c1);              // W^3
    cmul2(yr[2][1], yi[2][1], h, -h);                // W^2
    { const float2 r = yi[2][2], i = neg2(yr[2][2]); yr[2][2] = r; yi[2][2] = i; }   // W^4 = -i
    cmul2(yr[2][3], yi[2][3], -h, -h);               // W^6
    cmul2(yr[3][1], yi[3][1], s1, -c1);              // W^3
    cmul2(yr[3][2], yi[3][2], -h, -h);               // W^6
    cmul2(yr[3][3], yi[3][3], -c1, s1);              // W^9 = -W^1
#pragma unroll
    for (int k2 = 0; k2 < 4; k2++) {
        float2 tr[4] = {yr[0][k2], yr[1][k2], yr[2][k2], yr[3][k2]};
        float2 ti[4] = {yi[0][k2], yi[1][k2], yi[2][k2], yi[3][k2]};
        dft4(tr, ti);
#pragma unroll
        for (int k1 = 0; k1 < 4; k1++) { re[k2 + 4 * k1] = tr[k1]; im[k2 + 4 * k1] = ti[k1]; }
    }
}

DSPX_HD void dftn(float2 (&re)[4], float2 (&im)[4]) { dft4(re, im); }
DSPX_HD void dftn(float2 (&re)[8], float2 (&im)[8]) { dft8(re, im); }
DSPX_HD void dftn(float2 (&re)[16], float2 (&im)[16]) { dft16(re, im); }

// exchange-tile address (in float4 units) of element (k_a, x, c): x = b before pass 2, k_b after
DSPX_HD int w8_addr(int ka, int x, int c) { return ((ka * 8 + x) << 3) | (c ^ (ka & 7)); }

constexpr int W8_CHUNK = 8;               // bins per mel chunk
constexpr int W8_CSTRIDE = 8;             // float2 slots per chunk in the power tile: chunks are contiguous, so the
                                          // scattered power stores of consecutive bins stay conflict-free; the reads
                                          // are de-conflicted by a per-lane rotation (w8_mel_chunks)
constexpr int W8_WROW = 20;               // floats per chunk row of the weight table (a0 b0 .. a7 b7 + pad)

// Geometry for first-pass radix R1: M = 64 R1 complex points (n_fft = 128 R1), J = 8 R1 output residues.
template <int R1> struct W8Geo {
    static constexpr int M = 64 * R1, P = 128 * R1, J = 8 * R1;
    static constexpr int LOG_R1 = R1 == 4 ? 2 : (R1 == 8 ? 3 : 4);
    static constexpr int SETS2 = R1 / 4;                 // radix-8 transforms per lane in pass 2
    static constexpr int UNITS = R1 >= 8 ? R1 / 8 : 1;   // mirror-pair units per lane in pass 3
    static constexpr int ACTIVE3 = R1 >= 8 ? 32 : 16;    // lanes that own a unit in pass 3
};

struct W8Tables {            // offsets (in floats) into the packed table blob / shared memory
    int win, tw1, tw2, ptw, ppos, cw, cflag, fdesc, dct, total;
    int rounds, n_slots;     // mel chunks: 32 lanes x rounds (rounds odd)
    int n_segs;              // run pieces emitted by the mel chunks
    int seg_slots;           // float2 slots of the area that holds their sums (filter ranges start at even slots)
    int cw_lanes;            // DCT: coefficient lanes per part (16 or 32)
    int dct_row;             // DCT: floats per (part, coefficient) table row (multiple of 4, odd number of 16-byte units)
    int lm_part;             // log-mel row: float2 slots per part (filters f = part, part + parts, ... ; multiple of 2)
    int tile_floats;         // per-warp exchange / power tile
    int r1;                  // first-pass radix (4, 8, 16)
    int x2;                  // n_fft 4096 (feat_warp8_x2.cuh): one frame per item, its even / odd samples in the (A, B) halves
    int win4, ptw2, ppos4;   // x2 tables: window per float4 of samples, exp(-2 pi i k / 4096), four tile positions per slot
};

struct W8Params {
    const float *clips;
    int64_t n_clips, clip_stride, n_frames;
    uint32_t pairs_per_clip, n_items;
    int hop, n_mels, n_mfcc, prefetch, share, take;
    float alpha;
    float win_a, win_b;      // see W8Ctx
    W8Tables tb;
    const float *tables;     // global copy of the blob
    float *logmel, *mfcc;    // either may be null
    int64_t lm_ts, lm_fs;    // log-mel strides between frames / filters ([B,T,M]: M,1; [B,1,M,T]: 1,T)
    float2 *stft;            // STFT mode: complex spectrum [n_clips, n_frames, M + 1]
    long long *eacc;         // embedding accumulators [n_clips][2][n_mfcc] (fixed point, see w8_embed_accumulate) or null
    const int *peaks;        // PCM variant: max |sample| of every clip (peak normalisation), null = divide by 32768 only
    // RAGGED variant (appended: the fields above keep their offsets): items are global frame-pair indices
    const dspx_ragged_clip *rtab;   // per-clip start, n_frames, first_frame (dspx_ragged_layout)
    const uint32_t *rpairs;         // [n_clips + 1] first pair of every clip, then the total: the array the search walks
};

struct W8Ctx {               // everything one warp needs for one frame pair
    const float2 *win, *tw1, *tw2, *ptw;
    const int2 *ppos;
    const float4 *win4;      // x2 tables (n_fft 4096)
    const float2 *ptw2;
    const int4 *ppos4;
    const float *cw;
    const int *cflag;
    const int2 *fdesc;       // {first slot, count} of every filter's run-piece sums
    const float *dct;
    float4 *xbuf;
    float2 *pbuf, *seg, *lm, *dsc;
    const float *fa, *fb;    // first sample of frame A / frame B
    int firstA, firstB;      // frame starts at sample 0 of its clip (no predecessor for pre-emphasis)
    float alpha;
    float win_a, win_b;      // 0.5 w[n] = win_a + win_b cos(2 pi n / P): hann (0.25, -0.25), hamming (0.27, -0.23), rect (0.5, 0)
    int n_mels, n_mfcc, rounds, cw_lanes, dct_row, lm_part, validB;
    int take;                // samples of a frame that enter the transform (= n_fft except in the general variant)
    float *logmelA, *logmelB, *mfccA, *mfccB;   // rows of the two frames (null when not requested)
    int64_t lm_fs;
    float2 *stftA, *stftB;   // STFT mode: rows of the two frames
    long long *eacc;         // this clip's embedding accumulators: sum x [n_mfcc], sum x^2 [n_mfcc]
    float pcm_m, pcm_r;      // PCM variant: the clip's max |sample| m (0 = no normalisation) and 1 / m
};

struct W8Power {             // |X|^2 of the bins one pass-3 unit owns, carried across the syncwarp
    float2 lo[9], hi[9];
};

// The per-warp tile holds, in turn, the FFT exchange data (4 M floats) and then the power spectrum in
// chunk order followed by the mel segments, the log-mel row and the DCT scratch (all live only after
// the last FFT pass has been read).
DSPX_HD int w8_warp_floats(const W8Tables &tb, int n_mels)
{
    (void)n_mels;
    return (tb.tile_floats + 3) & ~3;
}

// distance (float2 slots) between the two part rows of the log-mel row: = 8 (mod 16), so the 64-bit stores of the
// even filters (part 0) and the odd filters (part 1) of a half-warp fall into different halves of the bank space
DSPX_HD int w8_lm_stride(int lm_part) { return ((lm_part + 7) & ~15) + 8; }

DSPX_HD void w8_carve(float *tables_smem, float *warp_smem, const W8Tables &tb, int n_mels, W8Ctx &c)
{
    c.win = reinterpret_cast<const float2 *>(tables_smem + tb.win);
    c.tw1 = reinterpret_cast<const float2 *>(tables_smem + tb.tw1);
    c.tw2 = reinterpret_cast<const float2 *>(tables_smem + tb.tw2);
    c.ptw = reinterpret_cast<const float2 *>(tables_smem + tb.ptw);
    c.ppos = reinterpret_cast<const int2 *>(tables_smem + tb.ppos);
    c.win4 = reinterpret_cast<const float4 *>(tables_smem + tb.win4);
    c.ptw2 = reinterpret_cast<const float2 *>(tables_smem + tb.ptw2);
    c.ppos4 = reinterpret_cast<const int4 *>(tables_smem + tb.ppos4);
    c.cw = tables_smem + tb.cw;
    c.cflag = reinterpret_cast<const int *>(tables_smem + tb.cflag);
    c.fdesc = reinterpret_cast<const int2 *>(tables_smem + tb.fdesc);
    c.dct = tables_smem + tb.dct;
    c.xbuf = reinterpret_cast<float4 *>(warp_smem);
    c.pbuf = reinterpret_cast<float2 *>(warp_smem);
    // power tile: float2 (frame A, frame B) per bin, or one float per bin in the x2 (single frame) mode
    c.seg = c.pbuf + (tb.x2 ? (W8_CSTRIDE * tb.n_slots + 16) / 2 : (W8_CSTRIDE * tb.n_slots + 16));
    c.lm = c.seg + tb.seg_slots;                             // seg_slots is even: 16-byte aligned for the DCT's 128-bit loads
    c.dsc = c.lm + (32 / tb.cw_lanes) * w8_lm_stride(tb.lm_part);
}

// ---- window and first-pass twiddles without table loads (R1 <= 8) ---------------------------------------
// Both are functions of one angle per thread: u = exp(-2 pi i tid / M) (the k_a = 1 twiddle, one 8-byte load).
// Twiddles are its powers (depth-3 product tree); the window of row a, sample i is
// win_a + win_b cos(phi_i + 2 pi a / R1) with cos phi_0 = Re u, sin phi_0 = -Im u and phi_1 = phi_0 + 2 pi / P.
// The shared-memory pipe is the kernel's bottleneck; these ~90 FP32 instructions per frame pair replace 60 of its
// wavefronts (+5 % measured).  Rounding differs from the tables by a few 1e-7 (tolerance 1e-4).
DSPX_HD float2 w8_cmul(float2 a, float2 b) { return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x)); }

template <int R1> struct W8Trig {
    float2 C, S, D, E;                                 // (cos, sin)(phi_0 | phi_1) packed, and (C -+ S) / sqrt 2
    float2 u[R1 - 1];                                  // u^1 .. u^(R1-1)
    DSPX_HD explicit W8Trig(float2 u1)
    {
        constexpr float dc = R1 == 4 ? 0.99992470183914450299f : 0.99998117528260110909f;    // cos(2 pi / P), P = 128 R1
        constexpr float ds = R1 == 4 ? 0.01227153828571992608f : 0.00613588464915447536f;    // sin(2 pi / P)
        const float c0 = u1.x, s0 = -u1.y;
        C = make_float2(c0, fmaf(c0, dc, -s0 * ds));
        S = make_float2(s0, fmaf(s0, dc, c0 * ds));
        if constexpr (R1 == 8) {
            const float2 h = bc2(0.70710678118654752440f);
            D = mul2(sub2(C, S), h);
            E = mul2(add2(C, S), h);
        }
        u[0] = u1;
        u[1] = w8_cmul(u1, u1);
        u[2] = w8_cmul(u[1], u1);
        if constexpr (R1 == 8) {
            u[3] = w8_cmul(u[1], u[1]);
            u[4] = w8_cmul(u[3], u1);
            u[5] = w8_cmul(u[3], u[1]);
            u[6] = w8_cmul(u[3], u[2]);
        }
    }
    // (0.5 w[n], 0.5 w[n + 1]) for n = 128 a + 2 tid: cos(phi + 2 pi a / R1) is one of +-C, +-S, +-D, +-E
    DSPX_HD float2 window(int a, float wa, float wb) const
    {
        const int k = a * (8 / R1);                    // eighth-root index
        const float2 v = (k == 0 || k == 4) ? C : (k == 2 || k == 6) ? S : (k == 1 || k == 5) ? D : E;
        const bool neg = k == 2 || k == 3 || k == 4 || k == 5;      // cos(phi + k pi/4): C, D, -S, -E, -C, -D, S, E
        return fma2(v, bc2(neg ? -wb : wb), bc2(wa));
    }
};

template <int R1, bool TRIG, class Trig> DSPX_HD float2 w8_window_of(const W8Ctx &c, const Trig &t, int s, int a, int lane)
{
    if (TRIG) return t.window(a, c.win_a, c.win_b);
    return c.win[(s * R1 + a) * 32 + lane];
}
template <int R1, bool TRIG, class Trig> DSPX_HD float2 w8_twiddle_of(const W8Ctx &c, const Trig &t, int s, int ka, int lane)
{
    if (TRIG) return t.u[(ka - 1) % 7];
    return c.tw1[(s * (R1 - 1) + ka - 1) * 32 + lane];
}

// ---- PCM16 ingest inside the sample loads (general variant only; SURVEY 8f row f2) ---------------------------
// load_audio + normalize_audio (src/utils/audio.py:19-38) of a 16-bit PCM clip are x = s / 32768 and x / max|x|,
// i.e. the correctly rounded quotient s / m with m = max|s| (both scalings are exact).  q = s * (1/m) followed by one
// fma refinement, q' = q + (s - m q) / m, IS that quotient for every |s| <= m <= 32768: verified exhaustively
// (1 073 807 359 pairs, tests/test_host_and_abi.py::test_pcm16_quotient_is_exact), so the fused path feeds the
// transform bit-for-bit the samples dspx_pcm16_to_float writes -- without the float32 copy of the clips in HBM.
DSPX_HD float w8_pcm_to_float(int s, float m, float r)
{
    const float x = (float)s;
    if (m == 0.f) return x * (1.0f / 32768.0f);               // no normalisation, or an all-zero clip
    const float q = x * r;
    return fmaf(fmaf(-m, q, x), r, q);
}

template <bool PCM> struct W8Sample { using type = float; };
template <> struct W8Sample<true> { using type = int16_t; };

template <bool PCM>
DSPX_HD float w8_fetch(const typename W8Sample<PCM>::type *p, const W8Ctx &c)
{
    if (PCM) return w8_pcm_to_float((int)*p, c.pcm_m, c.pcm_r);
    return (float)*p;
}

// ---- phase A: load, pre-emphasis, window, radix-R1 over a, twiddle, store -----------------
// All loads of a set are issued before the first use (memory-level parallelism); the only
// sample without a predecessor is sample 0 of a clip (y[0] = x[0], src/dsp/mfcc.py:88).
// TRIG: window and twiddles computed (feature path, R1 <= 8) instead of loaded (STFT mode is HBM-bound and keeps
// the loads: the extra instructions cost it 2 %; R1 = 16 has no registers to spare)
// U4, the general variant: frames need not start on an 8-byte boundary (odd hop, odd clip stride, unaligned base) and
// may be shorter than the transform (frame_length < n_fft: zero padding, src/dsp/fft.py:34-36) or longer (truncation,
// fft.py:32-33).  The two samples of a lane are fetched with two 4-byte loads, each only if it lies inside the
// first c.take samples of the frame; the window comes from the table (zero past take).  Never combined with SHARE.
template <int R1, bool PRE, bool SHARE, bool TRIG, bool U4 = false, bool PCM = false>
DSPX_HD void w8_pass1(const W8Ctx &c, int lane)
{
    static_assert(!PCM || (U4 && !SHARE), "the PCM16 loads exist in the general variant only");
    if (SHARE) {
        // hop == n_fft / 2: frame B's rows 0..R1/2-1 are frame A's rows R1/2..R1-1.  Load the 3/2 R1
        // distinct rows once, pre-emphasise them once (scalar), and pair them up for the two frames.
        constexpr int SH = R1 / 2, NR = R1 + SH;
#pragma unroll
        for (int s = 0; s < 2; s++) {
            const int tid = lane + 32 * s;
            const float *pa = c.fa + 2 * tid;
            const float *ph = c.validB ? pa : pa - 128 * SH;             // no frame B: rows >= R1 replay frame A's rows
            float2 x[NR];
            float pv[NR];
#if defined(DSPX_ABL) && DSPX_ABL == 7        // timing only: no global sample loads at all
#pragma unroll
            for (int r = 0; r < NR; r++) { x[r] = make_float2(0.001f * (r + lane), 0.002f * (r - lane)); pv[r] = 0.003f * r; }
#else
#pragma unroll
            for (int r = 0; r < NR; r++) x[r] = *reinterpret_cast<const float2 *>((r >= R1 ? ph : pa) + 128 * r);
            if (PRE) {
#if defined(DSPX_ABL) && DSPX_ABL == 6        // timing only: no predecessor loads
#pragma unroll
                for (int r = 0; r < NR; r++) pv[r] = x[r].y;
#else
                const bool edge = c.firstA && tid == 0;
                pv[0] = *(edge ? pa : pa - 1);
                if (edge) pv[0] = 0.f;
#pragma unroll
                for (int r = 1; r < NR; r++) pv[r] = (r >= R1 ? ph : pa)[128 * r - 1];
#endif
            }
#endif
            float y0[NR], y1[NR];
#pragma unroll
            for (int r = 0; r < NR; r++) {
                y0[r] = x[r].x;
                y1[r] = x[r].y;
                if (PRE) {
                    y1[r] = DSPX_FSUB_RN(x[r].y, DSPX_FMUL_RN(c.alpha, x[r].x));
                    y0[r] = DSPX_FSUB_RN(x[r].x, DSPX_FMUL_RN(c.alpha, pv[r]));
                }
            }
            const W8Trig<(R1 <= 8 ? R1 : 8)> trig(c.tw1[(s * (R1 - 1)) * 32 + lane]);      // dead code unless TRIG
            float2 re[R1], im[R1];
#pragma unroll
            for (int a = 0; a < R1; a++) {
                const float2 w = w8_window_of<R1, TRIG>(c, trig, s, a, lane);    // (0.5 w[n], 0.5 w[n+1])
                re[a] = mul2(make_float2(y0[a], y0[a + SH]), bc2(w.x));
                im[a] = mul2(make_float2(y1[a], y1[a + SH]), bc2(w.y));
            }
            dftn(re, im);
            c.xbuf[w8_addr(0, tid >> 3, tid & 7)] = make_float4(re[0].x, re[0].y, im[0].x, im[0].y);
#pragma unroll
            for (int ka = 1; ka < R1; ka++) {
                const float2 w = w8_twiddle_of<R1, TRIG>(c, trig, s, ka, lane);
                cmul2(re[ka], im[ka], w.x, w.y);
                c.xbuf[w8_addr(ka, tid >> 3, tid & 7)] = make_float4(re[ka].x, re[ka].y, im[ka].x, im[ka].y);
            }
        }
        return;
    }
#pragma unroll
    for (int s = 0; s < 2; s++) {
        const int tid = lane + 32 * s;
        using S = typename W8Sample<PCM>::type;                               // float, or int16 (c.fa / c.fb then point at int16)
        const S *pa = reinterpret_cast<const S *>(c.fa) + 2 * tid, *pb = reinterpret_cast<const S *>(c.fb) + 2 * tid;
        float2 xa[R1], xb[R1];
        float pva[R1], pvb[R1];
#pragma unroll
        for (int a = 0; a < R1; a++) {
            if (U4) {
                const int n0 = 128 * a + 2 * tid;
                xa[a] = make_float2(n0 < c.take ? w8_fetch<PCM>(pa + 128 * a, c) : 0.f, n0 + 1 < c.take ? w8_fetch<PCM>(pa + 128 * a + 1, c) : 0.f);
                xb[a] = make_float2(n0 < c.take ? w8_fetch<PCM>(pb + 128 * a, c) : 0.f, n0 + 1 < c.take ? w8_fetch<PCM>(pb + 128 * a + 1, c) : 0.f);
            } else {
                xa[a] = *reinterpret_cast<const float2 *>(pa + 128 * a);
                xb[a] = *reinterpret_cast<const float2 *>(pb + 128 * a);
            }
        }
        if (PRE) {
            const bool edgeA = c.firstA && tid == 0, edgeB = c.firstB && tid == 0;
            const bool in0 = !U4 || 2 * tid < c.take;
            pva[0] = in0 ? w8_fetch<PCM>(edgeA ? pa : pa - 1, c) : 0.f;
            pvb[0] = in0 ? w8_fetch<PCM>(edgeB ? pb : pb - 1, c) : 0.f;
            if (edgeA) pva[0] = 0.f;
            if (edgeB) pvb[0] = 0.f;
#pragma unroll
            for (int a = 1; a < R1; a++) {
                const bool in = !U4 || 128 * a + 2 * tid < c.take;          // the sample this one precedes is inside the frame
                pva[a] = in ? w8_fetch<PCM>(pa + 128 * a - 1, c) : 0.f;
                pvb[a] = in ? w8_fetch<PCM>(pb + 128 * a - 1, c) : 0.f;
            }
        }
        const W8Trig<(R1 <= 8 ? R1 : 8)> trig(c.tw1[(s * (R1 - 1)) * 32 + lane]);      // unused (and dropped) for R1 = 16
        float2 re[R1], im[R1];
#pragma unroll
        for (int a = 0; a < R1; a++) {
            float2 y0 = make_float2(xa[a].x, xb[a].x), y1 = make_float2(xa[a].y, xb[a].y);
            if (PRE) {
                const float2 al = bc2(c.alpha);
                const float2 t0 = mul2(make_float2(pva[a], pvb[a]), al), t1 = mul2(y0, al);   // rounded products ...
                y1 = sub2(y1, t1);                                                          // ... rounded differences
                y0 = sub2(y0, t0);
            }
            const float2 w = w8_window_of<R1, TRIG>(c, trig, s, a, lane);       // (0.5 w[n], 0.5 w[n+1])
            re[a] = mul2(y0, bc2(w.x));
            im[a] = mul2(y1, bc2(w.y));
        }
        dftn(re, im);
        c.xbuf[w8_addr(0, tid >> 3, tid & 7)] = make_float4(re[0].x, re[0].y, im[0].x, im[0].y);
#pragma unroll
        for (int ka = 1; ka < R1; ka++) {
            const float2 w = w8_twiddle_of<R1, TRIG>(c, trig, s, ka, lane);     // exp(-2 pi i tid ka / M)
            cmul2(re[ka], im[ka], w.x, w.y);
            c.xbuf[w8_addr(ka, tid >> 3, tid & 7)] = make_float4(re[ka].x, re[ka].y, im[ka].x, im[ka].y);
        }
    }
}

// ---- phase B: radix-8 over b, in place, twiddle exp(-2 pi i c k_b / 64) ---------------------
template <int R1>
DSPX_HD void w8_pass2(const W8Ctx &c, int lane)
{
    const int cc = lane & 7;
    float2 tw[7];                                   // exp(-2 pi i c k_b / 64): the same for every set of this lane
#pragma unroll
    for (int kb = 1; kb < 8; kb++) tw[kb - 1] = c.tw2[(kb - 1) * 8 + cc];
#pragma unroll
    for (int s = 0; s < W8Geo<R1>::SETS2; s++) {
        const int ka = (lane >> 3) + 4 * s;
        float2 re[8], im[8];
#pragma unroll
        for (int b = 0; b < 8; b++) {
            const float4 v = c.xbuf[w8_addr(ka, b, cc)];
            re[b] = make_float2(v.x, v.y);
            im[b] = make_float2(v.z, v.w);
        }
        dft8(re, im);
        c.xbuf[w8_addr(ka, 0, cc)] = make_float4(re[0].x, re[0].y, im[0].x, im[0].y);
#pragma unroll
        for (int kb = 1; kb < 8; kb++) {
            cmul2(re[kb], im[kb], tw[kb - 1].x, tw[kb - 1].y);
            c.xbuf[w8_addr(ka, kb, cc)] = make_float4(re[kb].x, re[kb].y, im[kb].x, im[kb].y);
        }
    }
}

// packed-real split of one mirror pair (a = Z[k], b = Z[M-k]); the window carries the 1/2:
//   E = a + conj b, O = -i (a - conj b), T = W^k O, |X[k]|^2 = |E + T|^2, |X[M-k]|^2 = |E - T|^2
DSPX_HD void w8_split(float2 ar, float2 ai, float2 br, float2 bi, float2 w, float2 &plo, float2 &phi)
{
    const float2 er = add2(ar, br), ei = sub2(ai, bi);
    const float2 orr = add2(ai, bi), oi = sub2(br, ar);
    const float2 wr = bc2(w.x), wi = bc2(w.y);
    const float2 tr = fma2(neg2(oi), wi, mul2(orr, wr));
    const float2 ti = fma2(orr, wi, mul2(oi, wr));
    const float2 xr = add2(er, tr), xi = add2(ei, ti);
    const float2 yr = sub2(er, tr), yi = sub2(ei, ti);
    plo = fma2(xi, xi, mul2(xr, xr));
    phi = fma2(yi, yi, mul2(yr, yr));
}

DSPX_HD float2 sel2(bool p, float2 a, float2 b) { return p ? a : b; }

// bin index of slot m of pass-3 unit u (u = lane + 32 w); J = 8 R1 residues
DSPX_HD int w8_bin(int J, int u, int m)
{
    const int k0[9] = {0, J, 2 * J, 3 * J, 4 * J, J / 2, J / 2 + J, J / 2 + 2 * J, J / 2 + 3 * J};
    return u == 0 ? k0[m] : u + J * m;
}

// ---- phase C: radix-8 over c for residues j and J-j, split, power ---------------------------
// unit u pairs Z[u + J m] with its mirror Z[M - u - J m] = D2[7 - m]; unit 0 owns the two
// self-mirrored residues 0 and J/2: slots {0:(Z0,Z0) 1..3:(Z[Jm],Z[M-Jm]) 4:(Z[M/2],Z[M/2])
// 5..7:(Z[J/2+Jq],Z[M-J/2-Jq]) q=0..2} and a ninth slot for q = 3.
template <int R1>
DSPX_HD void w8_pass3(const W8Ctx &c, int lane, int w, W8Power &pw)
{
    using G = W8Geo<R1>;
    if (lane >= G::ACTIVE3) return;
    const int u = lane + 32 * w;
    const bool l0 = u == 0;
    const int j1 = u, j2 = l0 ? G::J / 2 : G::J - u;
    float2 r1[8], i1[8], r2[8], i2[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const float4 v = c.xbuf[w8_addr(j1 & (R1 - 1), j1 >> G::LOG_R1, q)];
        r1[q] = make_float2(v.x, v.y);
        i1[q] = make_float2(v.z, v.w);
        const float4 t = c.xbuf[w8_addr(j2 & (R1 - 1), j2 >> G::LOG_R1, q)];
        r2[q] = make_float2(t.x, t.y);
        i2[q] = make_float2(t.z, t.w);
    }
    dft8(r1, i1);          // Z[j1 + J m]
    dft8(r2, i2);          // Z[j2 + J m]
    const float2 *ptw = c.ptw + w * 9 * 32;
#pragma unroll
    for (int m = 0; m < 8; m++) {
        float2 ar = r1[m], ai = i1[m];
        if (m >= 5) { ar = sel2(l0, r2[m - 5], ar); ai = sel2(l0, i2[m - 5], ai); }
        const int b0 = m == 0 ? 0 : (m <= 4 ? 8 - m : 0);               // unit-0 partner index in D1 (m <= 4)
        float2 br, bi;
        if (m <= 4) { br = sel2(l0, r1[b0 & 7], r2[7 - m]); bi = sel2(l0, i1[b0 & 7], i2[7 - m]); }
        else { br = sel2(l0, r2[12 - m], r2[7 - m]); bi = sel2(l0, i2[12 - m], i2[7 - m]); }
        w8_split(ar, ai, br, bi, ptw[m * 32 + lane], pw.lo[m], pw.hi[m]);
    }
    if (l0) w8_split(r2[3], i2[3], r2[4], i2[4], ptw[8 * 32], pw.lo[8], pw.hi[8]);
}

// the spectrum is written once and never read back by this kernel: streaming (evict-first) stores keep
// L2 for the input rows that neighbouring frame pairs share (+2 % measured)
DSPX_HD void w8_stream_store(float2 *dst, float2 v)
{
#if defined(__CUDA_ARCH__)
    __stcs(dst, v);
#else
    *dst = v;
#endif
}

// ---- phase C': STFT mode -- same transforms and pairing, but the complex bins go straight to HBM ----
// X[k] = E + T, X[M-k] = conj(E - T); consecutive lanes hold consecutive bins: coalesced 8-byte stores.
DSPX_HD void w8_split_store(float2 ar, float2 ai, float2 br, float2 bi, float2 w, float2 *rowA, float2 *rowB,
                            int k, int mk, bool validB)
{
    const float2 er = add2(ar, br), ei = sub2(ai, bi);
    const float2 orr = add2(ai, bi), oi = sub2(br, ar);
    const float2 wr = bc2(w.x), wi = bc2(w.y);
    const float2 tr = fma2(neg2(oi), wi, mul2(orr, wr));
    const float2 ti = fma2(orr, wi, mul2(oi, wr));
    const float2 xr = add2(er, tr), xi = add2(ei, ti);
    const float2 yr = sub2(er, tr), yi = sub2(ti, ei);
    w8_stream_store(rowA + k, make_float2(xr.x, xi.x));
    w8_stream_store(rowA + mk, make_float2(yr.x, yi.x));
    if (validB) {
        w8_stream_store(rowB + k, make_float2(xr.y, xi.y));
        w8_stream_store(rowB + mk, make_float2(yr.y, yi.y));
    }
}

template <int R1>
DSPX_HD void w8_pass3_stft(const W8Ctx &c, int lane, int w)
{
    using G = W8Geo<R1>;
    if (lane >= G::ACTIVE3) return;
    const int u = lane + 32 * w;
    const bool l0 = u == 0;
    const int j1 = u, j2 = l0 ? G::J / 2 : G::J - u;
    float2 r1[8], i1[8], r2[8], i2[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const float4 v = c.xbuf[w8_addr(j1 & (R1 - 1), j1 >> G::LOG_R1, q)];
        r1[q] = make_float2(v.x, v.y);
        i1[q] = make_float2(v.z, v.w);
        const float4 t = c.xbuf[w8_addr(j2 & (R1 - 1), j2 >> G::LOG_R1, q)];
        r2[q] = make_float2(t.x, t.y);
        i2[q] = make_float2(t.z, t.w);
    }
    dft8(r1, i1);
    dft8(r2, i2);
    const float2 *ptw = c.ptw + w * 9 * 32;
    const bool vb = c.validB != 0;
#pragma unroll
    for (int m = 0; m < 8; m++) {
        float2 ar = r1[m], ai = i1[m];
        if (m >= 5) { ar = sel2(l0, r2[m - 5], ar); ai = sel2(l0, i2[m - 5], ai); }
        const int b0 = m == 0 ? 0 : (m <= 4 ? 8 - m : 0);
        float2 br, bi;
        if (m <= 4) { br = sel2(l0, r1[b0 & 7], r2[7 - m]); bi = sel2(l0, i1[b0 & 7], i2[7 - m]); }
        else { br = sel2(l0, r2[12 - m], r2[7 - m]); bi = sel2(l0, i2[12 - m], i2[7 - m]); }
        const int k = w8_bin(G::J, u, m);
        w8_split_store(ar, ai, br, bi, ptw[m * 32 + lane], c.stftA, c.stftB, k, G::M - k, vb);
    }
    if (l0) {
        const int k = w8_bin(G::J, 0, 8);
        w8_split_store(r2[3], i2[3], r2[4], i2[4], ptw[8 * 32], c.stftA, c.stftB, k, G::M - k, vb);
    }
}

// ---- phase D: power spectrum into the (re-used) tile, in mel-chunk order ---------------------------
// ppos[w][m][lane] = tile slots of bins k_m and M - k_m: bins of one mel chunk are contiguous,
// chunks sit W8_CSTRIDE slots apart, bins no filter uses go to a dump slot.
template <int R1>
DSPX_HD void w8_store_power(const W8Ctx &c, int lane, int w, const W8Power &pw)
{
    if (lane >= W8Geo<R1>::ACTIVE3) return;
    const int2 *ppos = c.ppos + w * 9 * 32;
#pragma unroll
    for (int m = 0; m < 8; m++) {
        const int2 p = ppos[m * 32 + lane];
        c.pbuf[p.x] = pw.lo[m];
        c.pbuf[p.y] = pw.hi[m];
    }
    if (lane + 32 * w == 0) {
        const int2 p = ppos[8 * 32];
        c.pbuf[p.x] = pw.lo[8];
        c.pbuf[p.y] = pw.hi[8];
    }
}

// ---- phase E: mel chunks ----------------------------------------------------------------------------
// Every bin k feeds (at most) filter g(k) with weight a_k and filter g(k)+1 with weight b_k
// (csrc/tables.cuh "bin view").  Runs of equal g are cut into chunks of 8 bins; lane l walks
// chunks l*R .. l*R+R-1, accumulating in registers while the run continues and dropping one
// (sum a P, sum b P) pair per run piece, each sum at the slot where its filter will read it.  Chunks are 64 B apart in the tile, so chunk parity picks
// the half of a 128-byte line and the lane reads its four 16-byte pieces rotated by (lane >> 1) & 3:
// the 128-bit loads of 8 neighbouring lanes hit 8 different bank groups (rounds is odd, so parity
// alternates with the lane).  The weight rows (80 B apart) are stored pre-rotated to match.
// Tile row of chunk ch = lane * rounds + r.  Neighbouring lanes must read rows of different parity (the two 64-byte
// halves of a 128-byte line): with an odd number of rounds the chunk index itself alternates, with an even number
// odd lanes swap their rows pairwise.
DSPX_HD int w8_chunk_row(int ch, int lane, int rounds) { return ch ^ (lane & ~rounds & 1); }
// The flag words (4 B) and weight rows (80 B) of a lane's chunks are consecutive; with an even number of rounds one
// more word / 16-byte unit per lane keeps the lane stride odd (conflict-free 32-bit and 128-bit loads).
DSPX_HD int w8_flag_index(int ch, int lane, int rounds) { return ch + (lane & -(~rounds & 1)); }
DSPX_HD int w8_cw_index(int ch, int lane, int rounds) { return ch * W8_WROW + 4 * (lane & -(~rounds & 1)); }

struct W8MelIn {                 // one chunk's operands: four 16-byte pieces of power values and of weights, and its flag word
    float4 p[4], w[4];
    int flag;
};

DSPX_HD void w8_mel_load(const W8Ctx &c, int lane, int r, W8MelIn &in)
{
    const int ch = lane * c.rounds + r;
    in.flag = c.cflag[w8_flag_index(ch, lane, c.rounds)];               // bit0 first, bit1 last, 8..19 / 20..31 slots of the sums
    const float4 *pp = reinterpret_cast<const float4 *>(c.pbuf + w8_chunk_row(ch, lane, c.rounds) * W8_CSTRIDE);
    const float4 *ww = reinterpret_cast<const float4 *>(c.cw + w8_cw_index(ch, lane, c.rounds));
    const int rot = (lane >> 1) & 3;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        in.p[q] = pp[(q + rot) & 3];                                    // (P0A P0B P1A P1B)
        in.w[q] = ww[q];                                                // (a0 b0 a1 b1)
    }
}

DSPX_HD void w8_mel_accumulate(const W8Ctx &c, const W8MelIn &in, float2 &sa, float2 &sb)
{
    // four independent chains (even / odd bins, a / b weights): short dependency depth
    float2 ca0 = make_float2(0.f, 0.f), cb0 = ca0, ca1 = ca0, cb1 = ca0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const float4 p = in.p[q], w = in.w[q];
        ca0 = fma2(make_float2(p.x, p.y), bc2(w.x), ca0);
        cb0 = fma2(make_float2(p.x, p.y), bc2(w.y), cb0);
        ca1 = fma2(make_float2(p.z, p.w), bc2(w.z), ca1);
        cb1 = fma2(make_float2(p.z, p.w), bc2(w.w), cb1);
    }
    const float2 ca = add2(ca0, ca1), cb = add2(cb0, cb1);
    if (in.flag & 1) { sa = ca; sb = cb; }
    else { sa = add2(sa, ca); sb = add2(sb, cb); }
    if (in.flag & 2) {
        c.seg[(in.flag >> 8) & 0xfff] = sa;
        c.seg[(unsigned)in.flag >> 20] = sb;
    }
}

DSPX_HD void w8_mel_chunks(const W8Ctx &c, int lane)
{
    float2 sa = make_float2(0.f, 0.f), sb = make_float2(0.f, 0.f);
#if defined(DSPX_MEL_PIPE)
    if (c.rounds == 3) {                                                // 40 mels at n_fft 512 / 1024: all loads of the next
        W8MelIn a, b;                                                   // round are in flight while this one is summed
        w8_mel_load(c, lane, 0, a);
        w8_mel_load(c, lane, 1, b);
        w8_mel_accumulate(c, a, sa, sb);
        w8_mel_load(c, lane, 2, a);
        w8_mel_accumulate(c, b, sa, sb);
        w8_mel_accumulate(c, a, sa, sb);
        return;
    }
#endif
    for (int r = 0; r < c.rounds; r++) {
        W8MelIn in;
        w8_mel_load(c, lane, r, in);
        w8_mel_accumulate(c, in, sa, sb);
    }
}

// ---- phase F: filter sums from the segments, floor, log, store log-mel ---------------------------------
DSPX_HD float w8_log(float x)
{
#if defined(__CUDA_ARCH__)
    return __logf(x);        // lg2.approx * ln 2: abs err < 1e-6 on values of magnitude 1..25 (tolerance 1e-4)
#else
    return logf(x);
#endif
}

// Sum of one filter's run pieces: they sit in consecutive slots starting at an even (16-byte aligned) slot, so three
// 128-bit loads fetch up to six of them and the count only predicates the adds (slots past the count hold other
// filters' sums or stale tile data and are never added).  Filters with more pieces finish in a loop.
DSPX_HD float2 w8_filter_sum(const W8Ctx &c, int2 d)
{
    const float4 *sp = reinterpret_cast<const float4 *>(c.seg + d.x);
    const float4 v0 = sp[0], v1 = sp[1], v2 = sp[2];
    float2 s0 = make_float2(0.f, 0.f), s1 = s0;
    if (d.y > 0) s0 = make_float2(v0.x, v0.y);
    if (d.y > 1) s1 = make_float2(v0.z, v0.w);
    if (d.y > 2) s0 = add2(s0, make_float2(v1.x, v1.y));
    if (d.y > 3) s1 = add2(s1, make_float2(v1.z, v1.w));
    if (d.y > 4) s0 = add2(s0, make_float2(v2.x, v2.y));
    if (d.y > 5) s1 = add2(s1, make_float2(v2.z, v2.w));
    for (int i = 6; i < d.y; i++) s0 = add2(s0, c.seg[d.x + i]);
    return add2(s0, s1);
}

// The row kept for the DCT is stored part-major -- slot (f % parts) * w8_lm_stride(lm_part) + f / parts with parts = 32 / cw_lanes --
// so that a DCT lane finds the filters it sums in consecutive slots; slots past n_mels are zeroed (the table is
// zero there too, but the tile still holds FFT data).  Two filters per lane are in flight at a time.
DSPX_HD void w8_logmel_one(const W8Ctx &c, int f, int psh, float2 s)
{
    const int slot = ((f & psh) ? w8_lm_stride(c.lm_part) : 0) + (f >> psh);
    if (f >= c.n_mels) {                                                // padding of the part rows
        c.lm[slot] = make_float2(0.f, 0.f);
        return;
    }
    const float2 v = make_float2(w8_log(fmaxf(s.x, 1e-10f)), w8_log(fmaxf(s.y, 1e-10f)));
    c.lm[slot] = v;
    if (c.logmelA) {
        c.logmelA[f * c.lm_fs] = v.x;
        if (c.validB) c.logmelB[f * c.lm_fs] = v.y;
    }
}

DSPX_HD void w8_logmel(const W8Ctx &c, int lane)
{
    const int psh = c.cw_lanes == 16 ? 1 : 0;                           // log2(parts)
    const int n_slots = c.lm_part << psh;
    const int2 *fd = c.fdesc;
    for (int f0 = lane; f0 < n_slots; f0 += 64) {
        const int f1 = f0 + 32;
        const int2 d0 = fd[f0 < c.n_mels ? f0 : 0], d1 = fd[f1 < c.n_mels ? f1 : 0];
        const float2 s0 = w8_filter_sum(c, d0), s1 = w8_filter_sum(c, d1);
        w8_logmel_one(c, f0, psh, s0);
        if (f1 < n_slots) w8_logmel_one(c, f1, psh, s1);
    }
}

// ---- phase G: DCT-II (table carries the factor 2) ------------------------------------------------------
// lane = part * cw_lanes + q: coefficient c0 + q, summed over the filters of `part` (f = part, part + parts, ...).
// The lane's table row and the part's log-mel row are both contiguous, so one 128-bit table load and two
// 128-bit (broadcast) log-mel loads feed four packed FMAs.  Table rows are an odd number of 16-byte units
// apart: the eight lanes of a quarter warp hit eight different bank groups.
DSPX_HD float2 w8_dct_partial(const W8Ctx &c, int lane, int c0)
{
    const int sh = c.cw_lanes == 16 ? 4 : 5;
    const int q = lane & (c.cw_lanes - 1), part = lane >> sh;
    const int blk = c0 >> sh;                                               // c0 is a multiple of cw_lanes
    const float4 *col = reinterpret_cast<const float4 *>(c.dct + (size_t)(blk * 32 + part * c.cw_lanes + q) * c.dct_row);
    const float4 *lm = reinterpret_cast<const float4 *>(c.lm + part * w8_lm_stride(c.lm_part));
    float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
    const int n4 = c.lm_part >> 2;                                          // whole groups of four filters
#pragma unroll 5
    for (int i = 0; i < n4; i++) {
        const float4 w = col[i], a = lm[2 * i], b = lm[2 * i + 1];          // a = lm[4i], lm[4i+1]; b = lm[4i+2], lm[4i+3]
        acc0 = fma2(make_float2(a.x, a.y), bc2(w.x), acc0);
        acc1 = fma2(make_float2(a.z, a.w), bc2(w.y), acc1);
        acc0 = fma2(make_float2(b.x, b.y), bc2(w.z), acc0);
        acc1 = fma2(make_float2(b.z, b.w), bc2(w.w), acc1);
    }
    if (c.lm_part & 2) {                                                    // lm_part is even: at most one pair left
        const float4 a = lm[2 * n4];
        const float2 w = *reinterpret_cast<const float2 *>(&col[n4]);
        acc0 = fma2(make_float2(a.x, a.y), bc2(w.x), acc0);
        acc1 = fma2(make_float2(a.z, a.w), bc2(w.y), acc1);
    }
    return add2(acc0, acc1);
}

// Clip embeddings (src/retrieval/retrieval.py:19-23: mean and population std of every coefficient over the frames)
// without an MFCC round trip through HBM: every frame adds x and x^2 to per-clip accumulators.  The sums are kept
// in 64-bit FIXED POINT (x * 2^32, x^2 * 2^20) so that the atomic adds commute exactly -- the result does not
// depend on the order in which warps finish -- and embed_finalize_kernel turns them into mean / std in float64.
// Range: |x| < 2^15 over 2^15 frames; resolution 2^-33 per x, 2^-21 per x^2 (std error < 1e-6 for std > 0.01).
constexpr double W8_EFIX1 = 4294967296.0, W8_EFIX2 = 1048576.0;

// Out of line on the device: the float64 / 64-bit integer code must not take part in the register allocation of
// the main loop (inlined it cost the headline kernel 36 bytes of spills); it runs once per frame pair on 13 lanes.
#if defined(__CUDA_ARCH__)
__device__ __noinline__
#else
inline
#endif
void w8_embed_accumulate(long long *eacc, int n_mfcc, int q, float xa, float xb)
{
    const double a = (double)xa, b = (double)xb;
    const long long s1 = (long long)llrint(a * W8_EFIX1) + (long long)llrint(b * W8_EFIX1);
    const long long s2 = (long long)llrint(a * a * W8_EFIX2) + (long long)llrint(b * b * W8_EFIX2);
#if defined(__CUDA_ARCH__)
    atomicAdd(reinterpret_cast<unsigned long long *>(eacc + q), (unsigned long long)s1);
    atomicAdd(reinterpret_cast<unsigned long long *>(eacc + n_mfcc + q), (unsigned long long)s2);
#else
    eacc[q] += s1;
    eacc[n_mfcc + q] += s2;
#endif
}

// total = the lane's sum plus its partner's (lane ^ 16) when two parts share a coefficient
DSPX_HD void w8_dct_store(const W8Ctx &c, int lane, int c0, float2 total)
{
    const int q = c0 + lane;
    if (lane < c.cw_lanes && q < c.n_mfcc) {
        if (c.mfccA) {
            c.mfccA[q] = total.x;
            if (c.validB) c.mfccB[q] = total.y;
        }
        if (c.eacc) w8_embed_accumulate(c.eacc, c.n_mfcc, q, total.x, c.validB ? total.y : 0.f);
    }
}

#if defined(__CUDACC__)
// rtab (ragged batches): every clip's own frame count instead of n_frames
__global__ void embed_finalize_kernel(const long long *eacc, int64_t n_clips, int64_t n_frames, int n_coef, float *out,
                                      const dspx_ragged_clip *rtab = nullptr)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_clips * n_coef) return;
    const int64_t clip = i / n_coef;
    const int q = (int)(i - clip * n_coef);
    if (rtab) n_frames = rtab[clip].n_frames;
    const long long *e = eacc + clip * 2 * n_coef;
    const double mean = (double)e[q] / W8_EFIX1 / (double)n_frames;
    const double ex2 = (double)e[n_coef + q] / W8_EFIX2 / (double)n_frames;
    const double var = ex2 - mean * mean;
    out[clip * 2 * n_coef + q] = (float)mean;
    out[clip * 2 * n_coef + n_coef + q] = (float)sqrt(var > 0.0 ? var : 0.0);
}
#endif

// RAGGED: the clip that holds global frame pair `item` -- the last one whose first pair is <= item (binary search over
// rpairs, which is strictly increasing: every clip has at least one frame)
DSPX_HD uint32_t w8_ragged_clip(const W8Params &p, uint32_t item)
{
    uint32_t lo = 0, hi = (uint32_t)p.n_clips;                // rpairs[lo] <= item < rpairs[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (p.rpairs[mid] <= item) lo = mid;
        else hi = mid;
    }
    return lo;
}

// set the per-item fields of the context (item = clip * pairs_per_clip + pair; RAGGED: item = rpairs[clip] + pair)
template <bool PCM = false, bool RAGGED = false>
DSPX_HD void w8_set_item(const W8Params &p, W8Ctx &c, uint32_t item)
{
    if (RAGGED) {
        const uint32_t clip = w8_ragged_clip(p, item), pair = item - p.rpairs[clip];
        const dspx_ragged_clip &rc = p.rtab[clip];
        const int64_t tA = 2 * (int64_t)pair, tB = tA + 1;
        c.validB = tB < rc.n_frames;
        using S = typename W8Sample<PCM>::type;
        const S *base = reinterpret_cast<const S *>(p.clips) + rc.start;
        c.fa = reinterpret_cast<const float *>(base + tA * p.hop);
        c.fb = c.validB ? reinterpret_cast<const float *>(base + tB * p.hop) : c.fa;
        if (PCM) {
            const int m = p.peaks ? p.peaks[clip] : 0;
            c.pcm_m = (float)m;
            c.pcm_r = m > 0 ? 1.0f / (float)m : 0.f;
        }
        c.firstA = pair == 0;                                 // pre-emphasis restarts at sample 0 of every clip
        c.firstB = c.validB ? 0 : c.firstA;
        const int64_t rowA = rc.first_frame + tA, rowB = rowA + 1;
        c.logmelA = p.logmel ? p.logmel + rowA * p.n_mels : nullptr;
        c.logmelB = c.logmelA ? c.logmelA + p.n_mels : nullptr;
        c.lm_fs = 1;
        c.mfccA = p.mfcc ? p.mfcc + rowA * p.n_mfcc : nullptr;
        c.mfccB = p.mfcc ? p.mfcc + rowB * p.n_mfcc : nullptr;
        c.stftA = c.stftB = nullptr;
        c.eacc = p.eacc ? p.eacc + (int64_t)clip * 2 * p.n_mfcc : nullptr;
        return;
    }
    const uint32_t clip = item / p.pairs_per_clip, pair = item - clip * p.pairs_per_clip;
    const int64_t tA = 2 * (int64_t)pair, tB = tA + 1;
    c.validB = tB < p.n_frames;
    using S = typename W8Sample<PCM>::type;                  // strides and hops count samples of the clip's own type
    const S *base = reinterpret_cast<const S *>(p.clips) + (int64_t)clip * p.clip_stride;
    c.fa = reinterpret_cast<const float *>(base + tA * p.hop);
    c.fb = c.validB ? reinterpret_cast<const float *>(base + tB * p.hop) : c.fa;
    if (PCM) {
        const int m = p.peaks ? p.peaks[clip] : 0;
        c.pcm_m = (float)m;
        c.pcm_r = m > 0 ? 1.0f / (float)m : 0.f;              // IEEE division: the correctly rounded reciprocal
    }
    c.firstA = pair == 0;
    c.firstB = c.validB ? 0 : c.firstA;        // a missing frame B replays frame A
    const int64_t rowA = (int64_t)clip * p.n_frames + tA, rowB = rowA + 1;
    c.logmelA = p.logmel ? p.logmel + (int64_t)clip * p.n_frames * p.n_mels + tA * p.lm_ts : nullptr;
    c.logmelB = c.logmelA ? c.logmelA + p.lm_ts : nullptr;
    c.lm_fs = p.lm_fs;
    c.mfccA = p.mfcc ? p.mfcc + rowA * p.n_mfcc : nullptr;
    c.mfccB = p.mfcc ? p.mfcc + rowB * p.n_mfcc : nullptr;
    const int64_t n_bins = 64 * p.tb.r1 + 1;
    c.stftA = p.stft ? p.stft + rowA * n_bins : nullptr;
    c.stftB = c.stftA ? c.stftA + n_bins : nullptr;
    c.eacc = p.eacc ? p.eacc + (int64_t)clip * 2 * p.n_mfcc : nullptr;
}

// the whole per-item sequence; SYNC is __syncwarp() on the device and a no-op in the lane-loop replay
#if defined(__CUDACC__)
// pull the next item's samples towards L2 while this one is being transformed
template <bool RAGGED = false>
__device__ __forceinline__ void w8_prefetch(const W8Params &p, uint32_t item, int lane, int n_fft, int elem = 4)
{
    if (item >= p.n_items) return;
    const char *base;
    if (RAGGED) {
        const uint32_t clip = w8_ragged_clip(p, item);
        base = reinterpret_cast<const char *>(p.clips) + (p.rtab[clip].start + 2 * (int64_t)(item - p.rpairs[clip]) * p.hop) * elem;
    } else {
        const uint32_t clip = item / p.pairs_per_clip, pair = item - clip * p.pairs_per_clip;
        base = reinterpret_cast<const char *>(p.clips) + ((int64_t)clip * p.clip_stride + 2 * (int64_t)pair * p.hop) * elem;
    }
    const int span = (p.hop + n_fft) * elem;                   // bytes covered by the frame pair
    for (int off = lane * 128; off < span; off += 32 * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
}

// EMB: accumulate clip embeddings (w8_embed_accumulate); a template switch so that the plain feature kernels keep
// their register allocation (the extra pointer alone pushed the 96-register headline variant into spills).
// RAGGED: clips of different lengths (w8_set_item); a switch for the same reason.
template <int R1, bool PRE, bool STFT, bool SHARE, int NW, bool EMB = false, bool U4 = false, bool PCM = false,
          bool RAGGED = false>
__global__ void __launch_bounds__(NW * 32, (R1 == 16 || NW > 8) ? 1 : 2) feat_warp8_kernel(const W8Params p)
{
    using G = W8Geo<R1>;
    extern __shared__ __align__(16) float w8_smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wf = w8_warp_floats(p.tb, p.n_mels);
    // constant tables: global -> shared, once per CTA; zero the per-warp areas (pad slots of the
    // power tile are read with zero weights and must hold finite numbers)
    {
        const float4 *src = reinterpret_cast<const float4 *>(p.tables);
        float4 *dst = reinterpret_cast<float4 *>(w8_smem);
        for (int i = tid; i < p.tb.total / 4; i += NW * 32) dst[i] = src[i];
        float4 *z = reinterpret_cast<float4 *>(w8_smem + p.tb.total);
        for (int i = tid; i < NW * wf / 4; i += NW * 32) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();
    W8Ctx c;
    w8_carve(w8_smem, w8_smem + p.tb.total + warp * wf, p.tb, p.n_mels, c);
    c.alpha = p.alpha;
    c.win_a = p.win_a;
    c.win_b = p.win_b;
    c.n_mels = p.n_mels;
    c.n_mfcc = p.n_mfcc;
    c.rounds = p.tb.rounds;
    c.cw_lanes = p.tb.cw_lanes;
    c.dct_row = p.tb.dct_row;
    c.lm_part = p.tb.lm_part;
    c.take = p.take;
    const uint32_t n_warps = gridDim.x * NW;
    for (uint32_t item = blockIdx.x * NW + warp; item < p.n_items; item += n_warps) {
        w8_set_item<PCM, RAGGED>(p, c, item);
        if (!EMB) c.eacc = nullptr;
        w8_pass1<R1, PRE, SHARE, (!STFT && R1 <= 8 && !U4), U4, PCM>(c, lane);
        if (p.prefetch) w8_prefetch<RAGGED>(p, item + n_warps, lane, G::P, PCM ? 2 : 4);
        __syncwarp();
#if !defined(DSPX_ABL) || DSPX_ABL != 5
        w8_pass2<R1>(c, lane);
        __syncwarp();
#endif
        if (STFT) {
#pragma unroll
            for (int w = 0; w < G::UNITS; w++) w8_pass3_stft<R1>(c, lane, w);
            __syncwarp();                   // the tile is rewritten by the next item's first pass
            continue;
        }
        W8Power pw[G::UNITS];
#if defined(DSPX_ABL) && DSPX_ABL == 5
#pragma unroll
        for (int w = 0; w < G::UNITS; w++)
#pragma unroll
            for (int m = 0; m < 9; m++) pw[w].lo[m] = pw[w].hi[m] = make_float2(1.f + lane, 2.f + m);
#else
#pragma unroll
        for (int w = 0; w < G::UNITS; w++) w8_pass3<R1>(c, lane, w, pw[w]);
#endif
        __syncwarp();                       // every lane has read its inputs: the tile may become P[]
#if defined(DSPX_ABL) && DSPX_ABL == 4      // timing only: FFT passes alone (keep the power values alive)
        {
            float2 s = make_float2(0.f, 0.f);
#pragma unroll
            for (int m = 0; m < 9; m++) s = add2(s, add2(pw[0].lo[m], pw[0].hi[m]));
            if (s.x == 123.456f && c.mfccA) c.mfccA[0] = s.y;
            continue;
        }
#endif
#pragma unroll
        for (int w = 0; w < G::UNITS; w++) w8_store_power<R1>(c, lane, w, pw[w]);
        __syncwarp();
#if defined(DSPX_ABL) && DSPX_ABL == 3
        continue;
#endif
        w8_mel_chunks(c, lane);
        __syncwarp();
#if defined(DSPX_ABL) && DSPX_ABL == 2
        continue;
#endif
        w8_logmel(c, lane);
        __syncwarp();
#if defined(DSPX_ABL) && DSPX_ABL == 1
        continue;
#endif
        if (c.mfccA || c.eacc) {
            for (int c0 = 0; c0 < c.n_mfcc; c0 += c.cw_lanes) {
                float2 acc = w8_dct_partial(c, lane, c0);
                if (c.cw_lanes == 16) {
                    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16);
                    acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
                }
                w8_dct_store(c, lane, c0, acc);
            }
            __syncwarp();                   // the log-mel row is rewritten by the next item
        }
    }
}
#endif

// ---- host side: table blob, support check, launch -------------------------------------------------
// n_fft 4096 runs the 2048-point machinery (radix 16) on the even and the odd samples of a frame at once
inline bool warp8_x2(const dspx_plan *pl) { return pl->P == 4096; }
inline int warp8_radix(const dspx_plan *pl) { return pl->P == 512 ? 4 : (pl->P == 1024 ? 8 : ((pl->P == 2048 || pl->P == 4096) ? 16 : 0)); }

inline bool warp8_supported(const dspx_plan *pl)
{
    return warp8_radix(pl) != 0 && pl->cfg.frame_length >= 2 &&
           pl->cfg.n_mels <= 256 && pl->cfg.n_mfcc <= 128 && pl->host.two_band_ok;
}

// ---- which kernel runs a call ------------------------------------------------------------------------------------
// What the call asks for: log-mel / MFCC, embeddings without an MFCC output (accumulated inside the kernel, EMB), or
// the complex STFT.
enum W8Want { W8_WANT_FEATURES, W8_WANT_EMBED, W8_WANT_STFT };

enum W8Path {
    W8_GENERIC,       // feat_generic_kernel
    W8_X2,            // feat_warp8_x2_kernel (n_fft 4096)
    W8_X2_AL4,        //   with 16-byte loads: frame_length >= n_fft, hop and row stride multiples of 4, 16-byte aligned base
    W8_ALIGNED,       // feat_warp8_kernel with 8-byte loads: frame_length = n_fft, every frame on the 8-byte grid
    W8_SHARE,         //   and the two frames of a pair share rows: hop = n_fft / 2 (not at radix 16, whose 24 distinct
                      //   rows in flight would not fit its register budget)
    W8_U4,            // feat_warp8_kernel with 4-byte loads: frames off the 8-byte grid or shorter than n_fft
    W8_PCM16,         // feat_warp8_kernel on int16 samples (4-byte loads, conversion in the loads)
    W8_UNSUPPORTED,   // no kernel does this: the entry point returns DSPX_EUNSUPPORTED before it enqueues anything
};

// The one place that picks the kernel of a call.  samples, row_stride (in samples of `dtype`), n_clips and T (frames
// per clip) describe an equal-length batch; a ragged batch ignores them: its layout holds fewer than 2^31 frame pairs
// and starts float32 clips on the 8-byte grid (dspx_ragged_layout, dspx_features_ragged).  A ragged batch on a plan
// without a ragged kernel (the generic kernel, n_fft 4096) gets W8_UNSUPPORTED and runs one clip at a time.
inline W8Path warp8_select(const dspx_plan *pl, const void *samples, int64_t row_stride, int dtype, bool ragged,
                           int64_t n_clips, int64_t T, W8Want want)
{
    const bool pcm = dtype == DSPX_DTYPE_PCM16, warp8 = pl->kernel == DSPX_KERNEL_WARP8 && !warp8_x2(pl);
    if (ragged && (!warp8 || want == W8_WANT_STFT)) return W8_UNSUPPORTED;        // the RAGGED variants have no STFT mode
    if (!warp8) {
        if (pcm || want == W8_WANT_EMBED) return W8_UNSUPPORTED;
        // x2 items are single frames, 32-bit
        if (pl->kernel != DSPX_KERNEL_WARP8 || want == W8_WANT_STFT || n_clips * T >= (int64_t)0x7fffffff) return W8_GENERIC;
        const bool al4 = pl->cfg.frame_length >= pl->P && !(pl->cfg.hop_length & 3) && !(row_stride & 3) &&
                         !(reinterpret_cast<uintptr_t>(samples) & 15);
        return al4 ? W8_X2_AL4 : W8_X2;
    }
    const bool fits = ragged || n_clips * ((T + 1) / 2) < (int64_t)0x7fffffff;      // items are 32-bit frame pairs
    if (pcm) return fits && want == W8_WANT_FEATURES ? W8_PCM16 : W8_UNSUPPORTED;
    // frames on the 8-byte grid: even hop, even row stride, 8-byte aligned base
    const bool aligned = fits && pl->cfg.frame_length == pl->P && !(pl->cfg.hop_length & 1) &&
                         (ragged || (!(row_stride & 1) && !(reinterpret_cast<uintptr_t>(samples) & 7)));
    const W8Path fast = 2 * pl->cfg.hop_length == pl->P && warp8_radix(pl) != 16 ? W8_SHARE : W8_ALIGNED;
    if (want == W8_WANT_EMBED) return aligned ? fast : W8_UNSUPPORTED;
    if (want == W8_WANT_STFT) return aligned && pl->take_stft == pl->P ? fast : W8_GENERIC;
    return aligned ? fast : (fits ? W8_U4 : W8_GENERIC);
}


// ---- bank-conflict-free table layouts (host side) -------------------------------------------------------
// 64-bit shared-memory accesses are served per half-warp, one wavefront per set of lanes that touch 16 different
// 8-byte bank pairs (slot mod 16); ncu's per-instruction wavefront counts of the round-1 layout follow this model
// exactly (profiles/r02_warp8_layout.md).  Two layouts are chosen with it when the plan is built:
//
//  * which of the 8 slots of its chunk row a bin occupies.  Bins are the edges of a bipartite graph between chunk
//    rows and (store instruction, half-warp, row parity) groups; both kinds of node need pairwise different slots on
//    their edges, and a bipartite graph with degrees <= 8 always has such an edge colouring with 8 colours (Koenig):
//    every power store then takes its minimum of two wavefronts.
//  * where the run-piece sums of every filter sit (w8_seg_layout below).
inline void w8_edge_colour(int na, int nb, const std::vector<std::pair<int, int>> &edges, int ncol, std::vector<int> &colour)
{
    std::vector<int> ea((size_t)na * ncol, -1), eb((size_t)nb * ncol, -1);     // edge that uses colour c at a node
    colour.assign(edges.size(), -1);
    for (size_t e = 0; e < edges.size(); e++) {
        const int a = edges[e].first, b = edges[e].second;
        int ca = -1, cb = -1;
        for (int c = ncol - 1; c >= 0; c--) {
            if (ea[(size_t)a * ncol + c] < 0) ca = c;
            if (eb[(size_t)b * ncol + c] < 0) cb = c;
        }
        if (ca < 0 || cb < 0) continue;                                        // an over-full node: left to the caller
        if (eb[(size_t)b * ncol + ca] >= 0) {
            // ca is taken at b: swap ca <-> cb along the alternating path that starts there (it cannot reach a)
            std::vector<int> path;
            int node = b, want = ca;
            bool at_b = true;
            for (;;) {
                const int nxt = at_b ? eb[(size_t)node * ncol + want] : ea[(size_t)node * ncol + want];
                if (nxt < 0) break;
                path.push_back(nxt);
                node = at_b ? edges[nxt].first : edges[nxt].second;
                at_b = !at_b;
                want = want == ca ? cb : ca;
            }
            for (int pe : path) {
                ea[(size_t)edges[pe].first * ncol + colour[pe]] = -1;
                eb[(size_t)edges[pe].second * ncol + colour[pe]] = -1;
            }
            for (int pe : path) {
                colour[pe] = colour[pe] == ca ? cb : ca;
                ea[(size_t)edges[pe].first * ncol + colour[pe]] = pe;
                eb[(size_t)edges[pe].second * ncol + colour[pe]] = pe;
            }
        }
        colour[e] = ca;
        ea[(size_t)a * ncol + ca] = (int)e;
        eb[(size_t)b * ncol + ca] = (int)e;
    }
}

// wavefronts of one 64-bit access of a warp: slots[lane] in 8-byte units, < 0 = lane inactive
inline int w8_wavefronts64(const int *slots)
{
    int total = 0;
    for (int h = 0; h < 2; h++) {
        int seen[16][16], cnt[16] = {0}, worst = 0;
        for (int l = 16 * h; l < 16 * h + 16; l++) {
            const int sl = slots[l];
            if (sl < 0) continue;
            const int b = sl & 15;
            bool dup = false;
            for (int i = 0; i < cnt[b]; i++) dup = dup || seen[b][i] == sl;
            if (!dup) seen[b][cnt[b]++] = sl;
            worst = std::max(worst, cnt[b]);
        }
        total += worst;
    }
    return total;
}

// One value a filter sums: the `a` or `b` sum of run piece (segment) seg, stored by `lane` in round `round`.
struct W8SegEntry { int seg, is_b, lane, round; };

// Slots of the run-piece sums.  Filter g reads its entries from consecutive slots starting at an even one
// (w8_filter_sum: 128-bit loads); the lanes that end a run piece in round r store their sums there (two 64-bit
// stores per round).  Starts are placed so that the 16-byte units of 8 consecutive filters differ mod 8 (the loads
// of a quarter-warp are conflict-free), the order inside each filter by a pairwise-swap descent on the modelled
// wavefronts of the stores.
inline void w8_seg_layout(const std::vector<std::vector<W8SegEntry>> &filt, int rounds, std::vector<int> &f_first,
                          std::vector<std::vector<int>> &order, int &end_slot)
{
    const int n = (int)filt.size();
    f_first.assign(n, 0);
    order.assign(n, {});
    int slot = 0;
    for (int g = 0; g < n; g++) {
        slot = (slot + 1) & ~1;
        if (!filt[g].empty()) {
            for (int tries = 0; tries < 8; tries++, slot += 2) {
                bool clash = false;
                for (int o = g - (g & 7); o < g; o++) clash = clash || (!filt[o].empty() && ((f_first[o] >> 1) & 7) == ((slot >> 1) & 7));
                if (!clash) break;
            }
        }
        f_first[g] = slot;
        slot += (int)filt[g].size();
        for (int i = 0; i < (int)filt[g].size(); i++) order[g].push_back(i);
    }
    end_slot = slot;
    auto cost = [&]() {
        std::vector<int> slots((size_t)rounds * 2 * 32, -1);
        for (int g = 0; g < n; g++)
            for (int j = 0; j < (int)order[g].size(); j++) {
                const W8SegEntry &e = filt[g][order[g][j]];
                slots[((size_t)e.round * 2 + e.is_b) * 32 + e.lane] = f_first[g] + j;
            }
        int c = 0;
        for (int i = 0; i < rounds * 2; i++) c += w8_wavefronts64(&slots[(size_t)i * 32]);
        return c;
    };
    int best = cost();
    for (int pass = 0; pass < 6; pass++) {
        bool improved = false;
        for (int g = 0; g < n; g++) {
            const int m = (int)order[g].size();
            for (int i = 0; i < m; i++)
                for (int j = i + 1; j < m; j++) {
                    std::swap(order[g][i], order[g][j]);
                    const int c = cost();
                    if (c < best) { best = c; improved = true; }
                    else std::swap(order[g][i], order[g][j]);
                }
        }
        if (!improved) break;
    }
}

inline void warp8_build_tables(const dspx_plan *pl, std::vector<float> &blob, W8Tables &tb)
{
    const HostTables &h = pl->host;
    const int R1 = warp8_radix(pl), M = 64 * R1, P = 2 * M, J = 8 * R1;
    const bool x2 = warp8_x2(pl);                           // then P = 2048 is the length of each half-rate sequence
    const int n_mels = pl->cfg.n_mels, n_mfcc = pl->cfg.n_mfcc, n_bins = x2 ? 2 * M + 1 : M + 1;
    const int units = R1 >= 8 ? R1 / 8 : 1;
    tb.x2 = x2 ? 1 : 0;
    // --- mel chunks from the bin view: runs of equal g, cut into chunks of 8 bins ---
    struct Chunk { int run, start, count; };
    std::vector<Chunk> chunks;
    std::vector<int> run_g;
    for (int k = 0; k < n_bins;) {
        const int g = h.bin_filt[k];
        if (g < 0) { k++; continue; }
        int e = k;
        while (e < n_bins && h.bin_filt[e] == g) e++;
        const int run = (int)run_g.size();
        run_g.push_back(g);
        for (int s = k; s < e; s += W8_CHUNK) chunks.push_back({run, s, std::min(W8_CHUNK, e - s)});
        k = e;
    }
    const int n_chunks = (int)chunks.size();
    int rounds = std::max(1, (n_chunks + 31) / 32);
    if (x2 && rounds % 2 == 0) rounds++;                 // the x2 reader has no row swap (w8_chunk_row): odd rounds only
    tb.r1 = R1;
    tb.rounds = rounds;
    tb.n_slots = 32 * rounds;
    tb.cw_lanes = n_mfcc <= 16 ? 16 : 32;
    const int dct_blocks = (n_mfcc + tb.cw_lanes - 1) / tb.cw_lanes;
    const int parts = 32 / tb.cw_lanes;
    tb.lm_part = (((n_mels + parts - 1) / parts) + 1) & ~1;             // filters per part, rounded up to a pair
    tb.dct_row = (tb.lm_part + 3) & ~3;
    if (((tb.dct_row / 4) & 1) == 0) tb.dct_row += 4;                    // odd number of 16-byte units per row
    auto al4 = [](int x) { return (x + 3) & ~3; };
    int off = 0;
    tb.win = off; off += 2 * R1 * 32 * 2;
    tb.tw1 = off; off += 2 * (R1 - 1) * 32 * 2;
    tb.tw2 = off; off += al4(7 * 8 * 2);
    tb.ptw = off; off += units * 9 * 32 * 2;
    tb.ppos = off; off += units * 9 * 32 * 2;
    tb.win4 = off; off += x2 ? 2 * R1 * 32 * 4 : 0;
    tb.ptw2 = off; off += x2 ? units * 9 * 32 * 2 : 0;
    tb.ppos4 = off; off += x2 ? units * 9 * 32 * 4 : 0;
    tb.cw = off; off += tb.n_slots * W8_WROW + 32 * 4;     // + the lane skew of even round counts (w8_cw_index)
    tb.cflag = off; off += tb.n_slots + 32;
    tb.fdesc = off; off += al4(n_mels * 2);
    tb.dct = off; off += dct_blocks * 32 * tb.dct_row;
    tb.total = al4(off);
    blob.assign(tb.total, 0.f);
    const double two_pi = 2.0 * M_PI;
    if (x2) {
        const int take = std::min(pl->cfg.frame_length, 2 * P);
        for (int s = 0; s < 2; s++)
            for (int a = 0; a < R1; a++)
                for (int l = 0; l < 32; l++)
                    for (int j = 0; j < 4; j++) {
                        const int n = 4 * ((l + 32 * s) + 64 * a) + j;   // sample of the 4096-point frame
                        blob[tb.win4 + ((s * R1 + a) * 32 + l) * 4 + j] = n < take ? (float)(0.5 * h.window[n]) : 0.f;
                    }
        for (int w = 0; w < units; w++)
            for (int m = 0; m < 9; m++)
                for (int l = 0; l < 32; l++) {
                    const double ang = -two_pi * (double)w8_bin(J, l + 32 * w, m) / (double)(2 * P);
                    blob[tb.ptw2 + ((w * 9 + m) * 32 + l) * 2] = (float)std::cos(ang);
                    blob[tb.ptw2 + ((w * 9 + m) * 32 + l) * 2 + 1] = (float)std::sin(ang);
                }
    }
    for (int s = 0; s < 2 && !x2; s++)
        for (int a = 0; a < R1; a++)
            for (int l = 0; l < 32; l++) {
                const int n = 128 * a + 2 * (l + 32 * s);
                const int take = std::min(pl->cfg.frame_length, P);          // zero padding / truncation (fft.py:32-36)
                blob[tb.win + ((s * R1 + a) * 32 + l) * 2] = n < take ? (float)(0.5 * h.window[n]) : 0.f;
                blob[tb.win + ((s * R1 + a) * 32 + l) * 2 + 1] = n + 1 < take ? (float)(0.5 * h.window[n + 1]) : 0.f;
            }
    for (int s = 0; s < 2; s++)
        for (int ka = 1; ka < R1; ka++)
            for (int l = 0; l < 32; l++) {
                const double ang = -two_pi * (double)((l + 32 * s) * ka) / (double)M;
                blob[tb.tw1 + ((s * (R1 - 1) + ka - 1) * 32 + l) * 2] = (float)std::cos(ang);
                blob[tb.tw1 + ((s * (R1 - 1) + ka - 1) * 32 + l) * 2 + 1] = (float)std::sin(ang);
            }
    for (int kb = 1; kb < 8; kb++)
        for (int c = 0; c < 8; c++) {
            const double ang = -two_pi * (double)(c * kb) / 64.0;
            blob[tb.tw2 + ((kb - 1) * 8 + c) * 2] = (float)std::cos(ang);
            blob[tb.tw2 + ((kb - 1) * 8 + c) * 2 + 1] = (float)std::sin(ang);
        }
    for (int w = 0; w < units; w++)
        for (int m = 0; m < 9; m++)
            for (int l = 0; l < 32; l++) {
                const double ang = -two_pi * (double)w8_bin(J, l + 32 * w, m) / (double)P;
                blob[tb.ptw + ((w * 9 + m) * 32 + l) * 2] = (float)std::cos(ang);
                blob[tb.ptw + ((w * 9 + m) * 32 + l) * 2 + 1] = (float)std::sin(ang);
            }
    // chunk c lives at (lane = c / rounds, round = c % rounds); its bins sit in the row of tile slots 8c .. 8c+7
    std::vector<int> pos(n_bins, W8_CSTRIDE * tb.n_slots + 8);          // dump slot for unused bins
    std::vector<int> chunk_of(n_bins, -1), slot_of(n_bins, -1);
    for (int ci = 0; ci < n_chunks; ci++)
        for (int j = 0; j < chunks[ci].count; j++) {
            chunk_of[chunks[ci].start + j] = ci;
            slot_of[chunks[ci].start + j] = j;
        }
    if (!x2) {
        // slot of every bin inside its row: edge colouring of (chunk row) x (store instruction, half-warp, row parity)
        std::vector<std::pair<int, int>> edges;
        std::vector<int> edge_bin;
        std::vector<char> seen(n_bins, 0);
        const int active = R1 >= 8 ? 32 : 16;
        for (int w = 0; w < units; w++)
            for (int m = 0; m < 8; m++)
                for (int sdx = 0; sdx < 2; sdx++)
                    for (int l = 0; l < active; l++) {
                        const int k0 = w8_bin(J, l + 32 * w, m);
                        if (k0 > M) continue;
                        const int k = sdx ? M - k0 : k0;
                        if (chunk_of[k] < 0 || seen[k]) continue;          // a self-mirrored bin is stored twice: first store counts
                        seen[k] = 1;
                        const int group = ((w * 8 + m) * 2 + sdx) * 2 + (l >> 4);
                        edges.push_back({chunk_of[k], group * 2 + (w8_chunk_row(chunk_of[k], chunk_of[k] / rounds, rounds) & 1)});
                        edge_bin.push_back(k);
                    }
        std::vector<int> colour;
        w8_edge_colour(n_chunks, units * 8 * 2 * 2 * 2, edges, W8_CHUNK, colour);
        std::vector<int> used(n_chunks, 0);
        for (int k = 0; k < n_bins; k++) slot_of[k] = -1;
        for (size_t e = 0; e < edges.size(); e++)
            if (colour[e] >= 0) { slot_of[edge_bin[e]] = colour[e]; used[edges[e].first] |= 1 << colour[e]; }
        for (int k = 0; k < n_bins; k++)                                  // over-full groups, bins only lane 0's ninth slot stores
            if (chunk_of[k] >= 0 && slot_of[k] < 0) {
                int c = 0;
                while (used[chunk_of[k]] & (1 << c)) c++;
                slot_of[k] = c;
                used[chunk_of[k]] |= 1 << c;
            }
    }
    std::vector<int32_t> cflag(tb.n_slots, 0);
    const int n_runs = (int)run_g.size();
    std::vector<int> seg_first(n_runs, 0), seg_cnt(n_runs, 0);
    std::vector<int> seg_chunk;                                          // chunk that ends (and stores) each run piece
    int seg = 0;
    for (int ci = 0; ci < n_chunks; ci++) {
        const Chunk &ch = chunks[ci];
        const int rot = x2 ? 0 : ((ci / rounds) >> 1) & 3;  // rotation used by the lane that owns this chunk
        for (int j = 0; j < ch.count; j++) {
            const int k = ch.start + j, sl = slot_of[k];
            pos[k] = W8_CSTRIDE * w8_chunk_row(ci, ci / rounds, rounds) + sl;
            const int piece = (((sl >> 1) - rot) & 3), jj = 2 * piece + (sl & 1);    // where the lane meets the bin in slot sl
            blob[tb.cw + w8_cw_index(ci, ci / rounds, rounds) + 2 * jj] = h.bin_wfall[k];
            blob[tb.cw + w8_cw_index(ci, ci / rounds, rounds) + 2 * jj + 1] = h.bin_wrise[k];
        }
        const bool first = (ci % rounds == 0) || chunks[ci - 1].run != ch.run;
        const bool last = (ci % rounds == rounds - 1) || ci == n_chunks - 1 || chunks[ci + 1].run != ch.run;
        if (first && seg_cnt[ch.run] == 0) seg_first[ch.run] = seg;
        cflag[ci] = (first ? 1 : 0) | (last ? 2 : 0) | (seg << 8);
        if (last) { seg_cnt[ch.run]++; seg++; seg_chunk.push_back(ci); }
    }
    tb.n_segs = std::max(seg, 1);
    // slots of the sums: filter g reads the b sums of run g-1 and the a sums of run g as one contiguous range
    std::vector<int> run_of_filter(n_mels + 1, -1);
    for (int r = 0; r < n_runs; r++)
        if (run_g[r] >= 0 && run_g[r] <= n_mels) run_of_filter[run_g[r]] = r;
    std::vector<std::vector<W8SegEntry>> filt(n_mels);
    for (int g = 0; g < n_mels; g++) {
        const int rb = g >= 1 ? run_of_filter[g - 1] : -1, ra = run_of_filter[g];
        if (rb >= 0) for (int i = 0; i < seg_cnt[rb]; i++) { const int sg = seg_first[rb] + i; filt[g].push_back({sg, 1, seg_chunk[sg] / rounds, seg_chunk[sg] % rounds}); }
        if (ra >= 0) for (int i = 0; i < seg_cnt[ra]; i++) { const int sg = seg_first[ra] + i; filt[g].push_back({sg, 0, seg_chunk[sg] / rounds, seg_chunk[sg] % rounds}); }
    }
    std::vector<int> f_first, f_cnt(n_mels, 0);
    std::vector<std::vector<int>> order;
    int end_slot = 0;
    w8_seg_layout(filt, rounds, f_first, order, end_slot);
    std::vector<int> slot_a(tb.n_segs, -1), slot_b(tb.n_segs, -1);
    for (int g = 0; g < n_mels; g++) {
        f_cnt[g] = (int)filt[g].size();
        for (int j = 0; j < f_cnt[g]; j++) {
            const W8SegEntry &e = filt[g][order[g][j]];
            (e.is_b ? slot_b : slot_a)[e.seg] = f_first[g] + j;
        }
    }
    const int dump = (end_slot + 1) & ~1;                 // sums no filter reads (b of the last run, a of run -1) land here
    tb.seg_slots = dump + 8;                              // + the dump slot and room for the 6-slot reads of the last filter
    for (int i = 0; i < tb.n_segs; i++) {
        if (slot_a[i] < 0) slot_a[i] = dump;
        if (slot_b[i] < 0) slot_b[i] = dump;
    }
    for (int ci = 0; ci < n_chunks; ci++) {
        const int sg = cflag[ci] >> 8;
        cflag[ci] = (cflag[ci] & 3) | (slot_a[sg] << 8) | (int32_t)((uint32_t)slot_b[sg] << 20);
    }
    for (int ci = 0; ci < tb.n_slots; ci++)
        reinterpret_cast<int32_t *>(blob.data() + tb.cflag)[w8_flag_index(ci, ci / rounds, rounds)] = cflag[ci];
    tb.tile_floats = std::max(4 * M, (x2 ? 1 : 2) * (W8_CSTRIDE * tb.n_slots + 16) + 2 * (tb.seg_slots + parts * w8_lm_stride(tb.lm_part) + 32)) + 16;
    int32_t *ppos = reinterpret_cast<int32_t *>(blob.data() + tb.ppos);
    for (int w = 0; w < units && !x2; w++)
        for (int m = 0; m < 9; m++)
            for (int l = 0; l < 32; l++) {
                int k = w8_bin(J, l + 32 * w, m);
                if (k > M) k = 0;                          // lanes without a unit (R1 = 4) never store
                ppos[((w * 9 + m) * 32 + l) * 2] = pos[k];
                ppos[((w * 9 + m) * 32 + l) * 2 + 1] = pos[M - k];
            }
    if (x2) {
        // slot (unit, m) of the sequence transforms holds bin k and its mirror M - k; the radix-2 combination turns them
        // into the four bins k, 2M - k, M - k, M + k of the 4096-point transform (one float each in the tile)
        int32_t *p4 = reinterpret_cast<int32_t *>(blob.data() + tb.ppos4);
        for (int w = 0; w < units; w++)
            for (int m = 0; m < 9; m++)
                for (int l = 0; l < 32; l++) {
                    int k = w8_bin(J, l + 32 * w, m);
                    if (k > M) k = 0;
                    int32_t *q = p4 + ((w * 9 + m) * 32 + l) * 4;
                    q[0] = pos[k];
                    q[1] = pos[2 * M - k];
                    q[2] = pos[M - k];
                    q[3] = pos[M + k];
                }
    }
    int32_t *fdesc = reinterpret_cast<int32_t *>(blob.data() + tb.fdesc);
    for (int g = 0; g < n_mels; g++) {
        fdesc[2 * g] = f_first[g];
        fdesc[2 * g + 1] = f_cnt[g];
    }
    // DCT table [block][part][q][dct_row]: row (part, q) holds coefficient block * cw_lanes + q for the filters
    // f = part, part + parts, ...; zero beyond n_mfcc and beyond n_mels
    for (int b = 0; b < dct_blocks; b++)
        for (int pt = 0; pt < parts; pt++)
            for (int q = 0; q < tb.cw_lanes; q++)
                for (int i = 0; i < tb.dct_row; i++) {
                    const int cidx = b * tb.cw_lanes + q, f = pt + parts * i;
                    blob[tb.dct + ((b * 32 + pt * tb.cw_lanes + q) * tb.dct_row) + i] =
                        (cidx < n_mfcc && f < n_mels && i < tb.lm_part) ? (float)h.dct2[(size_t)cidx * n_mels + f] : 0.f;
                }
}

inline size_t warp8_smem_bytes(const W8Tables &tb, int n_mels, int n_warps = W8_WARPS)
{
    return ((size_t)tb.total + (size_t)n_warps * w8_warp_floats(tb, n_mels)) * sizeof(float);
}

// ---- launch (not in csrc/emu.cu, which replays the phase functions on the host and instantiates no kernel) --------
#if defined(__CUDACC__) && !defined(DSPX_EMU)
struct W8PlanData {
    W8Tables tb;
    int ctas_per_sm;
    size_t smem;
    size_t smem_wide;        // 0 when the 20-warp configuration does not fit
    size_t smem_mid;         // shared memory of the W8_WARPS_MID-warp configuration (used when the wide one does not fit), or 0
    size_t smem_r16;         // n_fft 2048: shared memory of the W8_WARPS_R16-warp configuration, 0 when it does not fit
};

inline int warp8_prepare(dspx_plan *pl)
{
    std::vector<float> blob;
    W8Tables tb{};
    warp8_build_tables(pl, blob, tb);
    const size_t smem = warp8_smem_bytes(tb, pl->cfg.n_mels);
    if (smem > 227 * 1024) { set_error("warp8: tables too large for shared memory"); return DSPX_EUNSUPPORTED; }
    auto *pd = new W8PlanData();
    pd->tb = tb;
    pd->smem = smem;
    pd->ctas_per_sm = (tb.r1 != 16 && smem * 2 + 2048 <= 227 * 1024) ? 2 : 1;   // (x2 plans have r1 = 16: one CTA)
    const size_t wide = warp8_smem_bytes(tb, pl->cfg.n_mels, W8_WARPS_WIDE);
    pd->smem_wide = (tb.r1 != 16 && wide + 1024 <= 227 * 1024) ? wide : 0;
    const size_t mid = warp8_smem_bytes(tb, pl->cfg.n_mels, W8_WARPS_MID);
    pd->smem_mid = (tb.r1 != 16 && !pd->smem_wide && pd->ctas_per_sm == 1 && mid + 1024 <= 227 * 1024) ? mid : 0;
    const size_t r16 = warp8_smem_bytes(tb, pl->cfg.n_mels, W8_WARPS_R16);
    pd->smem_r16 = (tb.r1 == 16 && !tb.x2 && W8_WARPS_R16 > W8_WARPS && r16 + 1024 <= 227 * 1024) ? r16 : 0;
    pl->fast_host = pd;
    DSPX_CUDA_CHECK(cudaMalloc(&pl->d_fast_tables, blob.size() * sizeof(float)));
    DSPX_CUDA_CHECK(cudaMemcpy(pl->d_fast_tables, blob.data(), blob.size() * sizeof(float), cudaMemcpyHostToDevice));
    pl->fast_tables_bytes = blob.size() * sizeof(float);
    return DSPX_OK;
}

inline void warp8_release(dspx_plan *pl)
{
    delete static_cast<W8PlanData *>(pl->fast_host);
    pl->fast_host = nullptr;
}

// the launch fields that come from the plan alone
inline W8Params w8_plan_params(const dspx_plan *pl)
{
    const W8PlanData *pd = static_cast<const W8PlanData *>(pl->fast_host);
    W8Params p{};
    p.hop = pl->cfg.hop_length;
    p.n_mels = pl->cfg.n_mels;
    p.n_mfcc = pl->cfg.n_mfcc;
    p.prefetch = 1;
    p.take = std::min(pl->cfg.frame_length, pl->P);
    p.alpha = (float)pl->cfg.pre_emphasis;
    p.win_a = pl->cfg.window == DSPX_WINDOW_HANN ? 0.25f : (pl->cfg.window == DSPX_WINDOW_HAMMING ? 0.27f : 0.5f);
    p.win_b = pl->cfg.window == DSPX_WINDOW_HANN ? -0.25f : (pl->cfg.window == DSPX_WINDOW_HAMMING ? -0.23f : 0.f);
    p.tb = pd->tb;
    p.tables = static_cast<const float *>(pl->d_fast_tables);
    return p;
}

// ... and those of an equal-length batch: n_clips rows of clip_stride samples, T frames each, one frame pair per item.
// A ragged batch sets rtab, rpairs and n_items on top.
inline W8Params w8_batch_params(const dspx_plan *pl, const void *samples, int64_t n_clips, int64_t clip_stride, int64_t T,
                                float *logmel, float *mfcc, int nchw)
{
    W8Params p = w8_plan_params(pl);
    const int64_t pairs = (T + 1) / 2;
    p.clips = static_cast<const float *>(samples);
    p.n_clips = n_clips;
    p.clip_stride = clip_stride;
    p.n_frames = T;
    p.pairs_per_clip = (uint32_t)pairs;
    p.n_items = (uint32_t)(n_clips * pairs);
    p.logmel = logmel;
    p.mfcc = mfcc;
    p.lm_ts = nchw ? 1 : p.n_mels;
    p.lm_fs = nchw ? T : 1;
    return p;
}

// persistent grid: at most max_ctas CTAs, whose warps stride over the items
template <int R1, bool PRE, bool STFT, bool SHARE, int NW, bool EMB = false, bool U4 = false, bool PCM = false,
          bool RAGGED = false>
inline int w8_launch_nw(const W8Params &p, size_t smem, int device, int64_t max_ctas, cudaStream_t st)
{
    const int64_t ctas = std::min<int64_t>(((int64_t)p.n_items + NW - 1) / NW, max_ctas);
    static std::atomic<unsigned char> optin[64];
    DSPX_CUDA_CHECK(optin_max_smem(feat_warp8_kernel<R1, PRE, STFT, SHARE, NW, EMB, U4, PCM, RAGGED>, optin, device));
    feat_warp8_kernel<R1, PRE, STFT, SHARE, NW, EMB, U4, PCM, RAGGED><<<(unsigned)ctas, NW * 32, smem, st>>>(p);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

// warps per CTA: on the feature path one CTA of 20 (or 12) warps per SM when it fits beside the tables (radix 4 / 8) or
// of 10 warps (radix 16); otherwise 8-warp CTAs, as many per SM as fit
template <int R1, bool PRE, bool STFT, bool SHARE, bool EMB, bool U4, bool PCM, bool RAGGED>
inline int w8_launch_cfg(const W8Params &p, const W8PlanData *pd, int device, int sm_count, cudaStream_t st)
{
    if constexpr (!STFT && R1 != 16) {
        if (pd->smem_wide)
            return w8_launch_nw<R1, PRE, STFT, SHARE, W8_WARPS_WIDE, EMB, U4, PCM, RAGGED>(p, pd->smem_wide, device, sm_count, st);
        if (pd->smem_mid)
            return w8_launch_nw<R1, PRE, STFT, SHARE, W8_WARPS_MID, EMB, U4, PCM, RAGGED>(p, pd->smem_mid, device, sm_count, st);
    }
    if constexpr (!STFT && R1 == 16) {
        if (pd->smem_r16)
            return w8_launch_nw<R1, PRE, STFT, SHARE, W8_WARPS_R16, EMB, U4, PCM, RAGGED>(p, pd->smem_r16, device, sm_count, st);
    }
    return w8_launch_nw<R1, PRE, STFT, SHARE, W8_WARPS, EMB, U4, PCM, RAGGED>(p, pd->smem, device,
                                                                              (int64_t)sm_count * pd->ctas_per_sm, st);
}

// the radix and pre-emphasis switch over one variant <STFT, SHARE, EMB, U4, PCM, RAGGED> (radix 16 never shares rows,
// see W8_SHARE)
template <bool STFT, bool SHARE, bool EMB, bool U4, bool PCM, bool RAGGED>
inline int w8_launch_variant(const dspx_plan *pl, const W8Params &p, bool pre, cudaStream_t st)
{
    const W8PlanData *pd = static_cast<const W8PlanData *>(pl->fast_host);
    const int dev = pl->device, sms = pl->sm_count;
    switch (pd->tb.r1) {
        case 4: return pre ? w8_launch_cfg<4, true, STFT, SHARE, EMB, U4, PCM, RAGGED>(p, pd, dev, sms, st)
                           : w8_launch_cfg<4, false, STFT, SHARE, EMB, U4, PCM, RAGGED>(p, pd, dev, sms, st);
        case 8: return pre ? w8_launch_cfg<8, true, STFT, SHARE, EMB, U4, PCM, RAGGED>(p, pd, dev, sms, st)
                           : w8_launch_cfg<8, false, STFT, SHARE, EMB, U4, PCM, RAGGED>(p, pd, dev, sms, st);
        case 16: return pre ? w8_launch_cfg<16, true, STFT, false, EMB, U4, PCM, RAGGED>(p, pd, dev, sms, st)
                            : w8_launch_cfg<16, false, STFT, false, EMB, U4, PCM, RAGGED>(p, pd, dev, sms, st);
    }
    set_error("warp8: bad radix");
    return DSPX_EUNSUPPORTED;
}

// a path's variant; fused embeddings (EMB) when p.eacc is set
template <bool RAGGED>
inline int w8_launch_path(const dspx_plan *pl, W8Path path, const W8Params &p, bool pre, cudaStream_t st)
{
    const bool emb = p.eacc != nullptr;
    switch (path) {
        case W8_SHARE: return emb ? w8_launch_variant<false, true, true, false, false, RAGGED>(pl, p, pre, st)
                                  : w8_launch_variant<false, true, false, false, false, RAGGED>(pl, p, pre, st);
        case W8_ALIGNED: return emb ? w8_launch_variant<false, false, true, false, false, RAGGED>(pl, p, pre, st)
                                    : w8_launch_variant<false, false, false, false, false, RAGGED>(pl, p, pre, st);
        case W8_U4: return w8_launch_variant<false, false, false, true, false, RAGGED>(pl, p, pre, st);
        case W8_PCM16: return w8_launch_variant<false, false, false, true, true, RAGGED>(pl, p, pre, st);
        default: set_error("warp8: path %d is not a feat_warp8_kernel variant", (int)path); return DSPX_EUNSUPPORTED;
    }
}

// Launches feat_warp8_kernel on a path warp8_select chose: W8_ALIGNED, W8_SHARE, W8_U4 or W8_PCM16.  p.stft selects the
// STFT mode, p.eacc the fused embeddings, p.rtab a ragged batch; pre: apply pre-emphasis.
inline int launch_warp8(const dspx_plan *pl, W8Path path, W8Params p, bool pre, cudaStream_t st)
{
    p.share = path == W8_SHARE;
#ifdef DSPX_W8_LAB
    // benchmarks/lab/w8_lab.cu: only the headline instantiation, for quick builds of kernel variants
    (void)pre;
    return w8_launch_nw<8, true, false, true, W8_WARPS_WIDE>(p, static_cast<const W8PlanData *>(pl->fast_host)->smem_wide,
                                                             pl->device, pl->sm_count, st);
#else
    if (p.stft)
        return p.share ? w8_launch_variant<true, true, false, false, false, false>(pl, p, pre, st)
                       : w8_launch_variant<true, false, false, false, false, false>(pl, p, pre, st);
    return p.rtab ? w8_launch_path<true>(pl, path, p, pre, st) : w8_launch_path<false>(pl, path, p, pre, st);
#endif
}

// [n_clips + 1] first frame pair of every clip, then the total: the compact array w8_ragged_clip searches
__global__ void ragged_pairs_kernel(const dspx_ragged_clip *rtab, int64_t n_clips, uint32_t *rpairs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_clips) rpairs[i] = (uint32_t)rtab[i].first_pair;
    else if (i == n_clips) rpairs[i] = (uint32_t)(rtab[i - 1].first_pair + (rtab[i - 1].n_frames + 1) / 2);
}
#endif

}  // namespace dspx
