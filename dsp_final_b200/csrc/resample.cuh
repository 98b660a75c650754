// resample.cuh -- polyphase resampling on the GPU, bit-identical to scipy.signal.resample_poly on float32 input.
//
// The reference resamples every clip whose rate differs from the config's on the host (src/utils/audio.py:27-30,
// scipy.signal.resample_poly with its default Kaiser(5.0) design).  For float32 input, scipy 1.18.1 casts the filter
// to float32 and evaluates each output as a plain sequential sum of products, so performing the same float32
// operations in the same order (__fmul_rn then __fadd_rn, ascending input index) gives the same bits; DESIGN.md
// section 4.5 states the contract.
//
// Layout.  up and down are reduced by their gcd.  The output samples are viewed as rows of U = m * up outputs
// (m = 1 unless up < RS_K): all outputs in one column of that grid share one filter phase, and row r reads the input
// window of row 0 shifted by r * D samples (D = m * down).  A tile is NR rows x S columns.  Thread (lane, item)
// computes the RS_K consecutive outputs of one column group in row 32 * (item's row block) + lane, so the phase and
// the offsets between those outputs' windows are the same for all lanes of a warp: one table value read from shared
// memory is a broadcast, and each input sample a lane reads feeds up to RS_K accumulators.  The tile stages, per row,
// the W input samples its outputs read (zero outside the clip: adding a +-0 product never changes a sum that starts
// at +0, so this equals skipping those terms), at an odd stride RS so that 32 lanes read 32 banks, followed by the
// S table rows the tile's columns use, copied from the global table (which stays L2-resident, so every ratio is
// served by the same kernel, including ones whose full table would not fit in shared memory).
#pragma once

#include "dspx_internal.cuh"

#if defined(__CUDA_ARCH__)
#define DSPX_FADD_RN(a, b) __fadd_rn((a), (b))
#else
#define DSPX_FADD_RN(a, b) ((float)((float)(a) + (float)(b)))
#endif

namespace dspx {

constexpr int RS_THREADS = 256;                 // 8 warps
constexpr int RS_K = 4;                         // consecutive outputs per thread (independent accumulators)
constexpr int RS_MAX_S = 64;                    // columns per tile
constexpr size_t RS_SMEM_TARGET = 96 * 1024;    // tiles shrink until they fit here (two CTAs per SM)
constexpr int64_t RS_MAX_FACTOR = 1 << 20;      // largest reduced up / down

// Tile geometry of one ratio: a pure host function of (up, down, P), shared by the kernel launch and the CPU replay.
struct RsGeom {
    int64_t up = 1, down = 1;   // reduced
    int64_t remove = 0;         // scipy's n_pre_remove
    int P = 0;                  // taps per phase
    int m = 1;
    int64_t U = 1, D = 1;       // outputs per row, input shift per row
    int S = 1;                  // columns per tile
    int NR = 32;                // rows per tile (a multiple of 32)
    int W = 0;                  // input samples a row's tile columns read
    int RS = 1;                 // row stride in shared memory: W rounded up to odd
    int64_t n_chunks = 1;       // column chunks per row: ceil(U / S)
    size_t smem = 0;            // bytes: NR * RS input samples + S * P taps
};

DSPX_HD int64_t rs_ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

inline size_t rs_smem_bytes(int NR, int RS, int S, int P) { return ((size_t)NR * RS + (size_t)S * P) * sizeof(float); }

// Returns false when even the smallest tile (32 rows x 1 column) does not fit in shared memory: P above ~1700 taps,
// i.e. down / up above ~85.
inline bool rs_geometry(int64_t up, int64_t down, int P, int64_t remove, size_t max_smem, RsGeom *g)
{
    g->up = up;
    g->down = down;
    g->P = P;
    g->remove = remove;
    g->m = up >= RS_K ? 1 : (int)rs_ceil_div(RS_K, up);
    g->U = g->m * up;
    g->D = g->m * down;
    int S = (int)(g->U < RS_MAX_S ? g->U : RS_MAX_S);
    int RB = 1;
    for (;;) {
        // enough work items for 16 per CTA (2 per warp) before the tile is shrunk to fit
        const int groups = (int)rs_ceil_div(S, RS_K);
        RB = (int)rs_ceil_div(16, groups);
        if (RB > 32) RB = 32;
        for (;;) {
            const int W = (int)rs_ceil_div((int64_t)(S - 1) * down, up) + P;
            const int RS = W | 1;
            const size_t bytes = rs_smem_bytes(32 * RB, RS, S, P);
            if (bytes <= RS_SMEM_TARGET || (RB == 1 && S == 1 && bytes <= max_smem)) {
                g->S = S;
                g->NR = 32 * RB;
                g->W = W;
                g->RS = RS;
                g->n_chunks = rs_ceil_div(g->U, S);
                g->smem = bytes;
                return true;
            }
            if (RB == 1) break;
            RB /= 2;
        }
        if (S == 1) return false;
        S /= 2;
    }
}

// Phases of scipy's filter: h = w * float32(up), g = zeros(pre) ++ h ++ zeros(post), zero-padded to P * up taps,
// T[t][p] = g[(P - 1 - p) * up + t] (scipy.signal._upfirdn._pad_h).  Returns false for an unusable window.
inline bool rs_build_table(int64_t up, int64_t down, const float *w, int64_t L, std::vector<float> &T, int *P_out,
                           int64_t *remove_out)
{
    const int64_t half = (L - 1) / 2;
    const int64_t pre = down - half % down;
    // post: scipy's loop, smallest value with _output_len(L + pre + post, n_in, up, down) >= n_out + remove.  Both
    // sides are ceilings over down whose numerators differ by L - up - half, whatever n_in is; the window is required
    // to make that non-negative (scipy's own design has half = 10 max(up, down)), so post = 0 for every clip length.
    if (L - up - half < 0) return false;
    const int64_t G = pre + L;
    const int64_t P = rs_ceil_div(G, up);
    if (P > (1 << 20)) return false;
    T.assign((size_t)(P * up), 0.0f);
    const float fu = (float)up;
    for (int64_t t = 0; t < up; t++)
        for (int64_t p = 0; p < P; p++) {
            const int64_t k = (P - 1 - p) * up + t - pre;       // index into h
            T[(size_t)(t * P + p)] = (k >= 0 && k < L) ? DSPX_FMUL_RN(w[k], fu) : 0.0f;
        }
    *P_out = (int)P;
    *remove_out = (half + pre) / down;
    return true;
}

DSPX_HD int64_t rs_out_len(int64_t n_in, int64_t up, int64_t down) { return rs_ceil_div(n_in * up, down); }

// One clip as a tile sees it.
struct RsClip {
    const void *in;       // first sample of the clip (float32 or int16)
    int64_t n_in;
    float *out;
    int64_t n_out;
};

struct RsTile {
    int64_t i0;           // first output of the tile (row 0, first column)
    int64_t y0;           // remove + i0
    int64_t cbase;        // floor(y0 * down / up): input index of the last tap of that output
    int S;                // columns of this tile (the last chunk of a row may be narrower)
};

DSPX_HD int64_t rs_tiles(const RsGeom &g, int64_t n_out) { return rs_ceil_div(rs_ceil_div(n_out, g.U), g.NR) * g.n_chunks; }

DSPX_HD RsTile rs_tile(const RsGeom &g, int64_t tile)
{
    RsTile t;
    const int64_t rb = tile / g.n_chunks, chunk = tile - rb * g.n_chunks;
    const int64_t col = chunk * g.S;
    t.i0 = rb * g.NR * g.U + col;
    t.y0 = g.remove + t.i0;
    t.cbase = t.y0 * g.down / g.up;
    t.S = (int)(g.U - col < g.S ? g.U - col : g.S);
    return t;
}

DSPX_HD float rs_load(const void *in, int pcm, int64_t j)
{
    return pcm ? (float)static_cast<const int16_t *>(in)[j] * (1.0f / 32768.0f)      // exact
               : static_cast<const float *>(in)[j];
}

// Tile row r's inputs in shared memory: the W samples from cbase + r * D - P + 1 (zero outside the clip), then the
// row's pad slot; elements q0, q0 + dq, ...
DSPX_HD void rs_stage_row(const RsGeom &g, const RsTile &t, const RsClip &c, int pcm, int r, float *row, int q0, int dq)
{
    const int64_t j0 = t.cbase + r * g.D - g.P + 1;
    for (int q = q0; q < g.RS; q += dq) {
        const int64_t j = j0 + q;
        row[q] = (q < g.W && j >= 0 && j < c.n_in) ? rs_load(c.in, pcm, j) : 0.0f;
    }
}

// The table row of tile column s's phase, from the global [up][P] table tab; taps p0, p0 + dp, ...
DSPX_HD void rs_stage_phase(const RsGeom &g, const RsTile &t, const float *tab, int s, float *dst, int p0, int dp)
{
    const float *src = tab + (t.y0 + s) * g.down % g.up * g.P;
    for (int p = p0; p < g.P; p += dp) dst[p] = src[p];
}

DSPX_HD unsigned rs_abs_bits(float v)
{
    unsigned u;
    memcpy(&u, &v, sizeof(u));
    return u & 0x7fffffffu;        // non-negative floats order like their bit patterns
}

// The RS_K outputs of (work item, lane): row 32 * (item / groups) + lane, columns RS_K * (item % groups) + k.
// Stores them and returns the largest |y| bits among them.
DSPX_HD unsigned rs_group(const RsGeom &g, const RsTile &t, const RsClip &c, const float *xs, const float *ts, int item,
                          int lane)
{
    const int groups = (t.S + RS_K - 1) / RS_K;
    const int row = 32 * (item / groups) + lane;
    const int col0 = RS_K * (item % groups);
    int d[RS_K];                                  // window offsets of the outputs, relative to the tile's column 0
    int nk = 0;
#pragma unroll
    for (int k = 0; k < RS_K; k++) {
        if (col0 + k < t.S) nk = k + 1;
        d[k] = (int)((t.y0 + col0 + k) * g.down / g.up - t.cbase);
    }
    const float *x = xs + (int64_t)row * g.RS;
    const float *tb = ts + (int64_t)col0 * g.P;
    float acc[RS_K];
#pragma unroll
    for (int k = 0; k < RS_K; k++) acc[k] = 0.0f;
    int d_last = d[0];
#pragma unroll
    for (int k = 1; k < RS_K; k++) d_last = k < nk ? d[k] : d_last;      // no dynamic index: d stays in registers
    const int q_end = d_last + g.P;
    for (int q = d[0]; q < q_end; q++) {
        const float xv = x[q];
#pragma unroll
        for (int k = 0; k < RS_K; k++) {
            const int p = q - d[k];
            if (k < nk && (unsigned)p < (unsigned)g.P) acc[k] = DSPX_FADD_RN(acc[k], DSPX_FMUL_RN(xv, tb[k * g.P + p]));
        }
    }
    unsigned peak = 0;
    const int64_t i = t.i0 + (int64_t)row * g.U + col0;
#pragma unroll
    for (int k = 0; k < RS_K; k++) {
        if (k < nk && i + k < c.n_out) {
            c.out[i + k] = acc[k];
            const unsigned b = rs_abs_bits(acc[k]);
            peak = b > peak ? b : peak;
        }
    }
    return peak;
}

DSPX_HD int rs_items(const RsGeom &g, const RsTile &t) { return (g.NR / 32) * ((t.S + RS_K - 1) / RS_K); }

// normalize_audio: y / peak, the correctly rounded float32 quotient, when peak > 0 (a NaN peak compares false).
DSPX_HD float rs_normalize(float y, unsigned peak_bits)
{
    float peak;
    memcpy(&peak, &peak_bits, sizeof(peak));
#if defined(__CUDA_ARCH__)
    return peak > 0.0f ? __fdiv_rn(y, peak) : y;
#else
    return peak > 0.0f ? y / peak : y;
#endif
}

// Per-clip view of a batch: strided (rtab == nullptr) or ragged.
struct RsBatch {
    const void *in;
    int pcm;
    int64_t n_in, in_stride;       // strided
    float *out;
    int64_t out_stride;
    const dspx_resample_clip *rtab;
};

DSPX_HD RsClip rs_clip(const RsBatch &b, const RsGeom &g, int64_t clip)
{
    RsClip c;
    const size_t esz = b.pcm ? sizeof(int16_t) : sizeof(float);
    const int64_t in_start = b.rtab ? b.rtab[clip].in_start : clip * b.in_stride;
    c.in = static_cast<const char *>(b.in) + (size_t)in_start * esz;
    c.n_in = b.rtab ? b.rtab[clip].in_length : b.n_in;
    c.out = b.out + (b.rtab ? b.rtab[clip].out_start : clip * b.out_stride);
    c.n_out = b.rtab ? b.rtab[clip].out_length : rs_out_len(b.n_in, g.up, g.down);
    return c;
}

#if defined(__CUDACC__) && !defined(DSPX_EMU)
// grid (tiles of the longest clip, clips).  peaks: one unsigned per clip (|y| bits), or nullptr without normalisation.
__global__ void __launch_bounds__(RS_THREADS) resample_poly_kernel(RsGeom g, RsBatch b, const float *tab, unsigned *peaks)
{
    extern __shared__ float rs_smem[];
    const RsClip c = rs_clip(b, g, blockIdx.y);
    if ((int64_t)blockIdx.x >= rs_tiles(g, c.n_out)) return;
    const RsTile t = rs_tile(g, blockIdx.x);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *ts = rs_smem + (int64_t)g.NR * g.RS;
    for (int r = warp; r < g.NR; r += RS_THREADS / 32) rs_stage_row(g, t, c, b.pcm, r, rs_smem + (int64_t)r * g.RS, lane, 32);
    for (int s = warp; s < t.S; s += RS_THREADS / 32) rs_stage_phase(g, t, tab, s, ts + (int64_t)s * g.P, lane, 32);
    __syncthreads();
    const int n_items = rs_items(g, t);
    unsigned peak = 0;
    for (int item = warp; item < n_items; item += RS_THREADS / 32) {
        const unsigned p = rs_group(g, t, c, rs_smem, ts, item, lane);
        peak = p > peak ? p : peak;
    }
    if (peaks) {
        peak = __reduce_max_sync(0xffffffffu, peak);
        if (lane == 0 && peak) atomicMax(&peaks[blockIdx.y], peak);
    }
}

// up == down == 1 after reduction: scipy returns a copy of the input (its filter is not applied).
__global__ void __launch_bounds__(256) resample_copy_kernel(RsGeom g, RsBatch b, unsigned *peaks)
{
    const RsClip c = rs_clip(b, g, blockIdx.y);
    unsigned peak = 0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < c.n_out; i += (int64_t)gridDim.x * 256) {
        const float v = rs_load(c.in, b.pcm, i);
        c.out[i] = v;
        const unsigned u = rs_abs_bits(v);
        peak = u > peak ? u : peak;
    }
    if (peaks) {
        peak = __reduce_max_sync(0xffffffffu, peak);
        if ((threadIdx.x & 31) == 0 && peak) atomicMax(&peaks[blockIdx.y], peak);
    }
}

__global__ void __launch_bounds__(256) resample_normalize_kernel(RsGeom g, RsBatch b, const unsigned *peaks)
{
    const RsClip c = rs_clip(b, g, blockIdx.y);
    const unsigned pk = peaks[blockIdx.y];
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < c.n_out; i += (int64_t)gridDim.x * 256)
        c.out[i] = rs_normalize(c.out[i], pk);
}
#endif

}  // namespace dspx

// Immutable after creation, like dspx_plan: the reduced ratio, its tile geometry and the device phase table.
struct dspx_resampler {
    dspx::RsGeom g;
    bool identity = false;      // up == down == 1 after reduction
    int device = 0;
    float *d_tab = nullptr;     // [up][P]
};
