// decode.cuh -- WAV sample decoding and channel downmix on the GPU, bit-identical to load_audio (+ normalize_audio).
//
// The reference decodes every file on the host (src/utils/audio.py:19-31: soundfile.read, then np.mean over the channel
// axis).  This pass takes the data chunks as stored -- PCM 8/16/24/32-bit or IEEE float 32/64, C <= 32 channels
// interleaved -- and writes the float32 mono clip load_audio returns, bit for bit; DESIGN.md section 4.6 states the
// contract.  The downmix repeats numpy's float32 pairwise sum (np.mean(axis=1)): a plain running sum from +0 for
// C < 8, eight running sums combined as a tree and added to +0 for C >= 8, then one correctly rounded divide by C.
//
// Layout.  The grid is tiles x clips.  A tile is a run of frames of one clip (a multiple of 16 frames, at most
// DEC_MAX_FRAMES, chosen per clip so that its input bytes fit DEC_IN_BYTES).  Clip inputs start at 16-byte offsets,
// so a tile's input bytes start 16-byte aligned: the CTA stages them in shared memory with 16-byte loads, decodes
// from there (PCM24 and odd channel counts need no unaligned global loads; consecutive threads take consecutive
// frames), stages the float32 results, and writes them with 16-byte stores.  The peak |y| per clip is folded into the
// same pass (one atomicMax per warp, as the resampler does).  Normalising needs the peak before the divide, so it
// takes a second pass; each clip picks the cheaper one by bytes moved: when its frames are shorter than 8 bytes the
// second pass decodes the input again (2 in + 4 bytes per output, no store in the first pass), otherwise it
// re-reads the stored outputs (in + 12).
#pragma once

#include "dspx_internal.cuh"
#include "resample.cuh"

namespace dspx {

constexpr int DEC_THREADS = 256;
constexpr int DEC_MAX_FRAMES = 2048;                                       // output frames per tile
constexpr int DEC_IN_BYTES = 16384;                                        // staged input bytes per tile
constexpr size_t DEC_SMEM = DEC_IN_BYTES + DEC_MAX_FRAMES * sizeof(float);  // dynamic shared memory of a CTA
constexpr int64_t DEC_MAX_LEN = (int64_t)1 << 40;

enum DecMode { DEC_STORE = 0, DEC_PEAK = 1, DEC_NORM = 2 };

DSPX_HD int dec_bytes(int dtype)
{
    switch (dtype) {
    case DSPX_DTYPE_PCM8: return 1;
    case DSPX_DTYPE_PCM16: return 2;
    case DSPX_DTYPE_PCM24: return 3;
    case DSPX_DTYPE_PCM32: case DSPX_DTYPE_F32: return 4;
    case DSPX_DTYPE_F64: return 8;
    default: return 0;
    }
}

DSPX_HD int dec_tile_frames(const dspx_decode_clip &r)
{
    const int t = (DEC_IN_BYTES / (r.channels * dec_bytes(r.dtype))) & ~15;
    return t < DEC_MAX_FRAMES ? t : DEC_MAX_FRAMES;
}

DSPX_HD int64_t dec_tiles(const dspx_decode_clip &r) { return rs_ceil_div(r.n_frames, dec_tile_frames(r)); }

// Normalising: the second pass decodes again when a frame is shorter than the 8 bytes a divide pass would re-read.
DSPX_HD bool dec_recompute(const dspx_decode_clip &r) { return r.channels * dec_bytes(r.dtype) < 8; }

DSPX_HD float dec_f32(uint32_t u)
{
    float f;
    memcpy(&f, &u, sizeof(f));
    return f;
}

DSPX_HD uint32_t dec_u32(float f)
{
    uint32_t u;
    memcpy(&u, &f, sizeof(u));
    return u;
}

// The NaN an x86 float operation returns, so that the device gives numpy's bits: the first NaN operand, quieted, or
// the default NaN (0xffc00000) when the operation made one (inf - inf).  The GPU would return 0x7fffffff.
DSPX_HD float dec_nan(float a, float b)
{
    if (a != a) return dec_f32(dec_u32(a) | 0x00400000u);
    if (b != b) return dec_f32(dec_u32(b) | 0x00400000u);
    return dec_f32(0xffc00000u);
}

DSPX_HD float dec_add(float a, float b)
{
    const float r = DSPX_FADD_RN(a, b);
    return r == r ? r : dec_nan(a, b);
}

// One sample from the staged bytes: read_wav's value, exactly (DESIGN.md 4.6).
DSPX_HD float dec_sample(const unsigned char *p, int dtype)
{
    switch (dtype) {
    case DSPX_DTYPE_PCM8: return DSPX_FMUL_RN((float)((int)p[0] - 128), 1.0f / 128.0f);
    case DSPX_DTYPE_PCM16: {
        int16_t s;
        memcpy(&s, p, 2);
        return DSPX_FMUL_RN((float)s, 1.0f / 32768.0f);
    }
    case DSPX_DTYPE_PCM24: {
        const int32_t s = (int32_t)(((uint32_t)p[0] << 8) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 24)) >> 8;
        return DSPX_FMUL_RN((float)s, 1.0f / 8388608.0f);
    }
    case DSPX_DTYPE_PCM32: {
        int32_t s;
        memcpy(&s, p, 4);
        return DSPX_FMUL_RN((float)s, 1.0f / 2147483648.0f);     // (float)s rounds once; the scaling is exact
    }
    case DSPX_DTYPE_F32: {
        float f;
        memcpy(&f, p, 4);
        return f;
    }
    default: {
        double d;
        memcpy(&d, p, 8);
        if (d != d) {                                              // NaN: sign, quiet bit and the top payload bits
            uint64_t u;
            memcpy(&u, &d, 8);
            return dec_f32((uint32_t)(u >> 32 & 0x80000000u) | 0x7fc00000u | (uint32_t)(u >> 29 & 0x003fffffu));
        }
        return (float)d;
    }
    }
}

// np.mean over the C float32 samples sample(0) ... sample(C - 1) of one frame (C == 1: the sample itself, as load_audio
// does not average).  Shared by the WAV and FLAC decoders (DESIGN.md 4.6, 4.7).
template <class Sample>
DSPX_HD float dec_mean(int C, Sample sample)
{
    if (C == 1) return sample(0);
    float s;
    if (C < 8) {
        s = 0.0f;
        for (int c = 0; c < C; c++) s = dec_add(s, sample(c));
    } else {
        float r[8];
#pragma unroll
        for (int j = 0; j < 8; j++) r[j] = sample(j);
        int i = 8;
        for (; i + 8 <= C; i += 8) {
#pragma unroll
            for (int j = 0; j < 8; j++) r[j] = dec_add(r[j], sample(i + j));
        }
        s = dec_add(dec_add(dec_add(r[0], r[1]), dec_add(r[2], r[3])), dec_add(dec_add(r[4], r[5]), dec_add(r[6], r[7])));
        for (; i < C; i++) s = dec_add(s, sample(i));
        s = dec_add(0.0f, s);              // numpy adds the pairwise sum to the reduction's identity: -0 becomes +0
    }
    if (s != s) return dec_nan(s, s);
#if defined(__CUDA_ARCH__)
    return __fdiv_rn(s, (float)C);
#else
    return s / (float)C;
#endif
}

// np.mean(frame, axis=1) of one frame of C samples at p.
DSPX_HD float dec_mix(const unsigned char *p, int C, int dtype)
{
    const int b = dec_bytes(dtype);
    return dec_mean(C, [=](int c) { return dec_sample(p + c * b, dtype); });
}

// normalize_audio's y / peak (rs_normalize), with x86's default NaN where the quotient is one (inf / inf).
DSPX_HD float dec_normalize(float y, unsigned peak_bits)
{
    const float r = rs_normalize(y, peak_bits);
    return r == r || y != y ? r : dec_f32(0xffc00000u);
}

struct DecTile {
    int64_t f0;          // first frame
    int n;               // frames in this tile
    const unsigned char *in;   // its first input byte (16-byte aligned)
    int64_t in_bytes;
    float *out;          // its first output sample (16-byte aligned)
};

DSPX_HD DecTile dec_tile(const dspx_decode_clip &r, const unsigned char *in, float *out, int64_t tile)
{
    DecTile t;
    const int tf = dec_tile_frames(r);
    const int64_t fb = (int64_t)r.channels * dec_bytes(r.dtype);
    t.f0 = tile * tf;
    t.n = (int)(r.n_frames - t.f0 < tf ? r.n_frames - t.f0 : tf);
    t.in = in + r.in_offset + t.f0 * fb;
    t.in_bytes = t.n * fb;
    t.out = out + r.out_start + t.f0;
    return t;
}

// The tile's input bytes into shared memory: whole 16-byte chunks q0, q0 + dq, ..., then the tail byte by byte.
DSPX_HD void dec_stage(const DecTile &t, unsigned char *xs, int q0, int dq)
{
    const int nb = (int)t.in_bytes, n16 = nb >> 4;
    const uint4 *src = reinterpret_cast<const uint4 *>(t.in);
    uint4 *dst = reinterpret_cast<uint4 *>(xs);
#pragma unroll 4
    for (int q = q0; q < n16; q += dq) dst[q] = src[q];
    for (int q = (n16 << 4) + q0; q < nb; q += dq) xs[q] = t.in[q];
}

// Frames f0, f0 + df, ... of the tile decoded into ys (normalised by peak_bits when normalize); returns the largest |y|
// bits among them.
DSPX_HD unsigned dec_frames(const dspx_decode_clip &r, const DecTile &t, const unsigned char *xs, float *ys, bool store,
                            bool normalize, unsigned peak_bits, int f0, int df)
{
    const int fb = r.channels * dec_bytes(r.dtype);
    unsigned peak = 0;
    for (int f = f0; f < t.n; f += df) {
        float y = dec_mix(xs + f * fb, r.channels, r.dtype);
        const unsigned u = rs_abs_bits(y);
        peak = u > peak ? u : peak;
        if (normalize) y = dec_normalize(y, peak_bits);
        if (store) ys[f] = y;
    }
    return peak;
}

// The staged outputs to the clip with 16-byte stores (groups q0, q0 + dq, ...; the last partial group sample by
// sample).
DSPX_HD void dec_store(const DecTile &t, const float *ys, int q0, int dq)
{
    const int n4 = t.n >> 2;
    float4 *dst = reinterpret_cast<float4 *>(t.out);
    for (int q = q0; q < n4; q += dq) dst[q] = reinterpret_cast<const float4 *>(ys)[q];
    for (int f = 4 * n4 + q0; f < t.n; f += dq) t.out[f] = ys[f];
}

// The divide pass of a clip that is not decoded again: its stored outputs over the peak, in place, the same groups.
DSPX_HD void dec_divide(const DecTile &t, unsigned peak_bits, int q0, int dq)
{
    const int n4 = t.n >> 2;
    float4 *p = reinterpret_cast<float4 *>(t.out);
    for (int q = q0; q < n4; q += dq) {
        float4 v = p[q];
        v.x = dec_normalize(v.x, peak_bits);
        v.y = dec_normalize(v.y, peak_bits);
        v.z = dec_normalize(v.z, peak_bits);
        v.w = dec_normalize(v.w, peak_bits);
        p[q] = v;
    }
    for (int f = 4 * n4 + q0; f < t.n; f += dq) t.out[f] = dec_normalize(t.out[f], peak_bits);
}

// What a pass does with one clip: {stage and decode, store the outputs, fold the peak, normalise while decoding,
// divide the stored outputs}.
struct DecWork {
    bool decode, store, peak, normalize, divide;
};

DSPX_HD DecWork dec_work(const dspx_decode_clip &r, int mode)
{
    const bool rc = dec_recompute(r);
    switch (mode) {
    case DEC_STORE: return {true, true, false, false, false};
    case DEC_PEAK: return {true, !rc, true, false, false};
    default: return {rc, rc, false, rc, !rc};
    }
}

#if defined(__CUDACC__) && !defined(DSPX_EMU)
// grid (tiles of the longest clip, clips).  peaks: one unsigned per clip (|y| bits); unused in DEC_STORE mode.
__global__ void __launch_bounds__(DEC_THREADS) wav_decode_kernel(const unsigned char *in, const dspx_decode_clip *tab,
                                                                 float *out, unsigned *peaks, int mode)
{
    extern __shared__ uint4 dec_smem[];
    const dspx_decode_clip r = tab[blockIdx.y];
    if ((int64_t)blockIdx.x >= dec_tiles(r)) return;
    const DecTile t = dec_tile(r, in, out, blockIdx.x);
    const DecWork w = dec_work(r, mode);
    const unsigned pk = mode == DEC_NORM ? peaks[blockIdx.y] : 0u;
    if (w.divide) {
        dec_divide(t, pk, threadIdx.x, DEC_THREADS);
        return;
    }
    unsigned char *xs = reinterpret_cast<unsigned char *>(dec_smem);
    float *ys = reinterpret_cast<float *>(xs + DEC_IN_BYTES);
    dec_stage(t, xs, threadIdx.x, DEC_THREADS);
    __syncthreads();
    unsigned peak = dec_frames(r, t, xs, ys, w.store, w.normalize, pk, threadIdx.x, DEC_THREADS);
    if (w.peak) {
        peak = __reduce_max_sync(0xffffffffu, peak);
        if ((threadIdx.x & 31) == 0 && peak) atomicMax(&peaks[blockIdx.y], peak);
    }
    if (!w.store) return;
    __syncthreads();
    dec_store(t, ys, threadIdx.x, DEC_THREADS);
}
#endif

}  // namespace dspx
