// flac.cuh -- FLAC decoding and channel downmix on the GPU, bit-identical to the samples a file holds, scaled and
// downmixed as the WAV decoder does it (decode.cuh; DESIGN.md section 4.7 states the contract).
//
// The host finds the frames (fl_parse_file for dspx_flac_layout: STREAMINFO, header CRC-8, frame numbering) and
// writes a table of them.  The
// device then runs two kernels:
//   flac_frame_kernel  one thread per frame.  A subframe is a serial unit -- a Rice partition stores no length, so the
//                      residual is walked code by code, and the prediction is a recurrence over the previous `order`
//                      samples -- and a frame's subframes follow each other in the bitstream, so the frame is the unit.
//                      The thread checks the frame's CRC-16, then decodes each subframe's integers into the workspace,
//                      restoring the prediction as it reads the residual (the last `order` samples live in
//                      registers, and so do the coefficients up to order 8).  Thread-per-frame keeps as many bit
//                      readers in flight as there are frames (~10^5 for 2000 five-second stereo clips), where a CTA
//                      per frame would allow at most 32 per SM.
//   flac_mix_kernel    one CTA per frame: channel decorrelation, scaling, the downmix of decode.cuh (dec_mean), the
//                      peak per file and the stores; with normalisation a second launch divides the stored outputs.
// The input is untrusted.  The bit reader loads whole aligned words only when they lie inside the frame, reads the
// edge words byte by byte, and returns zeros past the frame's end; reading there sets the frame's status.
#pragma once

#include <algorithm>

#include "decode.cuh"

namespace dspx {

constexpr int FL_THREADS = 64;          // flac_frame_kernel: frames per CTA
constexpr int FL_MIX_THREADS = 256;
constexpr int FL_MAX_ORDER = 32;
constexpr int FL_MAX_BLOCK = 65535;

enum FlMode { FL_STORE = 0, FL_PEAK = 1, FL_NORM = 2 };

DSPX_HD bool fl_wide(int bps) { return bps == 32; }    // the side channel of a 32-bit stream has 33 bits: int64 storage
DSPX_HD int fl_channels(int assignment) { return assignment < 8 ? assignment + 1 : 2; }
DSPX_HD int64_t fl_ws_bytes(int bps, int assignment, int block)
{
    return (((int64_t)block * fl_channels(assignment) * (fl_wide(bps) ? 8 : 4)) + 15) & ~(int64_t)15;
}

// CRC-16 (polynomial 0x8005, MSB first, initial 0) table entry, as FLAC frames use it.
DSPX_HD uint16_t fl_crc16_entry(int i)
{
    unsigned c = (unsigned)i << 8;
    for (int k = 0; k < 8; k++) c = (c & 0x8000u) ? (c << 1) ^ 0x8005u : c << 1;
    return (uint16_t)c;
}

// ---- bit reader ----

struct FlBits {
    const unsigned char *base;   // the frame's first byte rounded down to 4 bytes
    int64_t lo, hi;              // the frame's bytes, relative to base
    int64_t next;                // next 4-byte word to load
    uint64_t buf;                // unread bits, most significant first; the bits below them are zero
    int n;                       // how many
    int64_t used;                // bits consumed, from base
    int64_t end;                 // bit where the frame's CRC-16 starts, from base
};

DSPX_HD uint32_t fl_bswap(uint32_t w)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0, 0x0123);
#else
    return __builtin_bswap32(w);
#endif
}

// Word i of the frame as a big-endian integer; the bytes outside the frame read as zero and are not loaded.
DSPX_HD uint32_t fl_word(const FlBits &b, int64_t i)
{
    const int64_t a = 4 * i;
    if (a >= b.lo && a + 4 <= b.hi) {
        uint32_t w;
#if defined(__CUDA_ARCH__)
        w = __ldg(reinterpret_cast<const unsigned *>(b.base + a));
#else
        memcpy(&w, b.base + a, 4);
#endif
        return fl_bswap(w);
    }
    uint32_t w = 0;
    for (int j = 0; j < 4; j++)
        if (a + j >= b.lo && a + j < b.hi) w |= (uint32_t)b.base[a + j] << (24 - 8 * j);
    return w;
}

DSPX_HD void fl_refill(FlBits &b)
{
    if (b.n <= 32) {
        b.buf |= (uint64_t)fl_word(b, b.next++) << (32 - b.n);
        b.n += 32;
    }
}

// The next k bits (0 <= k <= 32) as an unsigned integer.
DSPX_HD uint32_t fl_read(FlBits &b, int k)
{
    if (k == 0) return 0;
    fl_refill(b);
    const uint32_t v = (uint32_t)(b.buf >> (64 - k));
    b.buf <<= k;
    b.n -= k;
    b.used += k;
    return v;
}

// The next k bits (0 <= k <= 33) as a two's complement integer.
DSPX_HD int64_t fl_sread(FlBits &b, int k)
{
    if (k == 0) return 0;
    uint64_t v = k > 32 ? (uint64_t)fl_read(b, k - 32) << 32 | fl_read(b, 32) : fl_read(b, k);
    return (int64_t)(v << (64 - k)) >> (64 - k);
}

// Zeros up to the next one bit, consumed with it.  Stops once past the frame's end (the caller sees the overrun).
DSPX_HD uint32_t fl_unary(FlBits &b)
{
    uint32_t q = 0;
    for (;;) {
        fl_refill(b);
        if (b.buf) {
#if defined(__CUDA_ARCH__)
            const int z = __clzll((long long)b.buf);
#else
            const int z = __builtin_clzll(b.buf);
#endif
            b.buf <<= z;
            b.buf <<= 1;
            b.n -= z + 1;
            b.used += z + 1;
            return q + (uint32_t)z;
        }
        q += (uint32_t)b.n;
        b.used += b.n;
        b.n = 0;
        if (b.used > b.end) return q;
    }
}

DSPX_HD FlBits fl_bits(const unsigned char *in, int64_t frame_offset, int64_t frame_bytes, int64_t start)
{
    FlBits b;
    const int64_t a = frame_offset & ~(int64_t)3;
    b.base = in + a;
    b.lo = frame_offset - a;
    b.hi = b.lo + frame_bytes;
    b.end = (b.hi - 2) * 8;
    const int64_t s = b.lo + start;
    b.next = s >> 2;
    b.buf = 0;
    b.n = 0;
    b.used = (s & ~(int64_t)3) * 8;
    fl_read(b, (int)(s & 3) * 8);
    return b;
}

// CRC-16 of the frame's bytes before its last two, compared with those two.
DSPX_HD bool fl_crc_ok(const FlBits &frame, const uint16_t *table)
{
    unsigned crc = 0;
    const int64_t last = frame.hi - 2;
    for (int64_t i = frame.lo >> 2; 4 * i < last; i++) {
        const uint32_t w = fl_word(frame, i);
        for (int j = 0; j < 4; j++) {
            const int64_t a = 4 * i + j;
            if (a >= frame.lo && a < last) crc = ((crc << 8) ^ table[((crc >> 8) ^ (w >> (24 - 8 * j))) & 0xff]) & 0xffff;
        }
    }
    unsigned stored = 0;
    for (int64_t a = last; a < frame.hi; a++) {
        const uint32_t w = fl_word(frame, a >> 2);
        stored = stored << 8 | ((w >> (24 - 8 * (a & 3))) & 0xff);
    }
    return crc == stored;
}

// ---- subframes ----

// A predicted run: x[order .. n) = residual + (sum_j coef[j] * x[i-1-j]) >> shift, reading the residual's Rice
// partitions as it goes.  The history is registers (MAXO of them, zero past `order`), and so are the coefficients for
// MAXO <= 8; above that they are read from `coef` (shared memory on the device), which keeps the rare high orders
// from setting the kernel's register count.  T is the
// storage type; A the accumulator: uint32_t (wrapping) is exact when no partial sum leaves 32 bits or the shift is 0 (the
// fixed predictors: the result is exact modulo 2^32 and fits), else int64_t.
template <class T, class A, int MAXO>
DSPX_HD int fl_predict(FlBits &b, T *x, int n, int order, const int32_t *coef, int shift)
{
    const int method = (int)fl_read(b, 2);
    if (method > 1) return DSPX_FLAC_RESERVED;
    const int pbits = method ? 5 : 4, escape = method ? 31 : 15;
    const int porder = (int)fl_read(b, 4);
    const int parts = 1 << porder;
    if (n % parts) return DSPX_FLAC_INVALID;
    const int psize = n / parts;
    if (psize < order) return DSPX_FLAC_INVALID;
    A h[MAXO], c[MAXO];
#pragma unroll
    for (int j = 0; j < MAXO; j++) {
        h[j] = j < order ? (A)x[order - 1 - j] : (A)0;
        if (MAXO <= 8) c[j] = j < order ? (A)coef[j] : (A)0;
    }
    int i = order;
    for (int p = 0; p < parts; p++) {
        const int k = (int)fl_read(b, pbits);
        const int stop = (p + 1) * psize;
        const int raw = k == escape ? (int)fl_read(b, 5) : -1;
        for (; i < stop; i++) {
            int64_t r;
            if (raw >= 0) {
                r = fl_sread(b, raw);
            } else {
                const uint64_t u = (uint64_t)fl_unary(b) << k | fl_read(b, k);
                r = (int64_t)(u >> 1) ^ -(int64_t)(u & 1);
            }
            A acc = 0;
#pragma unroll
            for (int j = 0; j < MAXO; j++) acc += (MAXO <= 8 ? c[j] : (j < order ? (A)coef[j] : (A)0)) * h[j];
            A v;
            if (sizeof(A) == 4)
                v = (A)(uint32_t)r + (A)((int32_t)acc >> shift);
            else
                v = (A)r + (A)((int64_t)acc >> shift);
#pragma unroll
            for (int j = MAXO - 1; j > 0; j--) h[j] = h[j - 1];
            h[0] = v;
            x[i] = (T)(sizeof(A) == 4 ? (int64_t)(int32_t)v : (int64_t)v);
        }
        if (b.used > b.end) return DSPX_FLAC_OVERRUN;
    }
    return 0;
}

template <class T, class A>
DSPX_HD int fl_predict_any(FlBits &b, T *x, int n, int order, const int32_t *coef, int shift)
{
    if (order <= 8) return fl_predict<T, A, 8>(b, x, n, order, coef, shift);
    return fl_predict<T, A, FL_MAX_ORDER>(b, x, n, order, coef, shift);
}

// One subframe of n samples of sbps bits into x; coef: scratch for FL_MAX_ORDER coefficients.  Returns DSPX_FLAC_* bits.
template <class T>
DSPX_HD int fl_subframe(FlBits &b, T *x, int n, int sbps, int32_t *coef)
{
    if (fl_read(b, 1)) return DSPX_FLAC_RESERVED;
    const int type = (int)fl_read(b, 6);
    int wasted = 0;
    if (fl_read(b, 1)) wasted = (int)fl_unary(b) + 1;
    if (b.used > b.end) return DSPX_FLAC_OVERRUN;
    if (wasted >= sbps) return DSPX_FLAC_INVALID;
    const int bps = sbps - wasted;
    int st = 0;
    if (type == 0) {
        const T v = (T)fl_sread(b, bps);
        for (int i = 0; i < n; i++) x[i] = v;
    } else if (type == 1) {
        for (int i = 0; i < n; i++) x[i] = (T)fl_sread(b, bps);
    } else if ((type >= 8 && type <= 12) || type >= 32) {
        const bool lpc = type >= 32;
        const int order = lpc ? type - 31 : type - 8;
        if (order > n) return DSPX_FLAC_INVALID;
        for (int i = 0; i < order; i++) x[i] = (T)fl_sread(b, bps);
        int shift = 0, prec = 0;
        if (lpc) {
            prec = (int)fl_read(b, 4) + 1;
            if (prec == 16) return DSPX_FLAC_RESERVED;
            shift = (int)fl_sread(b, 5);
            if (shift < 0) return DSPX_FLAC_NEG_SHIFT;
            for (int j = 0; j < order; j++) coef[j] = (int32_t)fl_sread(b, prec);
        } else {
            const int32_t fixed[5][4] = {{0, 0, 0, 0}, {1, 0, 0, 0}, {2, -1, 0, 0}, {3, -3, 1, 0}, {4, -6, 4, -1}};
            for (int j = 0; j < order; j++) coef[j] = fixed[order][j];
        }
        if (b.used > b.end) return DSPX_FLAC_OVERRUN;
        // 64-bit accumulation when bps + precision + ceil(log2 order) can exceed 32 (DESIGN.md 4.7)
        int lg = 0;
        while ((1 << lg) < order) lg++;
        if (sizeof(T) == 8 || (lpc && bps + prec + lg > 32))
            st = fl_predict_any<T, int64_t>(b, x, n, order, coef, shift);
        else
            st = fl_predict_any<T, uint32_t>(b, x, n, order, coef, shift);
    } else {
        return DSPX_FLAC_RESERVED;
    }
    if (!st && b.used > b.end) st = DSPX_FLAC_OVERRUN;
    if (!st && wasted)
        for (int i = 0; i < n; i++) x[i] = (T)(int64_t)((uint64_t)(int64_t)x[i] << wasted);
    return st;
}

// Channel c of a frame is a side channel (one bit more than the stream).
DSPX_HD bool fl_side(int assignment, int c)
{
    return (assignment == 8 && c == 1) || (assignment == 9 && c == 0) || (assignment == 10 && c == 1);
}

// A whole frame of the file at `in`: CRC-16, then every subframe into samples (channel after channel, block_size apart; int64_t when
// fl_wide(bps), else int32_t).  Returns its DSPX_FLAC_* status.
DSPX_HD int fl_frame(const unsigned char *in, const dspx_flac_frame &fr, int bps, void *samples, int32_t *coef,
                     const uint16_t *crc_table)
{
    FlBits b = fl_bits(in, fr.in_offset, fr.in_bytes, fr.header_bytes);
    if (!fl_crc_ok(b, crc_table)) return DSPX_FLAC_CRC;
    const int C = fl_channels(fr.assignment), n = fr.block_size;
    for (int c = 0; c < C; c++) {
        const int sbps = bps + (fl_side(fr.assignment, c) ? 1 : 0);
        const int st = fl_wide(bps) ? fl_subframe(b, static_cast<int64_t *>(samples) + (int64_t)c * n, n, sbps, coef)
                                    : fl_subframe(b, static_cast<int32_t *>(samples) + (int64_t)c * n, n, sbps, coef);
        if (st) return st;
    }
    return 0;
}

// ---- decorrelation, scaling, downmix ----

DSPX_HD int64_t fl_int(const void *samples, bool wide, int64_t i) {
    return wide ? static_cast<const int64_t *>(samples)[i] : static_cast<const int32_t *>(samples)[i];
}

// s / 2^(bps-1) in float32: exact for bps <= 24, correctly rounded above (read_wav's PCM scaling).
DSPX_HD float fl_scale(int64_t s, int bps)
{
    return DSPX_FMUL_RN((float)(int32_t)s, dec_f32((uint32_t)(127 - (bps - 1)) << 23));
}

// Output sample i of a frame: its channels decorrelated, scaled and averaged as np.mean does (dec_mean).
DSPX_HD float fl_mix(const dspx_flac_frame &fr, int bps, const void *samples, int i)
{
    const bool wide = fl_wide(bps);
    const int64_t n = fr.block_size;
    if (fr.assignment < 8)
        return dec_mean(fr.assignment + 1, [=](int c) { return fl_scale(fl_int(samples, wide, c * n + i), bps); });
    const int64_t a = fl_int(samples, wide, i), s = fl_int(samples, wide, n + i);
    int64_t l, r;
    if (fr.assignment == 8) {
        l = a;
        r = a - s;
    } else if (fr.assignment == 9) {
        l = a + s;
        r = s;
    } else {
        const int64_t m = (int64_t)((uint64_t)a << 1) | (s & 1);
        l = (m + s) >> 1;
        r = (m - s) >> 1;
    }
    return dec_mean(2, [=](int c) { return fl_scale(c ? r : l, bps); });
}

// Samples i0, i0 + di, ... of a frame to its file's output `out` (normalised by peak_bits when normalize); returns the largest |y| bits.
DSPX_HD unsigned fl_mix_frame(const dspx_flac_frame &fr, int bps, const void *samples, float *out, bool normalize,
                              unsigned peak_bits, int i0, int di)
{
    unsigned peak = 0;
    for (int i = i0; i < fr.block_size; i += di) {
        float y = fl_mix(fr, bps, samples, i);
        const unsigned u = rs_abs_bits(y);
        peak = u > peak ? u : peak;
        if (normalize) y = dec_normalize(y, peak_bits);
        out[fr.out_start + i] = y;
    }
    return peak;
}

DSPX_HD void fl_divide(const dspx_flac_frame &fr, float *out, unsigned peak_bits, int i0, int di)
{
    for (int i = i0; i < fr.block_size; i += di) out[fr.out_start + i] = dec_normalize(out[fr.out_start + i], peak_bits);
}

#if defined(__CUDACC__) && !defined(DSPX_EMU)
// grid ceil(n_frames / FL_THREADS): thread = frame.  samples: the workspace's sample region.
__global__ void __launch_bounds__(FL_THREADS) flac_frame_kernel(const unsigned char *in, const dspx_flac_file *files,
                                                                const dspx_flac_frame *frames, int64_t n_frames,
                                                                char *samples, int32_t *status)
{
    __shared__ uint16_t crc_table[256];
    __shared__ int32_t coef[FL_THREADS][FL_MAX_ORDER + 1];
    for (int i = threadIdx.x; i < 256; i += FL_THREADS) crc_table[i] = fl_crc16_entry(i);
    __syncthreads();
    const int64_t f = (int64_t)blockIdx.x * FL_THREADS + threadIdx.x;
    if (f >= n_frames) return;
    const dspx_flac_frame fr = frames[f];
    const dspx_flac_file &file = files[fr.file];
    status[f] = fl_frame(in + file.in_offset, fr, file.bps, samples + file.ws_start + fr.ws_offset, coef[threadIdx.x],
                         crc_table);
}

// grid n_frames: CTA = frame (its offsets relative to its file's row).  FL_STORE / FL_PEAK decode the frame's outputs
// (FL_PEAK folds |y| into peaks[file]); FL_NORM divides the stored outputs by that peak.  Frames with a non-zero status
// are skipped.
__global__ void __launch_bounds__(FL_MIX_THREADS) flac_mix_kernel(const dspx_flac_file *files, const dspx_flac_frame *frames,
                                                                  const char *samples, const int32_t *status, float *out,
                                                                  unsigned *peaks, int mode)
{
    const int64_t f = blockIdx.x;
    if (status[f]) return;
    const dspx_flac_frame fr = frames[f];
    if (mode == FL_NORM) {
        fl_divide(fr, out + files[fr.file].out_start, peaks[fr.file], threadIdx.x, FL_MIX_THREADS);
        return;
    }
    const dspx_flac_file &file = files[fr.file];
    unsigned peak = fl_mix_frame(fr, file.bps, samples + file.ws_start + fr.ws_offset, out + file.out_start, false, 0u,
                                 threadIdx.x, FL_MIX_THREADS);
    if (mode == FL_PEAK) {
        peak = __reduce_max_sync(0xffffffffu, peak);
        if ((threadIdx.x & 31) == 0 && peak) atomicMax(&peaks[fr.file], peak);
    }
}
#endif

// ---- host: stream parsing (dspx_flac_layout) ----

inline uint8_t fl_crc8(const unsigned char *p, int64_t n)
{
    unsigned c = 0;
    for (int64_t i = 0; i < n; i++) {
        c ^= p[i];
        for (int k = 0; k < 8; k++) c = (c & 0x80u) ? ((c << 1) ^ 0x07u) & 0xffu : (c << 1) & 0xffu;
    }
    return (uint8_t)c;
}

struct FlStreamInfo {
    int rate, channels, bps;
    int64_t total;
};

struct FlHeader {
    int len;              // header bytes through the CRC-8
    int block, assignment, variable;
    uint64_t number;
};

// The frame header at p[0 .. n) when it is a valid one for this stream (its CRC-8 checked when check_crc), else
// len == 0.
inline FlHeader fl_parse_header(const unsigned char *p, int64_t n, const FlStreamInfo &si, bool check_crc)
{
    FlHeader h{0, 0, 0, 0, 0};
    if (n < 6 || p[0] != 0xff || (p[1] & 0xfe) != 0xf8) return h;
    const int bs = p[2] >> 4, rc = p[2] & 15, asg = p[3] >> 4, ss = (p[3] >> 1) & 7;
    if (bs == 0 || rc == 15 || asg > 10 || ss == 3 || (p[3] & 1)) return h;
    if (fl_channels(asg) != si.channels) return h;
    static const int ss_bits[8] = {0, 8, 12, 0, 16, 20, 24, 32};
    if (ss != 0 && ss_bits[ss] != si.bps) return h;
    // UTF-8-like coded number: 1 .. 7 bytes
    int64_t at = 4;
    const unsigned b0 = p[at++];
    int extra;
    uint64_t v;
    if (b0 < 0x80) { extra = 0; v = b0; }
    else if ((b0 & 0xe0) == 0xc0) { extra = 1; v = b0 & 0x1f; }
    else if ((b0 & 0xf0) == 0xe0) { extra = 2; v = b0 & 0x0f; }
    else if ((b0 & 0xf8) == 0xf0) { extra = 3; v = b0 & 0x07; }
    else if ((b0 & 0xfc) == 0xf8) { extra = 4; v = b0 & 0x03; }
    else if ((b0 & 0xfe) == 0xfc) { extra = 5; v = b0 & 0x01; }
    else if (b0 == 0xfe) { extra = 6; v = 0; }
    else return h;
    const int variable = p[1] & 1;
    if (!variable && extra > 5) return h;               // a frame number has at most 31 bits
    if (at + extra > n) return h;
    for (int i = 0; i < extra; i++) {
        const unsigned c = p[at++];
        if ((c & 0xc0) != 0x80) return h;
        v = v << 6 | (c & 0x3f);
    }
    int block;
    if (bs == 1) block = 192;
    else if (bs <= 5) block = 576 << (bs - 2);
    else if (bs >= 8) block = 256 << (bs - 8);
    else {
        const int k = bs == 6 ? 1 : 2;
        if (at + k > n) return h;
        block = (k == 1 ? p[at] : p[at] << 8 | p[at + 1]) + 1;
        at += k;
        if (block > FL_MAX_BLOCK) return h;
    }
    int rate = si.rate;
    if (rc >= 12) {
        const int k = rc == 12 ? 1 : 2;
        if (at + k > n) return h;
        const int r = k == 1 ? p[at] : p[at] << 8 | p[at + 1];
        at += k;
        rate = rc == 12 ? r * 1000 : rc == 13 ? r : r * 10;
    } else if (rc) {
        static const int rates[12] = {0, 88200, 176400, 192000, 8000, 16000, 22050, 24000, 32000, 44100, 48000, 96000};
        rate = rates[rc];
    }
    if (rate != si.rate) return h;
    if (at + 1 > n || (check_crc && fl_crc8(p, at) != p[at])) return h;
    h.len = (int)at + 1;
    h.block = block;
    h.assignment = asg;
    h.variable = variable;
    h.number = v;
    return h;
}

struct FlFile {
    FlStreamInfo si;
    std::vector<dspx_flac_frame> frames;   // offsets relative to the file, its first output sample and its workspace
    int64_t samples;
    int64_t ws_bytes;                      // its frames' integers: their workspace_offsets end here
};

// The stream's end: the file's end without a trailing ID3v1 tag ("TAG", 128 bytes) and APEv2 tag (a 32-byte
// "APETAGEX" footer whose size covers the items and the footer, plus a 32-byte header when its flags say so), which
// taggers append after the last frame.
inline int64_t fl_stream_end(const unsigned char *p, int64_t size)
{
    if (size >= 128 && !memcmp(p + size - 128, "TAG", 3)) size -= 128;
    if (size >= 32 && !memcmp(p + size - 32, "APETAGEX", 8)) {
        const unsigned char *t = p + size - 32;
        const int64_t len = (int64_t)t[12] | (int64_t)t[13] << 8 | (int64_t)t[14] << 16 | (int64_t)t[15] << 24;
        const int64_t tag = len + ((t[23] & 0x80) ? 32 : 0);
        if (len >= 32 && tag <= size) size -= tag;
    }
    return size;
}

// Whether the valid header g at q is followed by the valid header of the frame after it.
inline bool fl_followed(const unsigned char *p, int64_t size, int64_t q, const FlHeader &g, const FlStreamInfo &si)
{
    const uint64_t want = g.number + (g.variable ? (uint64_t)g.block : 1);
    for (int64_t r = q + g.len; r + 1 < size; r++) {
        const void *hit = memchr(p + r, 0xff, (size_t)(size - 1 - r));
        if (!hit) return false;
        r = static_cast<const unsigned char *>(hit) - p;
        if ((p[r + 1] & 0xfe) != 0xf8) continue;
        const FlHeader n = fl_parse_header(p + r, size - r, si, true);
        if (n.len && n.variable == g.variable && n.number == want) return true;
    }
    return false;
}

// Parses one file; returns nullptr, or an error message with *where set to the byte offset of the problem.
inline const char *fl_parse_file(const unsigned char *p, int64_t size, FlFile &f, int64_t *where)
{
    int64_t pos = 0;
    *where = 0;
    if (size >= 10 && p[0] == 'I' && p[1] == 'D' && p[2] == '3') {
        if ((p[6] | p[7] | p[8] | p[9]) & 0x80) return "bad ID3v2 tag size";
        pos = 10 + ((int64_t)p[6] << 21 | (int64_t)p[7] << 14 | (int64_t)p[8] << 7 | p[9]) + ((p[5] & 0x10) ? 10 : 0);
    }
    *where = pos;
    if (pos + 4 > size || memcmp(p + pos, "fLaC", 4)) return "no fLaC stream marker";
    pos += 4;
    bool first = true, last = false;
    while (!last) {
        *where = pos;
        if (pos + 4 > size) return "metadata block header past the end of the file";
        last = p[pos] >> 7;
        const int type = p[pos] & 0x7f;
        const int64_t len = (int64_t)p[pos + 1] << 16 | p[pos + 2] << 8 | p[pos + 3];
        if (type == 127) return "invalid metadata block type 127";
        if (first != (type == 0)) return first ? "STREAMINFO is not the first metadata block" : "second STREAMINFO block";
        if (pos + 4 + len > size) return "metadata block past the end of the file";
        if (type == 0) {
            if (len != 34) return "STREAMINFO block length is not 34";
            const unsigned char *s = p + pos + 4;
            f.si.rate = s[10] << 12 | s[11] << 4 | s[12] >> 4;
            f.si.channels = ((s[12] >> 1) & 7) + 1;
            f.si.bps = ((s[12] & 1) << 4 | s[13] >> 4) + 1;
            f.si.total = (int64_t)(s[13] & 15) << 32 | (int64_t)s[14] << 24 | s[15] << 16 | s[16] << 8 | s[17];
            if (f.si.rate == 0) return "STREAMINFO sample rate 0";
            if (f.si.bps < 4) return "STREAMINFO bits per sample below 4";
        }
        first = false;
        pos += 4 + len;
    }
    if (pos < size) size = std::max(pos, fl_stream_end(p, size));
    f.samples = 0;
    f.ws_bytes = 0;
    f.frames.clear();
    int variable = -1;
    uint64_t number0 = 0;         // the first frame's number: a stream cut from a longer one need not start at 0
    while (pos < size) {
        *where = pos;
        const FlHeader h = fl_parse_header(p + pos, size - pos, f.si, true);
        if (!h.len) return "not a valid frame header";
        if (variable < 0) {       // every later frame starts where the search below found its expected number
            variable = h.variable;
            number0 = h.number;
        }
        const uint64_t next = number0 + (variable ? (uint64_t)(f.samples + h.block) : (uint64_t)f.frames.size() + 1);
        int64_t end = size;
        // The next frame: a sync code, a valid header and the expected number.  When none follows, this frame would
        // run to the end of the stream.  A damaged frame header is then reported at its own offset rather than as a
        // CRC-16 error of this frame: a header there with the expected number that fails only its CRC-8, or -- when
        // frames are evidently missing (STREAMINFO's total is not reached, or a valid header numbered past the
        // expected one follows, and so does the valid header after that: one alone may be sync-like residual data)
        // -- the first header that fails only its CRC-8.
        int64_t damaged = -1, damaged_any = -1, later = -1;
        const bool short_total = f.si.total != 0 && f.samples + h.block < f.si.total;
        for (int pass = 0; pass < 2 && end == size && damaged < 0; pass++)
            for (int64_t q = pos + h.len; q + 1 < size; q++) {
                const void *hit = memchr(p + q, 0xff, (size_t)(size - 1 - q));
                if (!hit) break;
                q = static_cast<const unsigned char *>(hit) - p;
                if ((p[q + 1] & 0xfe) != 0xf8) continue;
                const FlHeader g = fl_parse_header(p + q, size - q, f.si, pass == 0);
                if (!g.len || g.variable != variable) continue;
                if (pass == 0 && g.number == next) {
                    end = q;
                    break;
                }
                if (pass == 0 && g.number > next && later < 0 && fl_followed(p, size, q, g, f.si)) later = q;
                if (pass == 1 && g.number == next) {
                    damaged = q;
                    break;
                }
                if (pass == 1 && damaged_any < 0) damaged_any = q;
            }
        if (damaged < 0 && (short_total || later >= 0)) damaged = damaged_any;
        if (damaged >= 0) {
            *where = damaged;
            return "damaged frame header (CRC-8 mismatch)";
        }
        if (end - pos < h.len + 2) return "frame shorter than its header and CRC-16";
        if (end - pos > 0x7fffffff) return "frame longer than 2^31 bytes";
        dspx_flac_frame fr{};
        fr.in_offset = pos;
        fr.out_start = f.samples;
        fr.ws_offset = f.ws_bytes;
        fr.in_bytes = (int32_t)(end - pos);
        fr.header_bytes = h.len;
        fr.block_size = h.block;
        fr.assignment = h.assignment;
        f.frames.push_back(fr);
        f.samples += h.block;
        f.ws_bytes += fl_ws_bytes(f.si.bps, h.assignment, h.block);
        pos = end;
    }
    *where = size;
    if (f.frames.empty()) return "no audio frames";
    if (f.si.total != 0 && f.si.total != f.samples) return "STREAMINFO total samples differ from the frames' block sizes";
    return nullptr;
}

}  // namespace dspx
