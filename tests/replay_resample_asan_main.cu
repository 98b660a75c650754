// AddressSanitizer run of the resampler's tile decomposition (csrc/emu.cu replays rs_stage_row, rs_stage_phase and rs_group): each
// tile's inputs and table rows go into a heap buffer of exactly the kernel's dynamic shared-memory size, and the input
// and output buffers have exactly the clips' lengths, so a tile span that is too short, or a read or write past a clip,
// is reported.  Lengths sit on the tile edges; 44099/44100 has a 3.7 MB table (staged row by row from the global table).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../include/dspx.h"
extern "C" int emu_resample(int64_t up, int64_t down, const float *window, int64_t n_window, const void *in, int dtype,
                            int64_t n_clips, int64_t n_in, int64_t in_stride, int normalize, float *out, int64_t out_stride,
                            const dspx_resample_clip *table);
extern "C" int emu_resample_shape(int64_t up, int64_t down, const float *window, int64_t n_window, int64_t *out);

// Any window of scipy's length will do here: the test is about addresses, not values.
static std::vector<float> window_for(int64_t up, int64_t down)
{
    int64_t g = up, b = down;
    while (b) { const int64_t t = g % b; g = b; b = t; }
    const int64_t m = (up > down ? up : down) / g;
    std::vector<float> w(2 * 10 * m + 1);
    for (size_t i = 0; i < w.size(); i++) w[i] = (float)std::sin(0.001 * (double)i) / (float)m;
    return w;
}

int main()
{
    const int64_t ratios[][2] = {{16000, 44100}, {8000, 44100}, {22050, 44100}, {44100, 22050}, {7, 3}, {3, 7}, {44099, 44100}};
    for (const auto &r : ratios) {
        const int64_t up = r[0], down = r[1];
        const std::vector<float> w = window_for(up, down);
        int64_t shape[8];
        if (emu_resample_shape(up, down, w.data(), (int64_t)w.size(), shape) != 0) { printf("resample %lld/%lld: shape failed\n", (long long)up, (long long)down); return 1; }
        const int64_t S = shape[1], NR = shape[2], U = shape[6];
        int64_t g = up, b = down;
        while (b) { const int64_t t = g % b; g = b; b = t; }
        const int64_t u = up / g, d = down / g;
        // outputs: 1, S - 1, S, S + 1 columns, one full row, one full tile of rows, +- 1 around it
        const int64_t outs[] = {1, S - 1, S, S + 1, U, U * NR - 1, U * NR, U * NR + 1};
        std::vector<int64_t> lengths;
        for (int64_t o : outs) {
            if (o < 1 || o > 4000000) continue;
            const int64_t n = (o * d + u - 1) / u;        // shortest input with at least o outputs
            lengths.push_back(n);
            if (n > 1) lengths.push_back(n - 1);
        }
        const int64_t n = (int64_t)lengths.size();
        std::vector<dspx_resample_clip> table(n);
        int64_t at_in = 0, at_out = 0;
        for (int64_t i = 0; i < n; i++) {
            const int64_t n_out = (lengths[i] * u + d - 1) / d;
            table[i] = {at_in, lengths[i], at_out, n_out};
            at_in += lengths[i];
            at_out += (n_out + 3) & ~(int64_t)3;
        }
        std::vector<int16_t> pcm(at_in);
        for (auto &v : pcm) v = (int16_t)(rand() % 65536 - 32768);
        std::vector<float> f32(at_in);
        for (auto &v : f32) v = (float)rand() / RAND_MAX - 0.5f;
        std::vector<float> out(table[n - 1].out_start + table[n - 1].out_length);
        int rc = emu_resample(up, down, w.data(), (int64_t)w.size(), pcm.data(), DSPX_DTYPE_PCM16, n, 0, 0, 1, out.data(), 0, table.data());
        double s = 0;
        for (float v : out) s += v;
        const int rc2 = emu_resample(up, down, w.data(), (int64_t)w.size(), f32.data(), DSPX_DTYPE_F32, n, 0, 0, 0, out.data(), 0, table.data());
        for (float v : out) s += v;
        // one clip alone, strided: the last clip's length, in a buffer that ends with it
        const int64_t last = lengths[n - 1], last_out = table[n - 1].out_length;
        std::vector<float> one(last), one_out(last_out);
        for (auto &v : one) v = (float)rand() / RAND_MAX - 0.5f;
        const int rc3 = emu_resample(up, down, w.data(), (int64_t)w.size(), one.data(), DSPX_DTYPE_F32, 1, last, last, 1, one_out.data(), last_out, nullptr);
        printf("resample %lld/%lld: clips %lld rc %d finite %d\n", (long long)up, (long long)down, (long long)n, rc | rc2 | rc3,
               (int)std::isfinite(s));
    }
    return 0;
}
