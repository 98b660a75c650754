// AddressSanitizer run of the WAV decoder's tile decomposition (csrc/emu.cu replays dec_stage, dec_frames, dec_store and
// dec_divide): each tile's bytes go into a heap buffer of exactly the kernel's dynamic shared-memory size, and the input
// and output buffers end exactly where the last clip does, so a staged span that is too long, or a read or write past a
// clip, is reported.  Lengths sit on the tile edges, for 1, 3, 8 and 32 channels, every encoding, and PCM24 at odd lengths.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../include/dspx.h"
extern "C" int emu_decode(const void *in, const dspx_decode_clip *table, int64_t n_clips, int normalize, float *out);

static int bytes_of(int dtype)
{
    switch (dtype) {
    case DSPX_DTYPE_PCM8: return 1;
    case DSPX_DTYPE_PCM16: return 2;
    case DSPX_DTYPE_PCM24: return 3;
    case DSPX_DTYPE_F64: return 8;
    default: return 4;
    }
}

int main()
{
    const int dtypes[] = {DSPX_DTYPE_PCM8, DSPX_DTYPE_PCM16, DSPX_DTYPE_PCM24, DSPX_DTYPE_PCM32, DSPX_DTYPE_F32, DSPX_DTYPE_F64};
    const int chans[] = {1, 3, 8, 32};
    for (int dt : dtypes)
        for (int C : chans) {
            const int fb = C * bytes_of(dt);
            int tf = (16384 / fb) & ~15;                 // the kernel's tile (decode.cuh: dec_tile_frames)
            if (tf > 2048) tf = 2048;
            std::vector<int64_t> lengths = {1, 2, 15, 16, 17, tf - 1, tf, tf + 1, 2 * tf + 1, 3 * tf - 1};
            if (dt == DSPX_DTYPE_PCM24) lengths.insert(lengths.end(), {3, 5, 7, 33, 101});
            const int64_t n = (int64_t)lengths.size();
            std::vector<dspx_decode_clip> table(n);
            int64_t at_in = 0, at_out = 0;
            for (int64_t i = 0; i < n; i++) {
                at_in = (at_in + 15) & ~(int64_t)15;
                table[i] = {at_in, lengths[i], C, dt, at_out, lengths[i]};
                at_in += lengths[i] * fb;
                at_out += (lengths[i] + 3) & ~(int64_t)3;
            }
            std::vector<unsigned char> in(at_in);
            for (auto &v : in) v = (unsigned char)(rand() & 0x3f);   // no NaN or inf among the float encodings
            std::vector<float> out(table[n - 1].out_start + table[n - 1].out_length);
            int rc = 0;
            double s = 0;
            for (int normalize = 0; normalize < 2; normalize++) {
                rc |= emu_decode(in.data(), table.data(), n, normalize, out.data());
                for (float v : out) s += v;
            }
            printf("decode dtype %d channels %d: clips %lld rc %d finite %d\n", dt, C, (long long)n, rc, (int)std::isfinite(s));
        }
    return 0;
}
