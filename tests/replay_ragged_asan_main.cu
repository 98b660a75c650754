// AddressSanitizer run of the RAGGED warp8 mapping (csrc/emu.cu replays the kernel's w8_set_item): every buffer has
// exactly the size dspx_ragged_layout gives it, so a read past the last clip or a write past total_frames is reported.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../include/dspx.h"
extern "C" int emu_features_warp8_ragged(const dspx_config *cfg, const float *samples, const dspx_ragged_clip *table,
                                         int64_t n_clips, float *logmel, float *mfcc);
int main() {
    struct Case { int fl, hop, nfft; };
    const Case cases[] = {{1024, 512, 0}, {512, 256, 0}, {2048, 512, 0}, {1024, 441, 0}, {400, 160, 512}};
    for (const Case &c : cases) {
        dspx_config cfg{44100, c.fl, c.hop, c.nfft, 40, 13, 0.0, -1.0, 0.97, 0, 0};
        // one frame, an odd frame count, frame_length + hop - 1, a longer clip, one frame again (the buffer ends there)
        const int64_t lengths[] = {c.fl, c.fl + 2 * c.hop, c.fl + c.hop - 1, 9002, c.fl};
        const int64_t n = 5;
        std::vector<dspx_ragged_clip> table(n);          // what dspx_ragged_layout fills (libdspx.so is not linked here)
        int64_t at = 0, total = 0, pairs = 0;
        for (int64_t i = 0; i < n; i++) {
            const int64_t frames = 1 + (lengths[i] - c.fl) / c.hop;
            table[i] = {at, lengths[i], frames, total, pairs};
            at += (lengths[i] + 1) & ~(int64_t)1;
            total += frames;
            pairs += (frames + 1) / 2;
        }
        std::vector<float> samples(table[n - 1].start + lengths[n - 1]);
        for (auto &v : samples) v = (float)rand() / RAND_MAX - 0.5f;
        std::vector<float> lm(total * 40), mf(total * 13);
        const int rc = emu_features_warp8_ragged(&cfg, samples.data(), table.data(), n, lm.data(), mf.data());
        double s = 0;
        for (float v : mf) s += v;
        for (float v : lm) s += v;
        printf("ragged fl %d hop %d: frames %lld rc %d finite %d\n", c.fl, c.hop, (long long)total, rc, (int)std::isfinite(s));
    }
    return 0;
}
