#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
#include "../include/dspx.h"
extern "C" int emu_features_generic(const dspx_config *cfg, const float *clips, int64_t n_clips, int64_t clip_len, int64_t clip_stride, int stft_mode, int stft_pre, float *logmel, float *mfcc, float *stft_out, int fpc);
extern "C" int emu_features_warp8(const dspx_config *cfg, const float *clips, int64_t n_clips, int64_t clip_len, int64_t clip_stride, float *logmel, float *mfcc, float *stft_out, int stft_pre);
int main() {
    struct Case { int fl, hop, nfft, mels, mfcc; double pre; };
    Case cases[] = {{512,256,0,40,13,0.97},{1024,512,0,40,13,0.97},{2048,1024,0,40,13,0.97},{1024,300,0,128,40,0.0},{512,512,0,128,13,0.97},{2048,256,0,13,13,0.97},{1000,300,0,40,13,0.97},{400,160,512,40,13,0.97},{64,32,0,10,5,0.97},{1024,2048,0,1,1,0.97},{4096,1024,0,40,13,0.97}};
    for (auto &c : cases) {
        const int64_t L = 9002 + (c.fl == 4096 ? 4000 : 0), n = 2;
        std::vector<float> clips(n * L);
        for (auto &v : clips) v = (float)rand() / RAND_MAX - 0.5f;
        dspx_config cfg{44100, c.fl, c.hop, c.nfft, c.mels, c.mfcc, 0.0, -1.0, c.pre, 0, 0};
        const int64_t T = 1 + (L - c.fl) / c.hop;
        // exact-size output buffers so that ASan sees any overrun
        std::vector<float> lm(n * T * c.mels), mf(n * T * c.mfcc);
        int P = 1; while (P < (c.nfft ? c.nfft : c.fl)) P <<= 1;
        std::vector<float> st(n * T * (P / 2 + 1) * 2);
        int r1 = emu_features_generic(&cfg, clips.data(), n, L, L, 0, 0, lm.data(), mf.data(), nullptr, 5);
        int r2 = emu_features_generic(&cfg, clips.data(), n, L, L, 1, 0, nullptr, nullptr, st.data(), 0);
        int r3 = emu_features_warp8(&cfg, clips.data(), n, L, L, lm.data(), mf.data(), nullptr, 0);
        if (r3 == 0) r3 = emu_features_warp8(&cfg, clips.data(), n, L, L, nullptr, nullptr, st.data(), 0);
        double s = 0; for (float v : mf) s += v;
        printf("fl %d hop %d mels %d: generic %d stft %d warp8 %d checksum %.3f finite %d\n", c.fl, c.hop, c.mels, r1, r2, r3, s, (int)std::isfinite(s));
    }
    return 0;
}
