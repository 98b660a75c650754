// feat_warp8_x2.cuh -- n_fft 4096 on the warp8 machinery (the reference's extended grid has 4096-point frames:
// logs/precompute_mfcc_fl4096_hl256.log; reference ops: src/dsp/mfcc.py:86-109 as for feat_warp8.cuh).
//
// A 4096-sample frame x is the radix-2 combination of the transforms of its even and odd samples,
//     F[k] = E[k] + W_4096^k O[k],   F[2048 - k] = conj(E[k] - W_4096^k O[k]),        k = 0 .. 1024,
// and E, O are transforms of 2048 real samples each -- exactly what one frame pair of the radix-16 variant computes.
// So ONE frame rides in the (A, B) halves of the packed lanes: A = even samples, B = odd samples.  A 128-bit load
// x[4m .. 4m+3] is already (re A, re B, im A, im B) of complex point m of the two packed-real sequences; passes 1-3
// are those of feat_warp8 (R1 = 16); the split then yields E and O as complex values, the combination above gives
// four bins per slot (k, 2048 - k, 1024 - k, 1024 + k), and the mel / log / DCT tail runs on one frame
// (the power tile holds one float per bin instead of an (A, B) pair).
#pragma once

#include "feat_warp8.cuh"

namespace dspx {

struct W8Power4 {            // |F|^2 of the four bins of every slot of one pass-3 unit
    float p[9][4];
};

// ---- phase A: 16 float4 loads per set, pre-emphasis, window, radix 16, twiddle, store -------------------
// AL4: every float4 lies inside the frame and is 16-byte aligned (frame_length >= 4096, hop and stride multiples of 4)
template <bool PRE, bool AL4>
DSPX_HD void w8x2_pass1(const W8Ctx &c, int lane)
{
    constexpr int R1 = 16;
#pragma unroll
    for (int s = 0; s < 2; s++) {
        const int tid = lane + 32 * s;
        const float *pa = c.fa + 4 * tid;
        float4 x[R1];
        float pv[R1];
#pragma unroll
        for (int a = 0; a < R1; a++) {
            const int n0 = 256 * a + 4 * tid;
            if (AL4) {
                x[a] = *reinterpret_cast<const float4 *>(pa + 256 * a);
            } else {
                x[a].x = n0 < c.take ? pa[256 * a] : 0.f;
                x[a].y = n0 + 1 < c.take ? pa[256 * a + 1] : 0.f;
                x[a].z = n0 + 2 < c.take ? pa[256 * a + 2] : 0.f;
                x[a].w = n0 + 3 < c.take ? pa[256 * a + 3] : 0.f;
            }
            if (PRE) {
                const bool edge = c.firstA && n0 == 0;                   // sample 0 of the clip has no predecessor
                pv[a] = (n0 < c.take && !edge) ? pa[256 * a - 1] : 0.f;
            }
        }
        float2 re[R1], im[R1];
#pragma unroll
        for (int a = 0; a < R1; a++) {
            float y0 = x[a].x, y1 = x[a].y, y2 = x[a].z, y3 = x[a].w;
            if (PRE) {                                                   // rounded product, rounded difference (mfcc.py:87-88)
                y3 = DSPX_FSUB_RN(x[a].w, DSPX_FMUL_RN(c.alpha, x[a].z));
                y2 = DSPX_FSUB_RN(x[a].z, DSPX_FMUL_RN(c.alpha, x[a].y));
                y1 = DSPX_FSUB_RN(x[a].y, DSPX_FMUL_RN(c.alpha, x[a].x));
                y0 = DSPX_FSUB_RN(x[a].x, DSPX_FMUL_RN(c.alpha, pv[a]));
            }
            const float4 w = c.win4[(s * R1 + a) * 32 + lane];            // 0.5 w[4m .. 4m+3]
            re[a] = mul2(make_float2(y0, y1), make_float2(w.x, w.y));     // (even, odd) sequence: real parts
            im[a] = mul2(make_float2(y2, y3), make_float2(w.z, w.w));     //                        imaginary parts
        }
        dftn(re, im);
        c.xbuf[w8_addr(0, tid >> 3, tid & 7)] = make_float4(re[0].x, re[0].y, im[0].x, im[0].y);
#pragma unroll
        for (int ka = 1; ka < R1; ka++) {
            const float2 w = c.tw1[(s * (R1 - 1) + ka - 1) * 32 + lane];  // exp(-2 pi i tid ka / 1024)
            cmul2(re[ka], im[ka], w.x, w.y);
            c.xbuf[w8_addr(ka, tid >> 3, tid & 7)] = make_float4(re[ka].x, re[ka].y, im[ka].x, im[ka].y);
        }
    }
}

// packed-real split of both sequences, then their radix-2 combination: a = Z[k], b = Z[M - k] (M = 1024),
// w = exp(-2 pi i k / 2048), w2 = exp(-2 pi i k / 4096)
DSPX_HD void w8x2_split(float2 ar, float2 ai, float2 br, float2 bi, float2 w, float2 w2, float (&p)[4])
{
    const float2 er = add2(ar, br), ei = sub2(ai, bi);
    const float2 orr = add2(ai, bi), oi = sub2(br, ar);
    const float2 wr = bc2(w.x), wi = bc2(w.y);
    const float2 tr = fma2(neg2(oi), wi, mul2(orr, wr));
    const float2 ti = fma2(orr, wi, mul2(oi, wr));
    const float2 xr = add2(er, tr), xi = add2(ei, ti);          // (E[k], O[k])
    const float2 yr = sub2(er, tr), yi = sub2(ti, ei);          // (E[M-k], O[M-k])
    // F[k] = E[k] + W O[k], F[2M - k] = conj(E[k] - W O[k])
    const float t2r = fmaf(w2.x, xr.y, -w2.y * xi.y), t2i = fmaf(w2.x, xi.y, w2.y * xr.y);
    const float2 fr = add2(bc2(xr.x), make_float2(t2r, -t2r)), fi = add2(bc2(xi.x), make_float2(t2i, -t2i));
    const float2 pk = fma2(fi, fi, mul2(fr, fr));
    p[0] = pk.x;
    p[1] = pk.y;
    // mirror slot: exp(-2 pi i (M - k) / 4096) = -i conj(W) = (-w2.y, -w2.x)
    const float u2r = fmaf(-w2.y, yr.y, w2.x * yi.y), u2i = fmaf(-w2.y, yi.y, -w2.x * yr.y);
    const float2 gr = add2(bc2(yr.x), make_float2(u2r, -u2r)), gi = add2(bc2(yi.x), make_float2(u2i, -u2i));
    const float2 pm = fma2(gi, gi, mul2(gr, gr));
    p[2] = pm.x;                                                 // F[M - k]
    p[3] = pm.y;                                                 // F[M + k]
}

// ---- phase C: as w8_pass3<16>, with the combined split ------------------------------------------------
DSPX_HD void w8x2_pass3(const W8Ctx &c, int lane, int w, W8Power4 &pw)
{
    using G = W8Geo<16>;
    const int u = lane + 32 * w;
    const bool l0 = u == 0;
    const int j1 = u, j2 = l0 ? G::J / 2 : G::J - u;
    float2 r1[8], i1[8], r2[8], i2[8];
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const float4 v = c.xbuf[w8_addr(j1 & 15, j1 >> G::LOG_R1, q)];
        r1[q] = make_float2(v.x, v.y);
        i1[q] = make_float2(v.z, v.w);
        const float4 t = c.xbuf[w8_addr(j2 & 15, j2 >> G::LOG_R1, q)];
        r2[q] = make_float2(t.x, t.y);
        i2[q] = make_float2(t.z, t.w);
    }
    dft8(r1, i1);
    dft8(r2, i2);
    const float2 *ptw = c.ptw + w * 9 * 32, *ptw2 = c.ptw2 + w * 9 * 32;
#pragma unroll
    for (int m = 0; m < 8; m++) {
        float2 ar = r1[m], ai = i1[m];
        if (m >= 5) { ar = sel2(l0, r2[m - 5], ar); ai = sel2(l0, i2[m - 5], ai); }
        const int b0 = m == 0 ? 0 : (m <= 4 ? 8 - m : 0);
        float2 br, bi;
        if (m <= 4) { br = sel2(l0, r1[b0 & 7], r2[7 - m]); bi = sel2(l0, i1[b0 & 7], i2[7 - m]); }
        else { br = sel2(l0, r2[12 - m], r2[7 - m]); bi = sel2(l0, i2[12 - m], i2[7 - m]); }
        w8x2_split(ar, ai, br, bi, ptw[m * 32 + lane], ptw2[m * 32 + lane], pw.p[m]);
    }
    if (l0) w8x2_split(r2[3], i2[3], r2[4], i2[4], ptw[8 * 32], ptw2[8 * 32], pw.p[8]);
}

// ---- phase D: four powers per slot into the scalar tile (chunk order, table ppos4) ----------------------
DSPX_HD void w8x2_store_power(const W8Ctx &c, int lane, int w, const W8Power4 &pw)
{
    float *pb = reinterpret_cast<float *>(c.pbuf);
    const int4 *pp = c.ppos4 + w * 9 * 32;
#pragma unroll
    for (int m = 0; m < 8; m++) {
        const int4 q = pp[m * 32 + lane];
        pb[q.x] = pw.p[m][0];
        pb[q.y] = pw.p[m][1];
        pb[q.z] = pw.p[m][2];
        pb[q.w] = pw.p[m][3];
    }
    if (lane + 32 * w == 0) {
        const int4 q = pp[8 * 32];
        pb[q.x] = pw.p[8][0];
        pb[q.y] = pw.p[8][1];
        pb[q.z] = pw.p[8][2];
        pb[q.w] = pw.p[8][3];
    }
}

// ---- phase E: mel chunks of one frame (eight floats per chunk, weights a0 b0 .. a7 b7 unrotated) ---------
DSPX_HD void w8x2_mel_chunks(const W8Ctx &c, int lane)
{
    const float *pb = reinterpret_cast<const float *>(c.pbuf);
    float sa = 0.f, sb = 0.f;
    for (int r = 0; r < c.rounds; r++) {
        const int ch = lane * c.rounds + r;
        const int flag = c.cflag[ch];
        const float4 *pp = reinterpret_cast<const float4 *>(pb + ch * W8_CSTRIDE);
        const float4 *ww = reinterpret_cast<const float4 *>(c.cw + ch * W8_WROW);
        const float4 p0 = pp[0], p1 = pp[1], w0 = ww[0], w1 = ww[1], w2 = ww[2], w3 = ww[3];
        float ca = p0.x * w0.x, cb = p0.x * w0.y;
        ca = fmaf(p0.y, w0.z, ca); cb = fmaf(p0.y, w0.w, cb);
        ca = fmaf(p0.z, w1.x, ca); cb = fmaf(p0.z, w1.y, cb);
        ca = fmaf(p0.w, w1.z, ca); cb = fmaf(p0.w, w1.w, cb);
        ca = fmaf(p1.x, w2.x, ca); cb = fmaf(p1.x, w2.y, cb);
        ca = fmaf(p1.y, w2.z, ca); cb = fmaf(p1.y, w2.w, cb);
        ca = fmaf(p1.z, w3.x, ca); cb = fmaf(p1.z, w3.y, cb);
        ca = fmaf(p1.w, w3.z, ca); cb = fmaf(p1.w, w3.w, cb);
        if (flag & 1) { sa = ca; sb = cb; }
        else { sa += ca; sb += cb; }
        if (flag & 2) {
            c.seg[(flag >> 8) & 0xfff] = make_float2(sa, 0.f);
            c.seg[(unsigned)flag >> 20] = make_float2(sb, 0.f);
        }
    }
}

// item = clip * n_frames + frame: one frame per item, "frame B" does not exist
DSPX_HD void w8x2_set_item(const W8Params &p, W8Ctx &c, uint32_t item)
{
    const uint32_t clip = item / p.pairs_per_clip, t = item - clip * p.pairs_per_clip;      // pairs_per_clip = n_frames here
    c.validB = 0;
    const float *base = p.clips + (int64_t)clip * p.clip_stride;
    c.fa = base + (int64_t)t * p.hop;
    c.fb = c.fa;
    c.firstA = t == 0;
    c.firstB = c.firstA;
    const int64_t row = (int64_t)clip * p.n_frames + t;
    c.logmelA = p.logmel ? p.logmel + (int64_t)clip * p.n_frames * p.n_mels + (int64_t)t * p.lm_ts : nullptr;
    c.logmelB = nullptr;
    c.lm_fs = p.lm_fs;
    c.mfccA = p.mfcc ? p.mfcc + row * p.n_mfcc : nullptr;
    c.mfccB = nullptr;
    c.stftA = c.stftB = nullptr;
    c.eacc = nullptr;
}

#if defined(__CUDACC__) && !defined(DSPX_EMU)
template <bool PRE, bool AL4>
__global__ void __launch_bounds__(W8_WARPS * 32, 1) feat_warp8_x2_kernel(const W8Params p)
{
    constexpr int NW = W8_WARPS;
    extern __shared__ __align__(16) float w8_smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wf = w8_warp_floats(p.tb, p.n_mels);
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
        w8x2_set_item(p, c, item);
        w8x2_pass1<PRE, AL4>(c, lane);
        __syncwarp();
        w8_pass2<16>(c, lane);
        __syncwarp();
        W8Power4 pw[2];
#pragma unroll
        for (int w = 0; w < 2; w++) w8x2_pass3(c, lane, w, pw[w]);
        __syncwarp();
#pragma unroll
        for (int w = 0; w < 2; w++) w8x2_store_power(c, lane, w, pw[w]);
        __syncwarp();
        w8x2_mel_chunks(c, lane);
        __syncwarp();
        w8_logmel(c, lane);
        __syncwarp();
        if (c.mfccA) {
            for (int c0 = 0; c0 < c.n_mfcc; c0 += c.cw_lanes) {
                float2 acc = w8_dct_partial(c, lane, c0);
                if (c.cw_lanes == 16) {
                    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16);
                    acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
                }
                w8_dct_store(c, lane, c0, acc);
            }
            __syncwarp();
        }
    }
}

template <bool PRE, bool AL4>
inline int w8x2_launch(const W8Params &p, const W8PlanData *pd, int device, int sm_count, cudaStream_t st)
{
    static std::atomic<unsigned char> optin[64];
    DSPX_CUDA_CHECK(optin_max_smem(feat_warp8_x2_kernel<PRE, AL4>, optin, device));
    int64_t ctas = ((int64_t)p.n_items + W8_WARPS - 1) / W8_WARPS;
    if (ctas > sm_count) ctas = sm_count;
    feat_warp8_x2_kernel<PRE, AL4><<<(unsigned)ctas, W8_WARPS * 32, pd->smem, st>>>(p);
    DSPX_CUDA_CHECK(cudaGetLastError());
    return DSPX_OK;
}

// features of 4096-point frames; one launch, n_clips * n_frames items (al4: the W8_X2_AL4 path)
inline int launch_warp8_x2(const dspx_plan *pl, bool al4, const float *clips, int64_t n_clips, int64_t clip_stride, int64_t T,
                           float *logmel, float *mfcc, cudaStream_t st, int nchw)
{
    const W8PlanData *pd = static_cast<const W8PlanData *>(pl->fast_host);
    W8Params p = w8_batch_params(pl, clips, n_clips, clip_stride, T, logmel, mfcc, nchw);
    p.pairs_per_clip = (uint32_t)T;                          // one frame per item
    p.n_items = (uint32_t)(n_clips * T);
    const bool pre = pl->cfg.pre_emphasis > 0.0;
    if (al4) return pre ? w8x2_launch<true, true>(p, pd, pl->device, pl->sm_count, st) : w8x2_launch<false, true>(p, pd, pl->device, pl->sm_count, st);
    return pre ? w8x2_launch<true, false>(p, pd, pl->device, pl->sm_count, st) : w8x2_launch<false, false>(p, pd, pl->device, pl->sm_count, st);
}
#endif

}  // namespace dspx
