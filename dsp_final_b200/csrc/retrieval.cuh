// retrieval.cuh -- clip-embedding statistics, cosine scoring and top-k selection.
//
//   embed stats  src/retrieval/retrieval.py:19-23,38-41  concat(mean_t, std_t), ddof 0
//   normalise    src/retrieval/retrieval.py:46-48        row / (||row|| + 1e-10)
//   score        src/retrieval/retrieval.py:49           q_norm . db_norm^T
//   select       src/retrieval/retrieval.py:65           argsort(-sims)[:, :k]
//   hit@k        src/retrieval/retrieval.py:66-70
//
// Scores are float64 and are accumulated left to right with fused multiply-adds,
// a fixed, documented operation sequence (DESIGN.md "Retrieval"), so indices are
// reproducible bit for bit including ties (ties -> lower database index, the stable
// argsort order).  The score matrix is never materialised: a CTA keeps the
// running top-k of 64 queries in shared memory while database tiles stream
// through; warps select with ballots against the current k-th score.
#pragma once

#include "dspx_internal.cuh"

namespace dspx {

constexpr int TK_WARPS = 8;
constexpr int TK_QPW = 8;                        // queries per warp
constexpr int TK_QPC = TK_WARPS * TK_QPW;        // queries per CTA (64)
constexpr int TK_RPL = 4;                        // database rows per lane and tile
constexpr int TK_ROWS = 32 * TK_RPL;             // database rows per tile (128)
constexpr int TK_MAX_SPLITS = 32;

#if defined(__CUDACC__)

// ---- embedding statistics ---------------------------------------------------
// rtab (ragged batches): clip i is rtab[i].n_frames rows from row rtab[i].first_frame; the same summation order
__global__ void __launch_bounds__(128) embed_stats_kernel(const float *feats, int64_t n_frames, int n_coef,
                                                         float *out, const dspx_ragged_clip *rtab = nullptr)
{
    extern __shared__ double es_sm[];                  // [groups][n_coef] partials, then [n_coef] means
    const int64_t clip = blockIdx.x;
    const float *f = feats + (size_t)(rtab ? rtab[clip].first_frame : clip * n_frames) * n_coef;
    if (rtab) n_frames = rtab[clip].n_frames;
    const int cw = n_coef < 128 ? n_coef : 128;        // coefficient lanes per pass
    const int groups = 128 / cw;
    const int tid = threadIdx.x;
    const int ty = tid / cw, tx = tid - ty * cw;
    double *mean = es_sm + (size_t)groups * n_coef;
    for (int pass = 0; pass < 2; pass++) {
        for (int c0 = 0; c0 < n_coef; c0 += cw) {
            const int c = c0 + tx;
            double acc = 0.0;
            if (ty < groups && c < n_coef) {
                const double mu = pass ? mean[c] : 0.0;
                for (int64_t t = ty; t < n_frames; t += groups) {
                    const double v = (double)f[(size_t)t * n_coef + c] - mu;
                    acc += pass ? v * v : v;
                }
                es_sm[(size_t)ty * n_coef + c] = acc;
            }
        }
        __syncthreads();
        for (int c = tid; c < n_coef; c += 128) {
            double s = 0.0;
            for (int g = 0; g < groups; g++) s += es_sm[(size_t)g * n_coef + c];
            s /= (double)n_frames;
            if (pass == 0) mean[c] = s;
            else {
                out[(size_t)clip * 2 * n_coef + c] = (float)mean[c];
                out[(size_t)clip * 2 * n_coef + n_coef + c] = (float)sqrt(s);
            }
        }
        __syncthreads();
    }
}

// ---- CMVN: cepstral mean / variance normalisation over the frames of each clip ----------------------
// BASELINE.json north_star names "a log/CMVN epilogue"; the reference has none (src/dsp/mfcc.py:102-109 stop
// at log and DCT), so it is an option that defaults to off.  y[t,c] = (x[t,c] - mean_t x[.,c]) / (std_t x[.,c] + eps),
// population std, statistics in float64 exactly like embed_stats_kernel (same summation order), in place.
// One CTA per clip: two passes for the statistics, a third applies them (22 KB per clip: L2-resident).
__global__ void __launch_bounds__(128) cmvn_kernel(float *feats, int64_t n_frames, int n_coef, double eps)
{
    extern __shared__ double es_sm[];                  // [groups][n_coef] partials, [n_coef] means, [n_coef] 1/(std+eps)
    const int64_t clip = blockIdx.x;
    float *f = feats + (size_t)clip * n_frames * n_coef;
    const int cw = n_coef < 128 ? n_coef : 128;
    const int groups = 128 / cw;
    const int tid = threadIdx.x;
    const int ty = tid / cw, tx = tid - ty * cw;
    double *mean = es_sm + (size_t)groups * n_coef;
    double *rstd = mean + n_coef;
    for (int pass = 0; pass < 2; pass++) {
        for (int c0 = 0; c0 < n_coef; c0 += cw) {
            const int c = c0 + tx;
            double acc = 0.0;
            if (ty < groups && c < n_coef) {
                const double mu = pass ? mean[c] : 0.0;
                for (int64_t t = ty; t < n_frames; t += groups) {
                    const double v = (double)f[(size_t)t * n_coef + c] - mu;
                    acc += pass ? v * v : v;
                }
                es_sm[(size_t)ty * n_coef + c] = acc;
            }
        }
        __syncthreads();
        for (int c = tid; c < n_coef; c += 128) {
            double s = 0.0;
            for (int g = 0; g < groups; g++) s += es_sm[(size_t)g * n_coef + c];
            s /= (double)n_frames;
            if (pass == 0) mean[c] = s;
            else rstd[c] = 1.0 / (sqrt(s) + eps);
        }
        __syncthreads();
    }
    const int64_t total = n_frames * n_coef;
    for (int64_t i = tid; i < total; i += 128) {
        const int c = (int)(i % n_coef);
        f[i] = (float)(((double)f[i] - mean[c]) * rstd[c]);
    }
}

// ---- row normalisation to float64 ---------------------------------------------
template <typename T>
__global__ void normalize_rows_kernel(const T *x, int64_t n, int dim, double *out)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const T *row = x + (size_t)r * dim;
    double s = 0.0;
    for (int c = 0; c < dim; c++) {
        const double v = (double)row[c];
        s = fma(v, v, s);
    }
    const double inv = sqrt(s) + 1e-10;
    for (int c = 0; c < dim; c++) out[(size_t)r * dim + c] = (double)row[c] / inv;
}

// ---- top-k ---------------------------------------------------------------------
struct TopkParams {
    const double *qn;       // [nq, dim] normalised
    const double *dbn;      // [ndb, dim] normalised
    int64_t nq, ndb;
    int dim, k;
    int n_splits;           // database ranges handled by gridDim.y
    int64_t rows_per_split; // multiple of TK_ROWS
    int32_t *idx_out;       // n_splits == 1: [nq, k]; else partial [nq, n_splits, k]
    double *score_out;      // same shape (may be null only when n_splits == 1)
};

// Insert (cs, ci) into the sorted list of one query (descending score; equal scores keep
// arrival order, and rows arrive in ascending index).  Whole warp participates.
__device__ __forceinline__ void topk_warp_insert(double *ls, int32_t *li, int k, int &cnt, double cs, int32_t ci,
                                                 int lane)
{
    int p = 0;
    for (int base = 0; base < cnt; base += 32) {
        const int e = base + lane;
        const bool ge = (e < cnt) && (ls[e] >= cs);
        p += __popc(__ballot_sync(0xffffffffu, ge));
    }
    const int last = cnt < k ? cnt : k - 1;          // entries [p, last) move up by one
    if (p > last) return;                            // full list and not better than the tail
    for (int base = ((last - 1) >= 0 ? (last - 1) / 32 : 0) * 32; base >= 0 && base + 32 > p; base -= 32) {
        const int e = base + lane;
        const bool mv = (e >= p) && (e < last);
        double vs = 0.0;
        int32_t vi = 0;
        if (mv) { vs = ls[e]; vi = li[e]; }
        __syncwarp();
        if (mv) { ls[e + 1] = vs; li[e + 1] = vi; }
        __syncwarp();
    }
    if (lane == 0) { ls[p] = cs; li[p] = ci; }
    if (cnt < k) cnt++;
    __syncwarp();
}

// Slow path of the selection, kept out of line (the fast path is one vote per query and tile):
// offer the four scores this lane holds for one query, rows tile + 32 r + lane, in ascending row order.
struct TopkState {
    double thr;
    int cnt;
};

__device__ __noinline__ TopkState topk_offer(double s0, double s1, double s2, double s3, int64_t tile, int64_t r_end,
                                             double *ls, int32_t *li, int k, int cnt, double thr, int lane)
{
#pragma unroll 1
    for (int r = 0; r < TK_RPL; r++) {
        const double s = r == 0 ? s0 : (r == 1 ? s1 : (r == 2 ? s2 : s3));
        const int64_t gr = tile + 32 * r + lane;
        const bool cand = (gr < r_end) && (cnt < k || s > thr);
        unsigned mask = __ballot_sync(0xffffffffu, cand);
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            const double cs = __shfl_sync(0xffffffffu, s, src);
            if (cnt == k && !(cs > thr)) continue;
            topk_warp_insert(ls, li, k, cnt, cs, (int32_t)(tile + 32 * r + src), lane);
            if (cnt == k) thr = ls[k - 1];
        }
    }
    TopkState out;
    out.thr = thr;
    out.cnt = cnt;
    return out;
}

// asynchronous global->shared copies; src_bytes = 0 zero-fills (rows / columns past the end)
__device__ __forceinline__ void tk_cp_async16(double *dst, const double *src, bool valid)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    const int n = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(n));
}
// asynchronous 8-byte global->shared copy; src_bytes = 0 zero-fills (rows / columns past the end)
__device__ __forceinline__ void tk_cp_async8(double *dst, const double *src, bool valid)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    const int n = valid ? 8 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(src), "r"(n));
}
__device__ __forceinline__ void tk_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void tk_cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// CW = columns of the dimension chunk kept in shared memory (compile-time, even): 26 when the
// whole MFCC embedding fits (2 x 13), 32 otherwise (last chunk zero-padded: fma(0, 0, acc) == acc).
// A "stage" is one (database tile, dimension chunk) pair; stages are double-buffered with cp.async
// so the next tile streams in while the current one is scored.
template <int CW>
__global__ void __launch_bounds__(TK_WARPS * 32, 2) cosine_topk_kernel(const TopkParams p)
{
    constexpr int DS = 34;                                             // even row stride (doubles): 16-byte aligned pairs,
                                                                       // 272 B rows -> conflict-free 128-bit loads
    extern __shared__ __align__(16) unsigned char tk_raw[];
    const int n_chunks = (p.dim + CW - 1) / CW;
    const int q_bufs = n_chunks > 1 ? 2 : 1;
    double *s_db = reinterpret_cast<double *>(tk_raw);                 // [2][TK_ROWS][DS]
    double *s_q = s_db + 2 * TK_ROWS * DS;                             // [q_bufs][TK_QPC][DS]
    double *s_ls = s_q + q_bufs * TK_QPC * DS;                         // [TK_QPC][k]
    int32_t *s_li = reinterpret_cast<int32_t *>(s_ls + (size_t)TK_QPC * p.k);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t q0 = (int64_t)blockIdx.x * TK_QPC;
    const int split = blockIdx.y;
    const int64_t r_begin = (int64_t)split * p.rows_per_split;
    int64_t r_end = r_begin + p.rows_per_split;
    if (r_end > p.ndb) r_end = p.ndb;
    const int64_t n_tiles = (r_end - r_begin + TK_ROWS - 1) / TK_ROWS;
    const int64_t n_stages = n_tiles * n_chunks;
    const bool vec16 = (p.dim & 1) == 0 && ((reinterpret_cast<uintptr_t>(p.dbn) | reinterpret_cast<uintptr_t>(p.qn)) & 15) == 0;

    auto issue = [&](int64_t stage) {
        const int64_t tile = r_begin + (stage / n_chunks) * TK_ROWS;
        const int ch = (int)(stage % n_chunks), c0 = ch * CW, buf = (int)(stage & 1);
        double *db = s_db + buf * TK_ROWS * DS;
        double *qb = s_q + (n_chunks > 1 ? buf : 0) * TK_QPC * DS;
        const bool load_q = n_chunks > 1 || stage == 0;
        if (vec16) {                                   // even dim: every (row, even column) is 16-byte aligned
            constexpr int CP = CW / 2;
            for (int e = tid; e < TK_ROWS * CP; e += TK_WARPS * 32) {
                const int row = e / CP, c = 2 * (e - row * CP);
                const int64_t gr = tile + row;
                const bool ok = gr < r_end && c0 + c < p.dim;
                tk_cp_async16(db + row * DS + c, p.dbn + (ok ? (size_t)gr * p.dim + c0 + c : 0), ok);
            }
            if (load_q)
                for (int e = tid; e < TK_QPC * CP; e += TK_WARPS * 32) {
                    const int row = e / CP, c = 2 * (e - row * CP);
                    const int64_t gq = q0 + row;
                    const bool ok = gq < p.nq && c0 + c < p.dim;
                    tk_cp_async16(qb + row * DS + c, p.qn + (ok ? (size_t)gq * p.dim + c0 + c : 0), ok);
                }
        } else {
            for (int e = tid; e < TK_ROWS * CW; e += TK_WARPS * 32) {
                const int row = e / CW, c = e - row * CW;
                const int64_t gr = tile + row;
                const bool ok = gr < r_end && c0 + c < p.dim;
                tk_cp_async8(db + row * DS + c, p.dbn + (ok ? (size_t)gr * p.dim + c0 + c : 0), ok);
            }
            if (load_q)
                for (int e = tid; e < TK_QPC * CW; e += TK_WARPS * 32) {
                    const int row = e / CW, c = e - row * CW;
                    const int64_t gq = q0 + row;
                    const bool ok = gq < p.nq && c0 + c < p.dim;
                    tk_cp_async8(qb + row * DS + c, p.qn + (ok ? (size_t)gq * p.dim + c0 + c : 0), ok);
                }
        }
        tk_cp_commit();
    };

    int cnt[TK_QPW];
    double thr[TK_QPW];
#pragma unroll
    for (int qi = 0; qi < TK_QPW; qi++) { cnt[qi] = 0; thr[qi] = 0.0; }
    double acc[TK_QPW][TK_RPL];

    if (n_stages > 0) issue(0);
    for (int64_t stage = 0; stage < n_stages; stage++) {
        const int ch = (int)(stage % n_chunks), buf = (int)(stage & 1);
        const int64_t tile = r_begin + (stage / n_chunks) * TK_ROWS;
        if (stage + 1 < n_stages) { issue(stage + 1); tk_cp_wait<1>(); }
        else tk_cp_wait<0>();
        __syncthreads();                                               // this stage's bytes are visible to all
        if (ch == 0) {
#pragma unroll
            for (int qi = 0; qi < TK_QPW; qi++)
#pragma unroll
                for (int r = 0; r < TK_RPL; r++) acc[qi][r] = 0.0;
        }
        const double *db = s_db + buf * TK_ROWS * DS + lane * DS;
        const double *qrow = s_q + (n_chunks > 1 ? buf : 0) * TK_QPC * DS + (warp * TK_QPW) * DS;
#pragma unroll
        for (int cp = 0; cp < CW / 2; cp++) {
            double2 dv[TK_RPL];
#pragma unroll
            for (int r = 0; r < TK_RPL; r++) dv[r] = *reinterpret_cast<const double2 *>(db + 32 * r * DS + 2 * cp);
#pragma unroll
            for (int qi = 0; qi < TK_QPW; qi++) {
                const double2 qv = *reinterpret_cast<const double2 *>(qrow + qi * DS + 2 * cp);
#pragma unroll
                for (int r = 0; r < TK_RPL; r++) {
                    acc[qi][r] = fma(qv.x, dv[r].x, acc[qi][r]);
                    acc[qi][r] = fma(qv.y, dv[r].y, acc[qi][r]);
                }
            }
        }
        if (ch == n_chunks - 1) {
            // selection fast path: one vote per query and tile ("does any lane hold a score that beats the
            // current k-th?"); rows past r_end score 0 and are filtered out in topk_offer
#pragma unroll
            for (int qi = 0; qi < TK_QPW; qi++) {
                const int ql = warp * TK_QPW + qi;
                if (q0 + ql >= p.nq) continue;                          // warp-uniform
                const double mx = fmax(fmax(acc[qi][0], acc[qi][1]), fmax(acc[qi][2], acc[qi][3]));
                if (__any_sync(0xffffffffu, cnt[qi] < p.k || mx > thr[qi])) {
                    const TopkState st = topk_offer(acc[qi][0], acc[qi][1], acc[qi][2], acc[qi][3], tile, r_end,
                                                    s_ls + (size_t)ql * p.k, s_li + (size_t)ql * p.k, p.k, cnt[qi], thr[qi], lane);
                    cnt[qi] = st.cnt;
                    thr[qi] = st.thr;
                }
            }
        }
        __syncthreads();                                               // buffer `buf` may be refilled by stage + 2
    }

    // write this CTA's lists
    __syncwarp();
    for (int qi = 0; qi < TK_QPW; qi++) {
        const int ql = warp * TK_QPW + qi;
        const int64_t gq = q0 + ql;
        if (gq >= p.nq) continue;
        const double *ls = s_ls + (size_t)ql * p.k;
        const int32_t *li = s_li + (size_t)ql * p.k;
        const size_t o = ((size_t)gq * p.n_splits + split) * p.k;
        for (int e = lane; e < p.k; e += 32) {
            const bool have = e < cnt[qi];
            p.idx_out[o + e] = have ? li[e] : -1;
            if (p.score_out) p.score_out[o + e] = have ? ls[e] : -INFINITY;
        }
    }
}

inline size_t topk_smem_bytes(int dim, int k, int cw)
{
    const int n_chunks = (dim + cw - 1) / cw;
    return (size_t)(2 * TK_ROWS + (n_chunks > 1 ? 2 : 1) * TK_QPC) * 34 * 8 + (size_t)TK_QPC * k * 12;
}

// merge the per-split sorted lists of one query (one warp per query, one list per lane)
__global__ void __launch_bounds__(128) topk_merge_kernel(const int32_t *pidx, const double *pscore, int64_t nq,
                                                        int n_splits, int k, int32_t *idx_out, double *score_out)
{
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= nq) return;
    const size_t base = ((size_t)q * n_splits + lane) * k;
    int head = 0;
    for (int out = 0; out < k; out++) {
        double s = -INFINITY;
        int32_t id = 0x7fffffff;
        if (lane < n_splits && head < k && pidx[base + head] >= 0) { s = pscore[base + head]; id = pidx[base + head]; }
        double bs = s;
        int32_t bi = id;
        int bl = lane;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double os = __shfl_xor_sync(0xffffffffu, bs, off);
            const int32_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
            const int ol = __shfl_xor_sync(0xffffffffu, bl, off);
            if (os > bs || (os == bs && oi < bi)) { bs = os; bi = oi; bl = ol; }
        }
        if (lane == bl) head++;
        if (lane == 0) {
            idx_out[(size_t)q * k + out] = bi;
            if (score_out) score_out[(size_t)q * k + out] = bs;
        }
    }
}

// dense score matrix, same left-to-right fma chain as the top-k kernel
__global__ void __launch_bounds__(256) cosine_matrix_kernel(const double *qn, const double *dbn, int64_t nq, int64_t ndb,
                                                          int dim, double *sims)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t i = blockIdx.y;
    if (j >= ndb || i >= nq) return;
    const double *a = qn + (size_t)i * dim, *b = dbn + (size_t)j * dim;
    double acc = 0.0;
    for (int c = 0; c < dim; c++) acc = fma(a[c], b[c], acc);
    sims[(size_t)i * ndb + j] = acc;
}

// standalone DCT-II x2 (dct_type_2): one thread per output, float64 accumulation
__global__ void __launch_bounds__(256) dct2_kernel(const float *x, int64_t rows, int n, int n_mfcc, float *out)
{
    const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= rows * n_mfcc) return;
    const int64_t r = o / n_mfcc;
    const int k = (int)(o - r * n_mfcc);
    const float *row = x + (size_t)r * n;
    double acc = 0.0;
    for (int j = 0; j < n; j++) acc += (double)row[j] * cospi(((double)j + 0.5) * (double)k / (double)n);
    out[o] = (float)(2.0 * acc);
}

// hit@k: one thread per query, block-reduced, one atomic per block
__global__ void __launch_bounds__(256) hits_at_k_kernel(const int32_t *idx, int64_t nq, int k_stride, int k,
                                                       const int32_t *tdb, const int32_t *tq, unsigned long long *hits)
{
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int hit = 0;
    if (q < nq) {
        const int32_t want = tq[q];
        for (int r = 0; r < k && !hit; r++) {
            const int32_t j = idx[(size_t)q * k_stride + r];
            hit = (j >= 0) && (tdb[j] == want);
        }
    }
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    __shared__ int wsum[8];
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += wsum[w];
        if (s) atomicAdd(hits, (unsigned long long)s);
    }
}
#endif

}  // namespace dspx
