// retrieval_select.cuh -- which ranking kernel a dspx_cosine_topk call launches, with which grid, and the layout of its
// workspace.  Host code only, from the shape alone: dspx.cu launches what it says, and the test-only replay library
// (emu.cu) exposes it so that the selection and the workspace can be checked on machines without a GPU.
#pragma once

#include "retrieval.cuh"
#include "retrieval_f32.cuh"
#include "retrieval_tc.cuh"

namespace dspx {

// The three ranking kernels return the same lists: each scores every row it keeps exactly in float64.  The two filters
// first screen the database with a cheaper score (split fp16 on the tensor cores, packed FP32) against the running k-th
// score, minus a bound on that score's error.
enum TopkKernel { TOPK_TC, TOPK_F32, TOPK_F64 };

struct TopkLaunch {
    TopkKernel kernel;
    int cw;                     // template argument: 26 (MFCC embeddings, 2 x 13), else 0 (TOPK_TC) or 32
    dim3 grid;                  // (query tiles, database splits)
    int threads;
    size_t smem;                // dynamic shared memory
    int n_splits;
    int64_t rows_per_split;     // multiple of TK_ROWS
};

// float64 kernel: about two CTAs per SM, at least 4 tiles per split
static int topk_splits(int64_t nq, int64_t ndb, int sm_count)
{
    const int64_t qtiles = (nq + TK_QPC - 1) / TK_QPC;
    int64_t s = (2 * (int64_t)sm_count + qtiles - 1) / qtiles;
    const int64_t max_by_rows = (ndb + 4 * TK_ROWS - 1) / (4 * TK_ROWS);       // at least 4 tiles per split
    if (s > max_by_rows) s = max_by_rows;
    if (s > TK_MAX_SPLITS) s = TK_MAX_SPLITS;
    if (s < 1) s = 1;
    return (int)s;
}

// filter kernels, one CTA per SM: the split count whose grid fills whole waves (every extra split also restarts the
// running lists, which costs insertions -- the per-split penalty), at most 16, at least 8 tiles per split
static int64_t topk_wave_splits(int64_t qtiles, int64_t ndb, int sm_count)
{
    int64_t max_sp = (ndb + 8 * TK_ROWS - 1) / (8 * TK_ROWS);
    if (max_sp > 16) max_sp = 16;
    if (max_sp < 1) max_sp = 1;
    int64_t sp = 1;
    double best = 1e30;
    for (int64_t c = 1; c <= max_sp; c++) {
        const double waves = (double)((qtiles * c + sm_count - 1) / sm_count);
        const double cost = waves / (double)c * (1.0 + 0.02 * (double)c);
        if (cost < best - 1e-12) { best = cost; sp = c; }
    }
    return sp;
}

// The kernel of a call and its launch, from the shape alone:
//   dim <= 32 and k <= TC_MAX_K                                   tensor-core filter
//   dim <= 32 and the FP32 filter's lists fit in 200 KB of smem   FP32 filter (k <= 55 at dim 26, k <= 37 at dim 32)
//   otherwise                                                     float64 kernel
static TopkLaunch topk_select(int64_t nq, int64_t ndb, int dim, int k, int sm_count)
{
    TopkLaunch L{};
    const int cw = dim == 26 ? 26 : 32;
    int64_t qtiles;
    if (dim <= 32 && k <= TC_MAX_K) {
        L.kernel = TOPK_TC;
        L.cw = dim == 26 ? 26 : 0;
        L.threads = TC_THREADS;
        L.smem = topk_tc_smem_bytes(k);
        qtiles = (nq + TC_QT - 1) / TC_QT;
    } else if (dim <= 32 && topk_f32_smem_bytes(dim, k, cw) <= 200 * 1024) {
        L.kernel = TOPK_F32;
        L.cw = cw;
        L.threads = TKF_WARPS * 32;
        L.smem = topk_f32_smem_bytes(dim, k, cw);
        qtiles = (nq + TKF_QPC - 1) / TKF_QPC;
    } else {
        L.kernel = TOPK_F64;
        L.cw = cw;
        L.threads = TK_WARPS * 32;
        L.smem = topk_smem_bytes(dim, k, cw);
        qtiles = (nq + TK_QPC - 1) / TK_QPC;
    }
    const int64_t sp = L.kernel == TOPK_F64 ? topk_splits(nq, ndb, sm_count) : topk_wave_splits(qtiles, ndb, sm_count);
    int64_t rows = (ndb + sp - 1) / sp;
    rows = (rows + TK_ROWS - 1) / TK_ROWS * TK_ROWS;
    L.rows_per_split = rows;
    L.n_splits = (int)((ndb + rows - 1) / rows);
    L.grid = dim3((unsigned)qtiles, (unsigned)L.n_splits);
    return L;
}

struct TopkWs {
    double *qn, *dbn;                   // [nq, dim], [ndb, dim] normalised rows
    double *pscore;                     // per-split lists [nq, n_splits, k], n_splits <= TK_MAX_SPLITS
    int32_t *pidx;
    float *qf, *dbf;                    // operand images of the filter kernels: 32 floats per row covers both layouts (dim <= 32 there)
    size_t qf_bytes, dbf_bytes;
    unsigned long long *shared_thr;     // [nq] thresholds shared between splits
    int *split_done;                    // per (query tile, split): lists written
};

// One layout of the ranking workspace for the size query and the launches.  Returns its size; with base, also the pointers.
static size_t topk_ws_carve(int64_t nq, int64_t ndb, int dim, int k, char *base, TopkWs *ws)
{
    TopkWs w;
    w.qf_bytes = (size_t)((nq + TC_QT - 1) / TC_QT) * TC_QT * TC_KPAD * 4;
    w.dbf_bytes = (size_t)((ndb + TK_ROWS - 1) / TK_ROWS) * TK_ROWS * TC_KPAD * 4;
    size_t off = 0;
    auto take = [&](size_t bytes) -> char * {
        char *p = base ? base + off : nullptr;
        off += align256(bytes);
        return p;
    };
    w.qn = reinterpret_cast<double *>(take((size_t)nq * dim * 8));
    w.dbn = reinterpret_cast<double *>(take((size_t)ndb * dim * 8));
    w.pscore = reinterpret_cast<double *>(take((size_t)nq * TK_MAX_SPLITS * k * 8));
    w.pidx = reinterpret_cast<int32_t *>(take((size_t)nq * TK_MAX_SPLITS * k * 4));
    w.qf = reinterpret_cast<float *>(take(w.qf_bytes));
    w.dbf = reinterpret_cast<float *>(take(w.dbf_bytes));
    w.shared_thr = reinterpret_cast<unsigned long long *>(take((size_t)nq * 8));
    w.split_done = reinterpret_cast<int *>(take((size_t)((nq + TC_QT - 1) / TC_QT) * TK_MAX_SPLITS * 4));
    if (ws) *ws = w;
    return off + 1024;
}

}  // namespace dspx
