// retrieval_tc.cuh -- exact cosine top-k with a tensor-core (tcgen05, TF32) pre-filter.
//
// Same contract as cosine_topk_kernel (retrieval.cuh): float64 scores accumulated left to right with fused
// multiply-adds, descending order, ties to the lower database index -- the result is bit-identical.  The
// similarity matrix q . db^T is a GEMM, so the scores that only have to be *compared* against each query's
// current k-th score are produced by the 5th-generation tensor cores; the few pairs that pass are re-scored
// exactly in float64.  Replaces the argsort over the dense matrix of src/retrieval/retrieval.py:25-49.
//
// Arithmetic.  A single reduced-precision pass (TF32: 10 mantissa bits, ~1e-3 on a unit-vector dot product) would pass far
// too many pairs for tightly clustered embeddings.  Each float32 value v is therefore split into hi = v with the low 13
// mantissa bits cleared (11 significant bits) and lo = v - hi (< 2^-10 |v|), and the filter accumulates
// A_lo B_hi + A_hi B_lo + A_hi B_hi into one float32 TMEM accumulator.  Round 1 ran these as three TF32 passes (24 MMAs of
// K = 8 per 256 x 128 tile, 1536 tensor cycles).  hi has 11 significant bits: it is exact in fp16 as well, and so are all
// products (22 bits into a float32 accumulator), so since the last session of round 2 ALL THREE terms are kind::f16 MMAs
// (K = 16 per instruction: 12 MMAs, 768 cycles per tile) on ONE operand format for queries and database alike: a 128-byte row
// of 64 halves [S hi(0..31) | S lo(0..31)] with S = 2^11 (a power of two: exact).  S lifts the operands into fp16's normal
// range (S hi <= 2048, S lo < 2; a value only turns subnormal below 2^-25 of the norm, where even flushing it to zero costs
// < 1.5e-7 in total) and the accumulator holds S^2 * score; the scan compares against S^2 * threshold.  The three terms are
// K slices of the same two rows:  A[32..63] x B[0..31]  (lo hi),  A[0..31] x B[32..63]  (hi lo),  A[0..31] x B[0..31]  (hi hi).
// Error budget for unit vectors (sum |q_i d_i| <= 1), worst case:
//   inputs rounded to float32 (both sides)                                   2 * 2^-24          = 1.2e-7
//   A_lo B_lo dropped                                                        2^-10 * 2^-10      = 9.5e-7
//   lo rounded to 11 bits by fp16 (round to nearest: <= 2^-11 |lo|), 2 terms 2 * 2^-21          = 9.5e-7
//   float32 accumulation in the tensor core, allowing every one of the 16 + 1 addends of the two hi x hi MMAs to lose
//   2^-25 of the row's largest magnitude and a truncation of the accumulator per MMA          ~ 1.2e-6
// = 3.2e-6.  Measured against float64 (benchmarks/micro/umma_f16x.cu, profiles/r02_micro_umma_f16x.txt): <= 6.5e-7 on
// random, clustered and wide-dynamic-range unit vectors and with adversarial mantissas (all 13 low bits set, all residuals
// of one sign; the three TF32 passes of round 1: 1.2e-6).  TC_EPS = 6e-6 (round 1: 8e-6 over a 4.5e-6 bound), so every
// pair with s64 >= thr64 has s_tc > thr32 = float(thr64 - eps) and is re-scored.  eps only costs
// extra re-scores: on tightly clustered embeddings (every cosine near 1, thousands of rows within eps of the k-th score) the
// kernel degrades towards the all-float64 kernel's time instead of failing.
//
// The operand rows are written ONCE, by the normalisation kernel, already in the 128-byte-swizzled K-major tile image the
// tensor core reads (16 KB per 128 rows), so a database tile reaches shared memory as one bulk copy (cp.async.bulk, the TMA
// engine's 1-D form, completion on an mbarrier) issued by a single thread.  Until then two producer warps re-split every tile
// for every query tile with ordinary loads and stores (~1100 cycles per tile, as long as the MMAs themselves) and the epilogue
// warps that shared their schedulers were the laggards the issue thread waited for (profiles/r02_topk_tc_mixed_ab.txt).
//
// Structure of a CTA (352 threads, one per SM), 256 queries x one database split:
//   warps 0-7  epilogue: thread = one query.  All 128 scores of its accumulator row go to registers (four
//              tcgen05.ld.32x32b.x32 in flight at once), the TMEM buffer is handed back to the tensor core at once, and
//              only then are the scores compared with the thread's float threshold (3-input max tree per 32 columns, ONE vote
//              per tile, bit masks only for blocks in which some lane of the warp has a hit).  Rows that pass
//              wait in a per-query ring; the WARP re-scores them together in float64 (drain: one work list over the 32
//              rings, lane i scores item i, then every lane inserts its own rows in order into its unordered k-entry
//              list in shared memory: overwrite the worst entry, rescan for the new worst; rows arrive in index order,
//              so "strictly better than the current worst" keeps ties at the lower index; ordered once at the end).
//              Re-scoring happens when a ring is full, when the warp holds 64 pending rows, or -- preferably -- while
//              the warp would otherwise wait more than TC_IDLE_CYCLES for the next tile, i.e. while another warp's
//              re-scoring holds the pipeline up (an issue thread needs all four warps of its half to release a buffer).
//   warp 8     one lane: bulk copies of the query tiles (once) and of the database tiles into a 4-stage ring; mbarrier
//              expect_tx / complete_tx hand-off to the issue thread.
//   warps 9-10 one lane each: issues the 6 tcgen05.mma kind::f16 (M 128, N 128, K 16) of ITS query half (warps 0-3 / 4-7) per
//              tile into that half's double-buffered TMEM accumulator (2 x 2 x 128 columns) and commits to the mbarriers of
//              the smem stage (count 2) and of the buffer.  The halves are independent pipelines over the shared database
//              ring: an issue thread waits for the slowest of four warps, not of eight.
// Measured structure (profiles/r02_topk_tc_takeover.txt, r02_topk_tc_pipeline.md): the tensor core needs 768 cycles per tile
// (1536 with the three TF32 passes of round 1), the TMEM read-out 400-450 (320 B/clk per SM, overlapping with the MMAs:
// benchmarks/micro/umma_ld_overlap.cu); a tile without candidates takes a warp ~1470 cycles (two warps per scheduler:
// latency-bound), and a CTA of the first wave, whose lists start empty, ~3500: every sparse re-scoring pass of one warp
// stalls the other three of its half after two tiles.  The number of candidates is fixed by the scan order
// (k (1 + ln(n / k)) per query), so seeding thresholds from a sample or giving the first wave short splits only moves that
// work around (profiles/r02_topk_tc_seed_join_experiments.txt); what later CTAs gain comes from taking finished lists over.
#pragma once

#include <cuda_fp16.h>

#include "retrieval.cuh"

namespace dspx {

#if defined(__CUDACC__)

constexpr int TC_QT = 256;            // queries per CTA: two 128-row A tiles
constexpr int TC_ROWS = 128;          // database rows per tile (UMMA N)
constexpr int TC_STAGES = 4;          // database tiles in flight (16 KB each)
constexpr int TC_EPI_THREADS = 256;
constexpr int TC_THREADS = TC_EPI_THREADS + 32 + 64;      // + bulk-copy warp + two tensor-core issue warps (one per query half)
constexpr int TC_KPAD = 32;           // padded embedding dimension: 32 hi + 32 lo halves = one 128-byte swizzle row
constexpr int TC_TILE_BYTES = 128 * 128;                  // operand image of 128 rows
constexpr double TC_EPS = 6e-6;
constexpr float TC_S = 2048.f;                            // operand scale S = 2^11
constexpr float TC_SCALE = TC_S * TC_S;                   // the accumulator holds S^2 * score
// pending candidates per query: ring size; the warp re-scores when one ring holds TC_FIFO_TRIGGER rows or all 32 rings
// together hold TC_WARP_TRIGGER (one full scoring pass)
constexpr int TC_FIFO = 8, TC_FIFO_TRIGGER = 8, TC_WARP_TRIGGER = 64;
constexpr long long TC_IDLE_CYCLES = 3500;   // wait on acc_full after which an epilogue warp uses the stall to re-score
constexpr int TC_MAX_K = 24;          // the per-thread lists ([k][256] doubles + ints) share smem with the tiles

// Rows scaled by 1 / (||row|| + 1e-10) in float64 (src/retrieval/retrieval.py:46-48: the division, not a multiply by
// the reciprocal; the norm is the same left-to-right fma chain as normalize_rows_kernel, so out64 is bit-identical
// to it) plus the fp16 operand image the tensor-core filter reads: per 128 rows a 16 KB tile, row r at r * 128 bytes, its
// eight 16-byte chunks (chunks 0-3: S hi of columns 0-31, chunks 4-7: S lo; zero beyond dim and beyond n) at position
// chunk ^ (r & 7) -- the 128-byte swizzle of a K-major operand, so the kernel's bulk copy is a plain memcpy of the tile.
// A CTA owns NR_ROWS consecutive rows: they are one contiguous span of the input and of both outputs, so every global
// access is coalesced (the round-1 kernel had one thread walk one row: 26 strided stores per thread, 9x the HBM time of
// the copy).
constexpr int NR_ROWS = 64;

template <typename T>
__global__ void __launch_bounds__(128) normalize_rows_split16_kernel(const T *x, int64_t n, int64_t n_pad, int dim,
                                                                    double *out64, unsigned char *out16)
{
    __shared__ T s_in[NR_ROWS * TC_KPAD];
    __shared__ float s_f32[NR_ROWS * TC_KPAD];
    __shared__ double s_inv[NR_ROWS];
    const int tid = threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * NR_ROWS;
    const int64_t rows = (n - r0) < NR_ROWS ? ((n - r0) > 0 ? (n - r0) : 0) : NR_ROWS;      // real rows of this CTA
    const int64_t elems = rows * dim;
    const T *src = x + (size_t)r0 * dim;
    for (int64_t e = tid; e < elems; e += 128) s_in[e] = src[e];
    for (int e = tid; e < NR_ROWS * TC_KPAD; e += 128) s_f32[e] = 0.f;                     // padding columns and rows
    __syncthreads();
    if (tid < rows) {
        double s = 0.0;
        for (int c = 0; c < dim; c++) {
            const double v = (double)s_in[tid * dim + c];
            s = fma(v, v, s);
        }
        s_inv[tid] = sqrt(s) + 1e-10;
    }
    __syncthreads();
    double *dst = out64 + (size_t)r0 * dim;
    for (int64_t e = tid; e < elems; e += 128) {
        const int r = (int)(e / dim), c = (int)(e - (int64_t)r * dim);
        const double v = (double)s_in[e] / s_inv[r];
        dst[e] = v;
        s_f32[r * TC_KPAD + c] = (float)v;
    }
    __syncthreads();
    const int64_t pad_rows = (n_pad - r0) < NR_ROWS ? (n_pad - r0) : NR_ROWS;
    // r0 is a multiple of 64: the CTA's rows lie inside one 128-row tile
    unsigned char *tile = out16 + (size_t)(r0 >> 7) * TC_TILE_BYTES;
    for (int e = tid; e < pad_rows * 8; e += 128) {
        const int r = e >> 3, chunk = e & 7, rt = (int)((r0 + r) & 127);
        const float *v = s_f32 + r * TC_KPAD + (chunk & 3) * 8;
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const float a = v[2 * j], b = v[2 * j + 1];
            const float ah = __uint_as_float(__float_as_uint(a) & 0xffffe000u), bh = __uint_as_float(__float_as_uint(b) & 0xffffe000u);
            const __half2 h = chunk < 4 ? __floats2half2_rn(ah * TC_S, bh * TC_S)                 // exact: 11 significant bits
                                        : __floats2half2_rn((a - ah) * TC_S, (b - bh) * TC_S);   // residual, rounded to 11 bits
            w[j] = *reinterpret_cast<const uint32_t *>(&h);
        }
        *reinterpret_cast<uint4 *>(tile + rt * 128 + ((chunk ^ (rt & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

#ifdef DSPX_TC_PROFILE
// per-role cycle counters of CTA (0, 0): [0] mma wait acc_empty [1] mma wait full_b [2] mma issue [3] producer wait
// [4] producer store [5] epilogue wait acc_full [6] epilogue masks [7] epilogue enqueue+drain [8] tiles [9] total
__device__ long long tc_prof[16];
// event trace of CTA (0, 0), tiles 64..95: [tile - 64][0] mma: acc_empty seen [1] mma: issue done [2..9] epilogue warp w: acc_full seen
// [10..17] epilogue warp w: buffer released
__device__ long long tc_trace[32][18];
#define TC_TRACE(tile, slot) do { if (blockIdx.x == 0 && blockIdx.y == 0 && (tile) >= 64 && (tile) < 96) tc_trace[(tile) - 64][slot] = clock64(); } while (0)
#define TC_PROF_T0() long long _pt = clock64()
#define TC_PROF_ADD(i) do { const long long _n = clock64(); if (blockIdx.x == 0 && blockIdx.y == 0) tc_prof_local[i] += _n - _pt; _pt = _n; } while (0)
#else
#define TC_PROF_T0()
#define TC_PROF_ADD(i)
#define TC_TRACE(tile, slot)
#endif

struct TopkTcParams {
    TopkParams base;
    const unsigned char *qx;    // fp16 operand tiles of the queries: [ceil(nq / 256) * 2][16 KB] (normalize_rows_split16_kernel)
    const unsigned char *dbx;   // fp16 operand tiles of the database: [ceil(ndb / 128)][16 KB]
    unsigned long long *shared_thr;   // [nq] order-encoded k-th scores shared by the splits of a query (null: one split)
    int *done;                        // [query tiles][n_splits] set once a CTA's lists are in idx_out / score_out (null: one split)
};

// order-preserving double <-> uint64 (0 is below every double): lets atomicMax maintain a shared threshold
__device__ __forceinline__ unsigned long long tc_enc(double d)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double tc_dec(unsigned long long u)
{
    return __longlong_as_double((long long)((u >> 63) ? (u & 0x7fffffffffffffffull) : ~u));
}

__device__ __forceinline__ uint32_t tc_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void tc_mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t *bar)
{
    asm volatile("{ .reg .b64 st; mbarrier.arrive.shared::cta.b64 st, [%0]; }" ::"r"(tc_smem_u32(bar)) : "memory");
}
// bounded wait: a protocol error traps (launch failure) instead of hanging the GPU
__device__ __forceinline__ void tc_mbar_wait(uint64_t *bar, uint32_t parity)
{
    for (uint32_t spin = 0;; spin++) {
        uint32_t ok;
        // the suspend-time hint lets the hardware park the thread instead of re-issuing the wait: the two single-thread
        // roles share their schedulers with epilogue warps 0/4 and 1/5, which the issue thread ends up waiting for
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(tc_smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
        if (ok) return;
        if (spin > (1u << 28)) __trap();
    }
}

// K-major operand tile under SWIZZLE_128B: rows of 128 bytes, 8-row groups 1024 bytes apart
__device__ __forceinline__ uint64_t tc_desc(const void *tile)
{
    return (uint64_t)((tc_smem_u32(tile) >> 4) & 0x3fff) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}

__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p; }"
                 ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}

// mbarrier transaction count + the TMA engine's 1-D bulk copy global -> shared (completes on the barrier)
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_bulk_load(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(tc_smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(tc_smem_u32(bar)) : "memory");
}

// 32 accumulator columns of this thread's TMEM lane -> bit j set when column j passes the threshold
__device__ __forceinline__ uint32_t tc_ld_mask(uint32_t taddr, float thr32)
{
    uint32_t v[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) m |= (__uint_as_float(v[j]) > thr32) ? (1u << j) : 0u;
    return m;
}

// Issue / wait split of the same load: the wait names the destination registers as in/out operands so that no use of
// them can be scheduled above it.  With two register buffers the load of block i + 1 is in flight while block i is scanned.
__device__ __forceinline__ void tc_ld32_issue(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                   "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                   "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait(uint32_t (&v)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :: "memory");
}
// Almost every block of 32 columns is entirely below the threshold: a max tree (3-input FMNMX, log depth) decides that in
// 16 instructions per block, ONE vote covers the four blocks of a tile, and bit masks (bit j set when column j passes) are
// only built for the blocks in which some lane of the warp has a hit.
__device__ __forceinline__ float tc_top32(const uint32_t (&w)[32])
{
    float mx[11];
#pragma unroll
    for (int j = 0; j < 10; j++)
        mx[j] = fmaxf(fmaxf(__uint_as_float(w[3 * j]), __uint_as_float(w[3 * j + 1])), __uint_as_float(w[3 * j + 2]));
    mx[10] = fmaxf(__uint_as_float(w[30]), __uint_as_float(w[31]));
    const float t0 = fmaxf(fmaxf(mx[0], mx[1]), mx[2]), t1 = fmaxf(fmaxf(mx[3], mx[4]), mx[5]);
    const float t2 = fmaxf(fmaxf(mx[6], mx[7]), mx[8]), t3 = fmaxf(mx[9], mx[10]);
    return fmaxf(fmaxf(t0, t1), fmaxf(t2, t3));
}
// Bit j set when column j passes.  thr - v is negative exactly when v > thr (equal gives +0; an empty list has
// thr = -inf: everything passes; an inactive lane +inf: nothing does), so the mask is the sign bits: one FADD (FMA pipe)
// and one funnel shift per column, in four independent chains -- the compare / select / add form cost 2.5 ALU-pipe
// instructions per column, and the ALU pipe (max tree, masks, ring bookkeeping) is this kernel's busiest.
__device__ __forceinline__ uint32_t tc_bits32(const uint32_t (&w)[32], float thr32)
{
    uint32_t part[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int c = 0; c < 4; c++)
#pragma unroll
        for (int j = 7; j >= 0; j--)                               // highest column first: column 8 c + j ends up at bit j
            part[c] = __funnelshift_l(__float_as_uint(thr32 - __uint_as_float(w[8 * c + j])), part[c], 1);
    return (part[0] | (part[1] << 8)) | ((part[2] << 16) | (part[3] << 24));
}

inline size_t topk_tc_smem_bytes(int k)
{
    return (size_t)(2 + TC_STAGES) * TC_TILE_BYTES + (size_t)TC_QT * k * 12 + (size_t)TC_FIFO * TC_QT * 12 + 256;    // + 17 mbarriers, TMEM slot
}

// DIM > 0: the embedding dimension is a compile-time constant (all loads of the exact dot product in flight at
// once); DIM == 0: any dim <= 32.
template <int DIM>
__global__ void __launch_bounds__(TC_THREADS, 1) cosine_topk_tc_kernel(const TopkTcParams pp)
{
    const TopkParams &p = pp.base;
    extern __shared__ __align__(1024) unsigned char tc_raw[];     // the 128-byte swizzle pattern repeats every 1024 bytes
    if (tc_smem_u32(tc_raw) & 1023u) __trap();
    unsigned char *a_x = tc_raw;                                  // [2][16 KB]: query rows 0-127, 128-255
    unsigned char *b_x = a_x + 2 * TC_TILE_BYTES;                 // [TC_STAGES][16 KB]
    double *s_ls = reinterpret_cast<double *>(b_x + TC_STAGES * TC_TILE_BYTES);      // [k][256]
    double *s_sc = s_ls + (size_t)p.k * TC_QT;                                       // [TC_FIFO][256] scores of the pending rows
    int32_t *s_li = reinterpret_cast<int32_t *>(s_sc + (size_t)TC_FIFO * TC_QT);     // [k][256]
    int32_t *s_fifo = s_li + (size_t)p.k * TC_QT;                                    // [TC_FIFO][256] pending candidate rows
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_fifo + TC_FIFO * TC_QT);         // 8-byte aligned
    // acc_full / acc_empty: [query half][buffer]
    uint64_t *full_b = bars, *empty_b = bars + TC_STAGES, *acc_full = bars + 2 * TC_STAGES, *acc_empty = acc_full + 4;
    uint64_t *a_full = acc_empty + 4;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(a_full + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int dim = DIM > 0 ? DIM : p.dim;
    const int64_t q0 = (int64_t)blockIdx.x * TC_QT;
    const int split = blockIdx.y;
    const int64_t r_begin = (int64_t)split * p.rows_per_split;    // multiple of TC_ROWS
    int64_t r_end = r_begin + p.rows_per_split;
    if (r_end > p.ndb) r_end = p.ndb;
    const int64_t n_tiles = (r_end - r_begin + TC_ROWS - 1) / TC_ROWS;

    // ---- set-up: barriers, TMEM (the operand tiles arrive by bulk copy) ---------------------------
    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; s++) { tc_mbar_init(&full_b[s], 1); tc_mbar_init(&empty_b[s], 2); }    // both halves read a stage
        for (int b = 0; b < 4; b++) { tc_mbar_init(&acc_full[b], 1); tc_mbar_init(&acc_empty[b], TC_EPI_THREADS / 64); }
        tc_mbar_init(a_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    if (warp == TC_THREADS / 32 - 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tc_smem_u32(tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = *tmem_slot;

    if (tid < TC_EPI_THREADS) {
        // ===== epilogue: one query per thread =====
        const int ql = tid;                                        // = (warp >> 2) * 128 + (warp & 3) * 32 + lane
        const int64_t gq = q0 + ql;
        const bool active = gq < p.nq;
        double *ls = s_ls + ql;                                    // element e at ls[e * TC_QT]
        int32_t *li = s_li + ql;
        const int k = p.k;
        int cnt = 0;
        double thr = 0.0;                                          // k-th score of this thread's list once it is full
        // Splits of one query share the best k-th score any of them has reached (gthr): a row scoring below it
        // can never enter the merged top-k, so it is neither re-scored nor inserted.  This only prunes work --
        // every member of the final top-k scores >= gthr at all times and is among the k best of its own split.
        unsigned long long *gslot = (pp.shared_thr && active) ? pp.shared_thr + gq : nullptr;
        double gthr = -INFINITY;
        unsigned long long genc = 0;
        const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * TC_ROWS);
        // The two query halves (warps 0-3, 4-7) are separate pipelines: own accumulator barriers, own issue thread.  The
        // issue thread waits for the slowest warp of ITS half only, so a warp that is re-scoring holds up three others
        // instead of seven; the halves may drift apart by the depth of the smem ring.
        uint64_t *my_full = acc_full + (warp >> 2) * 2, *my_empty = acc_empty + (warp >> 2) * 2;
        // Candidates wait in a small per-thread ring in shared memory and are re-scored in lock step, one per lane
        // and round: a round costs the same whether 1 or 32 lanes have work (it is bound by the latency of the
        // float64 row loads), so the ring is drained only when some lane has TC_FIFO_TRIGGER entries, which fills
        // the rounds.  Each lane sees its rows in increasing order.
        int f_head = 0, f_cnt = 0, wpos = 0;
        bool thr_dirty = false;                                    // the list's k-th score or fill count changed since thr32c was formed
        int32_t *fifo = s_fifo + ql;
        // One exactly scored row into the thread's list.  Rows reach a list in an order in which every entry already there
        // with the same score has a lower index (own rows: increasing index; rows taken over from finished splits: see below).
        auto insert_row = [&](double s, int32_t row) {
            if (s < gthr) return;                          // below another split's k-th score
            if (cnt == k && !(s > thr)) return;            // ties with the current worst keep the lower index
            // the list is unordered while it runs: overwrite the worst entry, then find the new worst with k
            // independent loads (a sorted insert would be a dependent load-compare-store chain per position)
            const int pos = cnt < k ? cnt : wpos;
            ls[(size_t)pos * TC_QT] = s;
            li[(size_t)pos * TC_QT] = row;
            if (cnt < k) cnt++;
            thr_dirty = true;
            if (cnt == k) {
                double w = INFINITY, w1 = INFINITY;       // two independent scans (even / odd entries)
                int32_t wi = -1, wi1 = -1;
                int wp = 0, wp1 = 0;
                int e = 0;
                for (; e + 1 < k; e += 2) {
                    const double v = ls[(size_t)e * TC_QT], v1 = ls[(size_t)(e + 1) * TC_QT];
                    const int32_t vi = li[(size_t)e * TC_QT], vi1 = li[(size_t)(e + 1) * TC_QT];
                    if (v < w || (v == w && vi > wi)) { w = v; wi = vi; wp = e; }
                    if (v1 < w1 || (v1 == w1 && vi1 > wi1)) { w1 = v1; wi1 = vi1; wp1 = e + 1; }
                }
                if (e < k) {
                    const double v = ls[(size_t)e * TC_QT];
                    const int32_t vi = li[(size_t)e * TC_QT];
                    if (v < w || (v == w && vi > wi)) { w = v; wi = vi; wp = e; }
                }
                if (w1 < w || (w1 == w && wi1 > wi)) { w = w1; wp = wp1; }
                thr = w;
                wpos = wp;
                if (gslot && thr > gthr) atomicMax(gslot, tc_enc(thr));
            }
        };
        // Re-scoring is shared by the warp: the pending rows of all 32 queries form one work list (prefix sum of the ring
        // fill counts), lane i scores item i of it -- any query's row, the exact left-to-right float64 fma chain -- and
        // leaves the score next to the ring entry; then every lane inserts its own rows in order.  A scoring pass costs
        // the same whether 1 or 32 lanes have work (latency of the float64 row loads); with one candidate per lane and
        // pass, ~5 pending rows per warp kept 27 lanes idle for as many passes as the fullest ring held.
        auto drain = [&]() {
            for (;;) {
                if (!__any_sync(0xffffffffu, f_cnt > 0)) break;
                int pre = f_cnt;                                   // inclusive prefix sum of the fill counts
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, pre, o);
                    if (lane >= o) pre += v;
                }
                const int total = __shfl_sync(0xffffffffu, pre, 31);
                for (int w = lane; w - lane < total; w += 32) {    // warp-uniform trip count
                    int owner = 0;                                 // first lane whose prefix exceeds w
#pragma unroll
                    for (int step = 16; step >= 1; step >>= 1) {
                        const int pv = __shfl_sync(0xffffffffu, pre, owner + step - 1);
                        if (pv <= w) owner += step;
                    }
                    owner &= 31;
                    const int o_pre = __shfl_sync(0xffffffffu, pre, owner), o_cnt = __shfl_sync(0xffffffffu, f_cnt, owner);
                    const int o_head = __shfl_sync(0xffffffffu, f_head, owner);
                    if (w < total) {
                        const int slot = (o_head + (w - (o_pre - o_cnt))) & (TC_FIFO - 1);
                        const int oq = (tid & ~31) + owner;         // the owner's query slot in this CTA
                        const int64_t row = s_fifo[(size_t)slot * TC_QT + oq];
                        const double *d = p.dbn + (size_t)row * dim;
                        const double *qo = p.qn + (size_t)(q0 + oq) * dim;
                        double sc = 0.0;
                        if (DIM > 0) {
                            double dv[DIM > 0 ? DIM : 1], qv[DIM > 0 ? DIM : 1];
#pragma unroll
                            for (int c = 0; c < DIM; c++) { dv[c] = d[c]; qv[c] = qo[c]; }
#pragma unroll
                            for (int c = 0; c < DIM; c++) sc = fma(qv[c], dv[c], sc);
                        } else {
                            int c = 0;
                            for (; c + 8 <= dim; c += 8) {
                                double dv[8], qv[8];
#pragma unroll
                                for (int j = 0; j < 8; j++) { dv[j] = d[c + j]; qv[j] = qo[c + j]; }
#pragma unroll
                                for (int j = 0; j < 8; j++) sc = fma(qv[j], dv[j], sc);
                            }
                            for (; c < dim; c++) sc = fma(qo[c], d[c], sc);
                        }
                        s_sc[(size_t)slot * TC_QT + oq] = sc;
                    }
                }
                __syncwarp();
                while (f_cnt > 0) {                                // own rows, in increasing row order
                    const int slot = f_head & (TC_FIFO - 1);
                    const int64_t row = fifo[(size_t)slot * TC_QT];
                    const double s = s_sc[(size_t)slot * TC_QT + ql];
                    f_head++;
                    f_cnt--;
                    insert_row(s, (int32_t)row);
                }
                __syncwarp();
            }
        };
        // queue the rows flagged in m (block order = row order); drains when a ring is full or 'force'.  Called only when
        // some lane has a hit or 'force': every exit leaves all rings below their trigger (drain() empties them), so a tile
        // without a hit has nothing to do here.
        auto enqueue = [&](uint32_t (&m)[4], int64_t tile, bool force) {
            for (;;) {
#pragma unroll
                for (int cb = 0; cb < 4; cb++) {
                    while (m[cb] && f_cnt < TC_FIFO) {
                        const int j = __ffs(m[cb]) - 1;
                        m[cb] &= m[cb] - 1;
                        const int64_t row = tile + cb * 32 + j;
                        if (row < r_end) {
                            fifo[(size_t)((f_head + f_cnt) & (TC_FIFO - 1)) * TC_QT] = (int32_t)row;
                            f_cnt++;
                        }
                    }
                }
                const bool more = __any_sync(0xffffffffu, (m[0] | m[1] | m[2] | m[3]) != 0);
                if (more || force || __any_sync(0xffffffffu, f_cnt >= TC_FIFO_TRIGGER) ||
                    (int)__reduce_add_sync(0xffffffffu, (unsigned)f_cnt) >= TC_WARP_TRIGGER) drain();
                if (!more) break;
            }
        };
        // The float threshold the scan compares against.  Its float64 arithmetic (max, subtract, round down) is kept off
        // the per-tile path: the FP64 pipe is shared by the SM and eight warps arriving together after acc_full queued on
        // it for ~90 cycles per instruction (ncu); it is recomputed only when the list's k-th score or the shared one moved.
        float thr32c = active ? -INFINITY : INFINITY;
        unsigned long long genc_seen = 0;
        auto filter_threshold = [&]() -> float {
            if (!active) return INFINITY;
            if (thr_dirty || genc != genc_seen) {                  // integer tests only on the common path
                thr_dirty = false;
                genc_seen = genc;
                const double eff = cnt == k ? fmax(thr, gthr) : gthr;
                thr32c = eff == -INFINITY ? -INFINITY : __double2float_rd((eff - TC_EPS) * (double)TC_SCALE);   // power of two: exact
            }
            return thr32c;
        };
        // The shared threshold is read one tile ahead: the load is issued when a tile arrives and consumed when the NEXT one
        // does, so its L2 round trip never sits on the path of a warp that is behind (the issue thread waits for the slowest).
        auto load_shared_thr = [&]() -> unsigned long long {
            unsigned long long v = 0;
            if (gslot) asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(gslot) : "memory");
            return v;
        };
        genc = load_shared_thr();                                  // what earlier CTAs of this query already reached
        unsigned long long genc_next = genc;
        if (genc) gthr = tc_dec(genc);
        // Take over the lists of the splits of this query tile that have already finished (CTAs are dispatched in order
        // of their linear index, so these are lower splits: lower row indices).  A split's own k-th score says little about
        // the final one -- with s splits it sits near rank s * k of the whole database, and shared_thr, the best of those,
        // let ~7x the necessary rows through -- but the k-th score over everything ranked so far is as tight as a bound
        // can be.  The foreign rows only serve as the threshold: they are left out when the list is written (their own
        // split reported them), and an own row they displace has k better rows ahead of it in the database.
        if (pp.done && split > 0) {
            for (int j = 0; j < split; j++) {
                int fin;
                asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(fin) : "l"(pp.done + (size_t)blockIdx.x * p.n_splits + j) : "memory");
                if (!__all_sync(0xffffffffu, fin != 0)) continue;
                if (!active) continue;
                const size_t o = ((size_t)gq * p.n_splits + j) * k;
                for (int e = 0; e < k; e++) {
                    const int32_t fi = __ldcg(p.idx_out + o + e);
                    if (fi < 0) break;                             // lists are written compacted, best first
                    insert_row(__ldcg(p.score_out + o + e), fi);
                }
            }
            __syncwarp();
        }
#ifdef DSPX_TC_PROFILE
        long long tc_prof_local[16] = {0};
#endif
        TC_PROF_T0();
        for (int64_t t = 0; t < n_tiles; t++) {
            const int buf = (int)(t & 1);
            const int64_t tile = r_begin + t * TC_ROWS;
            // Wait for the tile.  A long wait means some other warp is re-scoring and holds the pipeline up (the issue
            // thread needs all eight warps to hand a buffer back): re-score what this warp has pending NOW, while the
            // time is free, instead of stalling everybody again when its own ring reaches the trigger.
            {
                const uint32_t parity = (uint32_t)((t >> 1) & 1);
                bool drained = false;
                const long long w0 = clock64();
                for (uint32_t spin = 0;; spin++) {
                    uint32_t ok;                                   // test_wait: try_wait would sleep through the whole stall
                    asm volatile("{ .reg .pred p; mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                                 : "=r"(ok) : "r"(tc_smem_u32(&my_full[buf])), "r"(parity) : "memory");
                    if (__all_sync(0xffffffffu, ok != 0)) break;
                    if (spin > (1u << 28)) __trap();
                    if (!drained && __any_sync(0xffffffffu, f_cnt > 0 && clock64() - w0 > TC_IDLE_CYCLES)) {
                        drain();
                        drained = true;
                    }
                }
            }
            TC_PROF_ADD(5);
            if (lane == 0) TC_TRACE(t, 2 + warp);
            __syncwarp();                                          // tcgen05.ld is warp-collective
            asm volatile("tcgen05.fence::after_thread_sync;");
            genc = genc_next;
            genc_next = load_shared_thr();                         // for the next tile
            if (genc) gthr = tc_dec(genc);
            const uint32_t acc = lane_base + (uint32_t)(buf * 2 * TC_ROWS);
            uint32_t m[4] = {0u, 0u, 0u, 0u};
            bool released = false, any_hit = true;
            if (t == 0) {
                // the list is empty: take the first tile 32 columns at a time so the threshold tightens as it fills
#pragma unroll
                for (int cb = 0; cb < 3; cb++) {
                    m[cb] = tc_ld_mask(acc + cb * 32, filter_threshold());
                    enqueue(m, tile, true);
                }
                m[3] = tc_ld_mask(acc + 96, filter_threshold());
            } else {
                // All 128 scores of the row go to registers first and the buffer is handed back to the tensor core BEFORE
                // they are scanned: the issue thread waits for the slowest of the eight warps, and what it waited for was
                // their scans (event trace in profiles/r02_topk_tc_pipeline.md), not the 4 x 4 KB of TMEM reads.
                const float thr32 = filter_threshold();
                uint32_t v0[32], v1[32], v2[32], v3[32];
                tc_ld32_issue(acc, v0);
                tc_ld32_issue(acc + 32, v1);
                tc_ld32_issue(acc + 64, v2);
                tc_ld32_issue(acc + 96, v3);
                tc_ld_wait(v0);
                tc_ld_wait(v1);
                tc_ld_wait(v2);
                tc_ld_wait(v3);
                asm volatile("tcgen05.fence::before_thread_sync;");
                __syncwarp();
                if (lane == 0) tc_mbar_arrive(&my_empty[buf]);
                if (lane == 0) TC_TRACE(t, 10 + warp);
                released = true;
                const float t0 = tc_top32(v0), t1 = tc_top32(v1), t2 = tc_top32(v2), t3 = tc_top32(v3);
                any_hit = __any_sync(0xffffffffu, fmaxf(fmaxf(t0, t1), fmaxf(t2, t3)) > thr32);
                if (any_hit) {
                    if (__any_sync(0xffffffffu, t0 > thr32)) m[0] = tc_bits32(v0, thr32);
                    if (__any_sync(0xffffffffu, t1 > thr32)) m[1] = tc_bits32(v1, thr32);
                    if (__any_sync(0xffffffffu, t2 > thr32)) m[2] = tc_bits32(v2, thr32);
                    if (__any_sync(0xffffffffu, t3 > thr32)) m[3] = tc_bits32(v3, thr32);
                }
            }
            if (!released) {
                asm volatile("tcgen05.fence::before_thread_sync;");
                __syncwarp();
                if (lane == 0) tc_mbar_arrive(&my_empty[buf]);    // the tensor core may overwrite this buffer now
                if (lane == 0) TC_TRACE(t, 10 + warp);
            }
            TC_PROF_ADD(6);
            {
                const bool force = t < 4 || t == n_tiles - 1;
                if (any_hit || force) enqueue(m, tile, force);
            }
            TC_PROF_ADD(7);
        }
#ifdef DSPX_TC_PROFILE
        if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0) { for (int i = 5; i < 8; i++) tc_prof[i] = tc_prof_local[i]; tc_prof[8] = n_tiles; }
#endif
        if (active) {
            // order the list once: score descending, ties to the lower index (selection sort in place)
            for (int a = 0; a + 1 < cnt; a++) {
                int best = a;
                double bs = ls[(size_t)a * TC_QT];
                int32_t bi = li[(size_t)a * TC_QT];
                for (int e = a + 1; e < cnt; e++) {
                    const double v = ls[(size_t)e * TC_QT];
                    const int32_t vi = li[(size_t)e * TC_QT];
                    if (v > bs || (v == bs && vi < bi)) { bs = v; bi = vi; best = e; }
                }
                if (best != a) {
                    ls[(size_t)best * TC_QT] = ls[(size_t)a * TC_QT];
                    li[(size_t)best * TC_QT] = li[(size_t)a * TC_QT];
                    ls[(size_t)a * TC_QT] = bs;
                    li[(size_t)a * TC_QT] = bi;
                }
            }
            const size_t o = ((size_t)gq * p.n_splits + split) * k;
            int w = 0;
            for (int e = 0; e < cnt; e++) {                        // rows taken over from other splits are not reported twice
                const int32_t ri = li[(size_t)e * TC_QT];
                if (ri < r_begin || ri >= r_end) continue;
                p.idx_out[o + w] = ri;
                if (p.score_out) p.score_out[o + w] = ls[(size_t)e * TC_QT];
                w++;
            }
            for (; w < k; w++) {
                p.idx_out[o + w] = -1;
                if (p.score_out) p.score_out[o + w] = -INFINITY;
            }
        }
        if (pp.done) __threadfence();                              // the lists, before the flag below
    } else if (warp == TC_EPI_THREADS / 32) {
        // ===== bulk copies: one thread =====
        // The operand images were written by normalize_rows_split16_kernel in the layout the tensor core reads, so a tile is
        // one 16 KB cp.async.bulk; TC_STAGES tiles are in flight (a copy takes ~1 us to land, a tile lasts ~0.5 us).
        if (lane == 0) {
#ifdef DSPX_TC_PROFILE
            long long tc_prof_local[16] = {0};
#endif
            tc_mbar_expect_tx(a_full, 2 * TC_TILE_BYTES);
            tc_bulk_load(a_x, pp.qx + (size_t)blockIdx.x * 2 * TC_TILE_BYTES, 2 * TC_TILE_BYTES, a_full);
            const unsigned char *src = pp.dbx + (size_t)(r_begin / TC_ROWS) * TC_TILE_BYTES;
            TC_PROF_T0();
            for (int64_t t = 0; t < n_tiles; t++) {
                const int s = (int)(t % TC_STAGES);
                tc_mbar_wait(&empty_b[s], (uint32_t)(((t / TC_STAGES) & 1) ^ 1));
                TC_PROF_ADD(3);
                tc_mbar_expect_tx(&full_b[s], TC_TILE_BYTES);
                tc_bulk_load(b_x + s * TC_TILE_BYTES, src + (size_t)t * TC_TILE_BYTES, TC_TILE_BYTES, &full_b[s]);
                TC_PROF_ADD(4);
            }
#ifdef DSPX_TC_PROFILE
            if (blockIdx.x == 0 && blockIdx.y == 0) { tc_prof[3] = tc_prof_local[3]; tc_prof[4] = tc_prof_local[4]; }
#endif
        }
    } else if (lane == 0) {
        // ===== tensor-core issue: one thread per query half =====
        // kind::f16: fp16 x fp16 -> float32 (formats 0, 0; accumulator format 1), N = 128, M = 128, both operands K-major
        const uint32_t idesc16 = (1u << 4) | ((uint32_t)(TC_ROWS >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const int a = warp - (TC_EPI_THREADS / 32 + 1);             // 0: queries 0-127, 1: queries 128-255
        uint64_t *my_full = acc_full + a * 2, *my_empty = acc_empty + a * 2;
#ifdef DSPX_TC_PROFILE
        long long tc_prof_local[16] = {0};
        const long long tc_start = clock64();
#endif
        tc_mbar_wait(a_full, 0);                                   // the query tiles have landed
        const uint64_t ad = tc_desc(a_x + a * TC_TILE_BYTES);
        TC_PROF_T0();
        for (int64_t t = 0; t < n_tiles; t++) {
            const int s = (int)(t % TC_STAGES), buf = (int)(t & 1);
            tc_mbar_wait(&my_empty[buf], (uint32_t)(((t >> 1) & 1) ^ 1));
            TC_PROF_ADD(0);
            if (a == 0) TC_TRACE(t, 0);
            tc_mbar_wait(&full_b[s], (uint32_t)((t / TC_STAGES) & 1));
            TC_PROF_ADD(1);
            asm volatile("tcgen05.fence::after_thread_sync;");
            // a 128-byte row holds K = 64 halves [S hi | S lo]: +2 per K = 16 step (32 bytes) in descriptor units, +4 = the lo half
            const uint64_t bd = tc_desc(b_x + s * TC_TILE_BYTES);
            const uint32_t d = tmem + (uint32_t)(buf * 2 * TC_ROWS + a * TC_ROWS);
            tc_mma_f16(d, ad + 4, bd, idesc16, 0);                 // A_lo B_hi   (small terms first)
            tc_mma_f16(d, ad + 6, bd + 2, idesc16, 1);
            tc_mma_f16(d, ad, bd + 4, idesc16, 1);                 // A_hi B_lo
            tc_mma_f16(d, ad + 2, bd + 6, idesc16, 1);
            tc_mma_f16(d, ad, bd, idesc16, 1);                     // A_hi B_hi
            tc_mma_f16(d, ad + 2, bd + 2, idesc16, 1);
            tc_commit(&empty_b[s]);                                // smem stage free once both halves' MMAs have read it
            tc_commit(&my_full[buf]);                              // this half's accumulators complete
            TC_PROF_ADD(2);
            if (a == 0) TC_TRACE(t, 1);
        }
#ifdef DSPX_TC_PROFILE
        if (a == 0 && blockIdx.x == 0 && blockIdx.y == 0) { for (int i = 0; i < 3; i++) tc_prof[i] = tc_prof_local[i]; tc_prof[9] = clock64() - tc_start; }
#endif
    }

    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    __syncwarp();
    if (pp.done && tid == 0)
        asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(pp.done + (size_t)blockIdx.x * p.n_splits + split), "r"(1) : "memory");
    if (warp == TC_THREADS / 32 - 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
}

#endif

}  // namespace dspx
