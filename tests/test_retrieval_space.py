"""Cosine top-k across the shapes that choose its kernel, against the float64 oracle (oracle/dsp_oracle.c).

dspx_cosine_topk returns the oracle's indices and float64 scores bit for bit, ties to the lower index (DESIGN.md 4.3),
through one of three kernels -- the tensor-core split-fp16 filter, the packed-FP32 filter, the float64 kernel -- each
with two template instantiations, and a merge of the per-split lists when the database is split.  topk_select
(csrc/retrieval_select.cuh) picks the kernel, the split count and the grid from (nq, ndb, dim, k, SM count).

CPU: topk_select and the workspace layout topk_ws_carve, through the test-only exports emu_topk_select and
emu_topk_workspace of libdspx_emu.so, over a grid of shapes that crosses every boundary of the choice; and the claims of
the GPU case list.  GPU (-m gpu): SWEEP, an explicit list of cases that together launch every instantiation with one
split and with several, every family with a grid larger than the GPU, the float64 kernel at 32 splits, both sides of
every query-tile edge, ndb at 127/128/129 and k == ndb, and k at 1, 24, 25, every FP32 ceiling and one above it, and 128.
Each case runs through five entry points and hard data; a profiled run checks that the kernel, grid, block and shared
memory that ran are what topk_select says.  Also: database rows above 2^24 (the 2 GiB and 4 GiB offsets),
cosine_similarity, hits@k and the API's edges.
"""
from __future__ import annotations

import ctypes as C
import json
import math
import subprocess
import sys
import zlib
from dataclasses import dataclass

import numpy as np
import pytest

from conftest import REPO

TC, F32, F64 = 0, 1, 2
FAMILY = {TC: "TC", F32: "F32", F64: "F64"}
QUERY_TILE = {TC: 256, F32: 128, F64: 64}           # queries per CTA of each kernel
THREADS = {TC: 352, F32: 512, F64: 256}
TC_MAX_K = 24
MAX_K = 128
MAX_SPLITS = {TC: 16, F32: 16, F64: 32}
F32_SMEM_LIMIT = 200 * 1024
OPTIN_SMEM = 227 * 1024
# largest k of the FP32 filter at each dim (its shared memory <= 200 KB); above it the float64 kernel runs
F32_CEILING = {1: 99, 2: 97, 13: 75, 25: 51, 26: 55, 27: 47, 31: 39, 32: 37}


# ---- the launch topk_select chooses, read through the replay library ------------------------------------------------
@dataclass(frozen=True)
class Launch:
    kernel: int
    cw: int                     # template argument
    grid: tuple
    threads: int
    smem: int                   # dynamic shared memory
    n_splits: int
    rows_per_split: int

    @property
    def name(self) -> str:
        return f"{FAMILY[self.kernel]}<{self.cw}>"


@pytest.fixture(scope="module")
def emu():
    from dsp_final_b200 import build

    build.build_native()
    return C.CDLL(str(build.build_emu()))


def select(emu, nq, ndb, dim, k, sm_count=148) -> Launch:
    out = np.zeros(8, np.int64)
    rc = emu.emu_topk_select(C.c_int64(nq), C.c_int64(ndb), C.c_int(dim), C.c_int(k), C.c_int(sm_count),
                             out.ctypes.data_as(C.c_void_p))
    assert rc == 0, (nq, ndb, dim, k, sm_count)
    v = [int(x) for x in out]
    return Launch(v[0], v[1], (v[2], v[3]), v[4], v[5], v[6], v[7])


WS_REGIONS = ("qn", "dbn", "pscore", "pidx", "qf", "dbf", "shared_thr", "split_done")


def workspace(emu, nq, ndb, dim, k):
    """({region: (offset, extent)}, total) of topk_ws_carve"""
    out = np.zeros(17, np.int64)
    rc = emu.emu_topk_workspace(C.c_int64(nq), C.c_int64(ndb), C.c_int(dim), C.c_int(k), out.ctypes.data_as(C.c_void_p))
    assert rc == 0, (nq, ndb, dim, k)
    return {r: (int(out[2 * i]), int(out[2 * i + 1])) for i, r in enumerate(WS_REGIONS)}, int(out[16])


# ---- CPU: topk_select and topk_ws_carve over the grid ----------------------------------------------------------------
GRID_NQ = (1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 10_240, 65_535, 1_000_000)
GRID_NDB = (1, 127, 128, 129, 1_023, 1_024, 1_025, 4_097, 300_000, 21_000_000, 2**31 - 2)
GRID_DIM = (1, 2, 13, 25, 26, 27, 31, 32, 33, 64, 65, 2048)
GRID_K = sorted({1, TC_MAX_K, TC_MAX_K + 1, MAX_K} | {c for c in F32_CEILING.values()}
                | {c + 1 for c in F32_CEILING.values()})
GRID_SM = (148, 132, 1)


def expected_kernel(dim, k):
    """DESIGN.md 4.3: the tensor-core filter iff dim <= 32 and k <= 24; else the FP32 filter iff dim <= 32 and its
    shared memory fits 200 KB (the ceilings of F32_CEILING); else the float64 kernel"""
    if dim <= 32 and k <= TC_MAX_K:
        return TC
    if dim <= 32 and k <= F32_CEILING[dim]:
        return F32
    return F64


def check_launch(L: Launch, nq, ndb, dim, k, tag):
    assert L.kernel == expected_kernel(dim, k), tag
    assert L.cw == (26 if dim == 26 else 0 if L.kernel == TC else 32), tag
    assert L.threads == THREADS[L.kernel], tag
    assert 0 < L.smem <= OPTIN_SMEM, tag
    if L.kernel == F32:
        assert L.smem <= F32_SMEM_LIMIT, tag
    assert 1 <= L.n_splits <= MAX_SPLITS[L.kernel], tag
    rps = L.rows_per_split
    assert rps > 0 and rps % 128 == 0, tag
    assert (L.n_splits - 1) * rps < ndb <= L.n_splits * rps, tag          # no split is empty
    assert L.grid == (-(-nq // QUERY_TILE[L.kernel]), L.n_splits), tag


def check_workspace(emu, lib, L: Launch, nq, ndb, dim, k, tag):
    regions, total = workspace(emu, nq, ndb, dim, k)
    assert total == lib.dspx_cosine_topk_workspace(nq, ndb, dim, k), tag
    end = 0
    for r in WS_REGIONS:                                                  # in carve order: aligned, disjoint, inside
        off, ext = regions[r]
        assert off % 256 == 0 and off >= end and ext >= 0, (tag, r)
        end = off + ext
    assert end <= total, tag
    need = {"qn": nq * dim * 8, "dbn": ndb * dim * 8, "shared_thr": nq * 8,
            "pscore": nq * L.n_splits * k * 8, "pidx": nq * L.n_splits * k * 4}
    if L.kernel == TC:
        need["split_done"] = L.grid[0] * L.n_splits * 4
        need["qf"] = -(-nq // 256) * 32 * 1024                            # fp16 split image: 128 B per row
        need["dbf"] = -(-ndb // 128) * 16 * 1024
    elif L.kernel == F32:
        need["qf"] = -(-nq // 128) * dim * 128 * 4                        # [tiles][dim][128] floats
        need["dbf"] = -(-ndb // 128) * dim * 128 * 4
    for r, n in need.items():
        assert regions[r][1] >= n, (tag, r, regions[r], n)


def test_selection_and_workspace_over_the_grid(emu):
    from dsp_final_b200 import _lib

    lib = _lib.load()
    n = 0
    for dim in GRID_DIM:
        for k in GRID_K:
            for ndb in GRID_NDB:
                if k > ndb:
                    continue
                for nq in GRID_NQ:
                    for sm in GRID_SM:
                        L = select(emu, nq, ndb, dim, k, sm)
                        check_launch(L, nq, ndb, dim, k, (nq, ndb, dim, k, sm))
                        n += 1
                        if sm == 148:
                            check_workspace(emu, lib, L, nq, ndb, dim, k, (nq, ndb, dim, k))
    assert n > 50_000


def test_kernel_order_and_ceilings(emu):
    """For each dim, k = 1..128 runs through the tensor-core filter, then the FP32 filter, then the float64 kernel, never
    back; the FP32 ceilings are the largest k whose lists fit 200 KB of shared memory."""
    for dim in sorted(set(GRID_DIM) | set(range(1, 34))):
        seq = [select(emu, 300, 100_000, dim, k) for k in range(1, MAX_K + 1)]
        kinds = [L.kernel for L in seq]
        assert kinds == sorted(kinds), dim
        if dim > 32:
            assert set(kinds) == {F64}, dim
            continue
        assert kinds[:TC_MAX_K] == [TC] * TC_MAX_K, dim
        f32 = [L for L in seq if L.kernel == F32]
        assert f32 and all(L.smem <= F32_SMEM_LIMIT for L in f32), dim
        ceiling = TC_MAX_K + len(f32)
        if dim in F32_CEILING:
            assert ceiling == F32_CEILING[dim], (dim, ceiling)
        if ceiling < MAX_K:                                               # the FP32 filter at ceiling + 1 would not fit
            assert seq[ceiling].kernel == F64, dim


def test_workspace_of_empty_inputs(emu):
    from dsp_final_b200 import _lib

    lib = _lib.load()
    for nq, ndb in ((0, 5), (3, 0), (0, 0)):                              # cosine_similarity sizes these
        regions, total = workspace(emu, nq, ndb, 26, 1)
        assert total == lib.dspx_cosine_topk_workspace(nq, ndb, 26, 1) and total >= 1024
    assert lib.dspx_cosine_topk_workspace(-1, 5, 26, 1) == 0
    assert lib.dspx_cosine_topk_workspace(5, 5, 0, 1) == 0
    assert lib.dspx_cosine_topk_workspace(5, 5, 26, 0) == 0


def test_empty_inputs_take_null_buffers():
    """An empty tensor has no storage (torch's data_ptr() is 0).  With no query, or no database row to score, the ranking
    and the matrix accept NULL for the empty buffers and return before they touch the device; a NULL buffer that holds
    data is still an error."""
    from dsp_final_b200 import _lib

    lib = _lib.load()
    rows = np.zeros((5, 26), np.float32)                       # never read: the calls return before any copy or launch
    n = lib.dspx_cosine_topk_workspace(5, 5, 26, 5)
    ws = np.zeros(n, np.uint8)
    p, w = rows.ctypes.data, ws.ctypes.data
    assert lib.dspx_cosine_topk(None, 0, p, 5, 26, _lib.DTYPE_F32, 5, None, None, w, n, None) == 0
    assert lib.dspx_cosine_matrix(None, 0, p, 5, 26, _lib.DTYPE_F32, None, w, n, None) == 0
    assert lib.dspx_cosine_matrix(p, 3, None, 0, 26, _lib.DTYPE_F32, None, w, n, None) == 0
    assert lib.dspx_cosine_topk(None, 3, p, 5, 26, _lib.DTYPE_F32, 5, p, None, w, n, None) == _lib.EINVAL
    assert lib.dspx_cosine_topk(p, 3, p, 5, 26, _lib.DTYPE_F32, 5, None, None, w, n, None) == _lib.EINVAL
    assert lib.dspx_cosine_matrix(p, 3, None, 5, 26, _lib.DTYPE_F32, None, w, n, None) == _lib.EINVAL


# ---- the GPU case list ------------------------------------------------------------------------------------------------
KINDS = ("clustered", "band", "negative", "identical", "scale", "straddle")


@dataclass(frozen=True)
class Case:
    nq: int
    ndb: int
    dim: int
    k: int
    kind: str
    kernel: str                 # claimed at 148 SMs (test_case_list_claims)
    split: bool                 # n_splits > 1
    waves: bool                 # more CTAs than SMs

    @property
    def id(self) -> str:
        return f"{self.kernel}-q{self.nq}-n{self.ndb}-d{self.dim}-k{self.k}-{self.kind}"


SWEEP = [
    # the shapes of the former test_retrieval_vs_oracle_shapes
    Case(1, 20, 26, 20, "scale", "TC<26>", False, False),               # k == ndb
    Case(63, 129, 26, 1, "identical", "TC<26>", False, False),
    Case(400, 1_600, 26, 20, "clustered", "TC<26>", True, False),
    Case(130, 40_000, 26, 20, "band", "TC<26>", True, False),
    Case(70, 3_000, 80, 10, "negative", "F64<32>", True, False),
    Case(33, 700, 128, 128, "clustered", "F64<32>", True, False),
    Case(5, 300_000, 26, 20, "straddle", "TC<26>", True, False),
    # grids larger than the GPU
    Case(10_240, 200_000, 13, 20, "band", "TC<0>", True, True),
    Case(8_000, 250_000, 29, 33, "band", "F32<32>", True, True),
    Case(5_000, 400_000, 26, 40, "straddle", "F32<26>", True, True),
    Case(9_000, 300_000, 100, 64, "straddle", "F64<32>", True, True),
    # the float64 kernel at 32 splits
    Case(5, 300_000, 26, 100, "straddle", "F64<26>", True, False),
    Case(130, 40_000, 64, 20, "straddle", "F64<32>", True, False),
    # query-tile edges (TC 128 / 256, FP32 128, float64 64), ndb 127 / 128 / 129, k == ndb
    Case(257, 129, 26, 24, "negative", "TC<26>", False, False),
    Case(255, 33_000, 25, 24, "band", "TC<0>", True, False),
    Case(256, 4_097, 27, 5, "straddle", "TC<0>", True, False),
    Case(128, 1_000, 2, 10, "clustered", "TC<0>", False, False),
    Case(129, 9_000, 31, 24, "scale", "TC<0>", True, False),
    Case(128, 1_024, 26, 25, "clustered", "F32<26>", False, False),
    Case(127, 3_000, 32, 37, "band", "F32<32>", True, False),
    Case(64, 128, 32, 38, "identical", "F64<32>", False, False),
    Case(63, 129, 33, 1, "clustered", "F64<32>", False, False),
    Case(65, 2_000, 26, 56, "scale", "F64<26>", True, False),
    Case(65, 128, 26, 128, "negative", "F64<26>", False, False),        # k == ndb
    Case(3, 127, 2, 127, "identical", "F64<32>", False, False),         # k == ndb
    # the FP32 ceilings and one above them, dims 1 ... 2048
    Case(1, 1_024, 1, 99, "negative", "F32<32>", False, False),
    Case(2, 5_000, 1, 100, "scale", "F64<32>", True, False),
    Case(600, 50_000, 13, 75, "straddle", "F32<32>", True, False),
    Case(100, 8_000, 13, 76, "clustered", "F64<32>", True, False),
    Case(255, 33_000, 25, 51, "negative", "F32<32>", True, False),
    Case(200, 9_000, 25, 52, "scale", "F64<32>", True, False),
    Case(129, 100_000, 26, 55, "band", "F32<26>", True, False),
    Case(64, 129, 27, 47, "identical", "F32<32>", False, False),
    Case(129, 6_000, 27, 48, "straddle", "F64<32>", True, False),
    Case(300, 20_000, 31, 39, "band", "F32<32>", True, False),
    Case(40, 5_000, 31, 40, "negative", "F64<32>", True, False),
    Case(70, 3_000, 65, 10, "scale", "F64<32>", True, False),
    Case(400, 1_600, 2048, 20, "clustered", "F64<32>", True, False),
]
IDS = [c.id for c in SWEEP]

# database rows above 2^24 (fp16 operand image past 2 GiB) and above 20 648 881 (float64 rows past 4 GiB at dim 26)
LARGE_NDB, LARGE_FROM = 21_000_000, 20_648_881
LARGE = {20: ("TC<26>", True), 30: ("F32<26>", True), 60: ("F64<26>", True)}


def test_case_list_claims(emu):
    """Every case selects the kernel, split regime and wave count it claims at 148 SMs, and the list covers what the
    module docstring says it covers."""
    got = {}
    for c in SWEEP:
        L = select(emu, c.nq, c.ndb, c.dim, c.k)
        got[c.id] = L
        assert (L.name, L.n_splits > 1, L.grid[0] * L.grid[1] > 148) == (c.kernel, c.split, c.waves), (c.id, L)
        assert c.kind in KINDS and c.k <= c.ndb
    for k, (name, split) in LARGE.items():
        L = select(emu, 8, LARGE_NDB, 26, k)
        assert (L.name, L.n_splits > 1) == (name, split), (k, L)
        assert L.n_splits * L.rows_per_split > LARGE_FROM
    assert select(emu, 8, LARGE_NDB, 26, 60).n_splits == 32
    coverage_claims(list(got.values()), 148)
    assert {c.dim for c in SWEEP} >= {1, 2, 13, 25, 26, 27, 31, 32, 33, 64, 65, 2048}
    assert any(80 <= c.dim <= 100 for c in SWEEP)
    ks = {(c.dim, c.k) for c in SWEEP}
    for dim, ceiling in F32_CEILING.items():
        if dim != 2:
            assert (dim, ceiling) in ks and (dim, ceiling + 1) in ks, dim
    assert {1, 24, 25, 128} <= {c.k for c in SWEEP}
    assert {127, 128, 129} <= {c.ndb for c in SWEEP}
    assert {c.ndb for c in SWEEP if c.k == c.ndb} >= {127, 128}
    for fam, edge in ((TC, 128), (TC, 256), (F32, 128), (F64, 64)):
        nqs = {c.nq for c in SWEEP if got[c.id].kernel == fam}
        assert {edge, edge + 1} <= nqs, (FAMILY[fam], edge, sorted(nqs))       # the last query of a tile, and one more
    assert set(KINDS) == {c.kind for c in SWEEP}


def coverage_claims(launches, sm_count):
    """launches: Launch (or what ran) of every case.  All six instantiations with one split and with several, every
    family with a grid larger than the GPU, the float64 kernel at 32 splits."""
    seen = {(L.name, L.n_splits > 1) for L in launches}
    for name in ("TC<26>", "TC<0>", "F32<26>", "F32<32>", "F64<26>", "F64<32>"):
        assert (name, False) in seen and (name, True) in seen, name
    for fam in (TC, F32, F64):
        assert any(L.kernel == fam and L.grid[0] * L.grid[1] > sm_count for L in launches), FAMILY[fam]
    assert any(L.kernel == F64 and L.n_splits == 32 for L in launches)


# ---- GPU: data, entry points and checks -------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def oracle_rows(nq: int, L: Launch) -> list:
    """Queries checked against the oracle, at most 64: the first and last of every query tile and, for the tensor-core
    filter, both 128-query halves of the first tile.  When the tile edges come to more than 64 queries (grids of more
    than 32 query tiles), query 0, query nq - 1 and the halves of the first tile stay, and the rest of the tile edges are
    thinned to an even spread."""
    qt = QUERY_TILE[L.kernel]
    rows, must = set(), {0, nq - 1}
    for t in range(-(-nq // qt)):
        rows |= {t * qt, min(nq, (t + 1) * qt) - 1}
        if L.kernel == TC:
            halves = {r for r in (t * qt + 127, t * qt + 128) if r < nq}
            rows |= halves
            if t == 0:
                must |= halves
    rows = sorted(rows)
    if len(rows) > 64:
        rest = [r for r in rows if r not in must]
        pick = np.linspace(0, len(rest) - 1, 64 - len(must)).round().astype(int)
        rows = sorted(must | {rest[i] for i in pick})
    return rows


def case_data(c: Case, L: Launch, sample: list):
    """float32 queries and database (every entry point converts them exactly to the same doubles): Gaussian rows with
    planted exact duplicates and zero rows, plus the case's harder kind."""
    rng = np.random.default_rng(zlib.crc32(c.id.encode()))
    f32 = np.float32
    q = rng.standard_normal((c.nq, c.dim), dtype=f32)
    db = rng.standard_normal((c.ndb, c.dim), dtype=f32)
    if c.kind == "clustered":                                  # every cosine > 0.9999
        base = rng.standard_normal(c.dim, dtype=f32) * f32(5.0)
        q = base + f32(0.01) * q
        db = base + f32(0.01) * db
    elif c.kind == "negative":                                 # every cosine < 0
        base = np.abs(rng.standard_normal(c.dim, dtype=f32)) + f32(0.5)
        q = base + f32(0.05) * q
        db = -base + f32(0.05) * db
    elif c.kind == "identical":                                # all ties
        db[:] = db[0]
    elif c.kind == "scale":                                    # norms far below the 1e-10 of the normalisation, and huge
        q[1::2] *= f32(1e-20)
        db[1::3] *= f32(1e30)
        db[2::3] *= f32(1e-30)
    if c.kind != "identical" and c.ndb > 2:
        db[c.ndb // 2] = db[0]                                 # exact duplicates
        db[c.ndb - 1] = db[1]
        if c.ndb > 10:
            db[7] = 0.0                                        # zero row: 0 / (0 + 1e-10)
    if c.nq > 2:
        q[c.nq // 2] = 0.0                                     # zero query: every score 0, ties throughout
    live = [i for i in sample if np.any(q[i])]
    if c.kind == "band":
        # per checked query, rows whose exact scores lie 1e-8 ... 1e-5 below 1 (log-uniform), so that hundreds of them lie
        # within float32 resolution of its k-th score and all within the filters' epsilon: the result rests on the exact
        # re-score and the tie order
        m = min(2000, c.ndb // (len(live) + 1))
        assert c.dim > 1 and m > c.k, c.id
        rows = rng.choice(c.ndb, len(live) * m, replace=False).reshape(len(live), m)
        for j, i in enumerate(live):
            v = q[i].astype(np.float64)
            u = rng.standard_normal((m, c.dim))
            u -= np.outer(u @ v, v) / (v @ v)
            u /= np.linalg.norm(u, axis=1, keepdims=True)
            s = np.linalg.norm(v) * np.sqrt(2.0 * 10.0 ** rng.uniform(-8, -5, m))   # 1 - cos ~ s^2 / (2 |v|^2)
            db[rows[j]] = (v + s[:, None] * u).astype(f32)
    elif c.kind == "straddle":
        # exact copies of a near-query row at the first and last rows of every split: ties across splits
        for j, i in enumerate(live):
            row = (q[i] * f32(1.5) + f32(0.01) * rng.standard_normal(c.dim, dtype=f32)).astype(f32)
            for s in range(L.n_splits):
                lo, hi = s * L.rows_per_split, min(c.ndb, (s + 1) * L.rows_per_split)
                db[[r for r in (lo + j, hi - 1 - j) if lo <= r < hi]] = row
    return np.ascontiguousarray(q, f32), np.ascontiguousarray(db, f32)


def entry_points(torch, q, db, k):
    """{name: (indices, scores) as NumPy} of one ranking through each entry point"""
    from dsp_final_b200 import retrieval as R

    def host(r):
        return tuple(x.cpu().numpy() if hasattr(x, "cpu") else x for x in r)

    out = {"numpy float32": R.cosine_topk(q, db, k, return_scores=True),
           "numpy float64": R.cosine_topk(q.astype(np.float64), db.astype(np.float64), k, return_scores=True)}
    qt, dt = torch.as_tensor(q).cuda(), torch.as_tensor(db).cuda()
    out["torch float32"] = host(R.cosine_topk(qt, dt, k, return_scores=True))

    def view(t):                                               # a column slice of a wider float64 tensor
        w = torch.full((t.shape[0], t.shape[1] + 3), 7.0, dtype=torch.float64, device="cuda")
        w[:, 2:2 + t.shape[1]] = t.double()
        return w[:, 2:2 + t.shape[1]]

    qv, dv = view(qt), view(dt)
    assert not qv.is_contiguous() or q.shape[0] <= 1
    out["torch float64 view"] = host(R.cosine_topk(qv, dv, k, return_scores=True))
    out["mixed float32 / float64"] = R.cosine_topk(q, db.astype(np.float64), k, return_scores=True)
    return out


def normalised(torch, x):
    t = torch.as_tensor(x).cuda().double() if not hasattr(x, "cuda") else x.double()
    return t / (torch.linalg.vector_norm(t, dim=1, keepdim=True) + 1e-10)


def check_structure(torch, q, db, idx, sc, tag):
    """Every query: indices in range and distinct, scores non-increasing, ties in index order, each score within 1e-12
    of float64 torch.matmul, and no row outside the list better than the k-th score by more than 1e-12."""
    I = torch.as_tensor(np.asarray(idx)).cuda().long() if not hasattr(idx, "cuda") else idx.long()
    S = torch.as_tensor(np.asarray(sc)).cuda() if not hasattr(sc, "cuda") else sc
    qn, dn = normalised(torch, q), normalised(torch, db)
    ndb = dn.shape[0]
    assert bool(((I >= 0) & (I < ndb)).all()), tag
    srt = I.sort(dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all()), (tag, "an index twice")
    assert bool((S[:, 1:] <= S[:, :-1]).all()), (tag, "scores increase")
    tie = S[:, 1:] == S[:, :-1]
    assert bool((I[:, 1:] > I[:, :-1])[tie].all()), (tag, "tie out of index order")
    step = max(1, (1 << 27) // ndb)
    for s in range(0, qn.shape[0], step):
        full = qn[s:s + step] @ dn.T
        err = (full.gather(1, I[s:s + step]) - S[s:s + step]).abs().max().item()
        assert err <= 1e-12, (tag, "score vs matmul", err)
        full.scatter_(1, I[s:s + step], -math.inf)
        worst = (full.max(dim=1).values - S[s:s + step, -1]).max().item()
        assert worst <= 1e-12, (tag, "a better row outside the list", worst)


@pytest.mark.gpu
@pytest.mark.parametrize("case", SWEEP, ids=IDS)
def test_case_matches_oracle(torch_cuda, emu, case):
    """Five entry points agree bit for bit; on the sample of oracle_rows, indices and scores equal the oracle's bit for
    bit; every query passes the structural checks."""
    torch = torch_cuda
    from oracle import oracle as O

    sm = torch.cuda.get_device_properties(0).multi_processor_count
    L = select(emu, case.nq, case.ndb, case.dim, case.k, sm)
    sample = oracle_rows(case.nq, L)
    q, db = case_data(case, L, sample)
    res = entry_points(torch, q, db, case.k)
    idx, sc = res["numpy float32"]
    assert idx.shape == (case.nq, case.k) and idx.dtype == np.int32 and sc.dtype == np.float64
    for name, (i2, s2) in res.items():
        assert np.array_equal(i2, idx) and np.array_equal(s2, sc), (case.id, name)
    want_idx, want_sc = O.cosine_topk(q[sample], db, case.k, return_scores=True)
    for j, i in enumerate(sample):
        assert np.array_equal(idx[i], want_idx[j]), (case.id, "query", i, idx[i][:8], want_idx[j][:8])
        assert np.array_equal(sc[i], want_sc[j]), (case.id, "query", i)
    check_structure(torch, q, db, idx, sc, case.id)


def _profiled_launches(out_path):
    """Runs every case of SWEEP once on random rows under one torch.profiler session and writes, per case, the ranking
    kernel's name, grid, block and shared memory and whether topk_merge_kernel ran.  Runs in a fresh process (see
    test_launches_match_selection)."""
    from pathlib import Path

    import torch
    from torch.profiler import ProfilerActivity, profile

    from dsp_final_b200 import retrieval as R

    torch.cuda.set_device(0)
    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    R.cosine_topk(torch.randn((3, 26), device="cuda"), torch.randn((300, 26), device="cuda"), 5)   # module load
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for c in SWEEP:
            q = torch.randn((c.nq, c.dim), generator=g, device="cuda")
            db = torch.randn((c.ndb, c.dim), generator=g, device="cuda")
            R.cosine_topk(q, db, c.k)
            torch.cuda.synchronize()
            del q, db
    trace = Path(out_path) / "trace.json"
    prof.export_chrome_trace(str(trace))
    events = sorted((e for e in json.loads(trace.read_text())["traceEvents"] if e.get("cat") == "kernel"),
                    key=lambda e: e["ts"])
    runs = []
    for e in events:
        name = e["name"]
        if "cosine_topk" in name and "kernel<" in name:
            runs.append({"name": name, "grid": e["args"]["grid"], "block": e["args"]["block"],
                         "smem": e["args"]["shared memory"], "merge": False})
        elif "topk_merge_kernel" in name and runs:
            runs[-1]["merge"] = True
    print(json.dumps({"sm": torch.cuda.get_device_properties(0).multi_processor_count, "runs": runs}))


def _launch_of(run) -> Launch:
    import re

    m = re.search(r"cosine_topk_(tc_|f32_)?kernel<(\d+)>", run["name"])
    assert m, run["name"]
    kernel = {"tc_": TC, "f32_": F32, None: F64}[m.group(1)]
    return Launch(kernel, int(m.group(2)), tuple(run["grid"][:2]), run["block"][0], run["smem"], run["grid"][1], 0)


@pytest.mark.gpu
def test_launches_match_selection(torch_cuda, tmp_path, emu):
    """The ranking kernel, template argument, grid, block and shared memory of every case are topk_select's at the
    device's SM count; topk_merge_kernel runs iff the database is split; the launches cover all the list claims.  The
    sweep is profiled in a fresh process: a torch.profiler session that an earlier test opened in this one can leave
    later sessions empty."""
    code = f"import sys; sys.path[:0] = [{str(REPO)!r}, {str(REPO / 'tests')!r}]; " \
           f"import test_retrieval_space; test_retrieval_space._profiled_launches({str(tmp_path)!r})"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    run = subprocess.run(cmd, capture_output=True, text=True, cwd=str(REPO), timeout=900)
    assert run.returncode == 0, run.stderr[-3000:]
    rec = json.loads(run.stdout.strip().splitlines()[-1])
    sm, runs = rec["sm"], rec["runs"]
    assert len(runs) == len(SWEEP), [r["name"] for r in runs]
    seen = []
    for c, r in zip(SWEEP, runs):
        want = select(emu, c.nq, c.ndb, c.dim, c.k, sm)
        got = _launch_of(r)
        print(f"{c.id}: {got.name} grid {r['grid']} block {r['block']} smem {r['smem']} merge {r['merge']}")
        assert (got.kernel, got.cw, got.grid, got.threads, got.smem) == \
               (want.kernel, want.cw, want.grid, want.threads, want.smem), (c.id, r, want)
        assert tuple(r["block"]) == (want.threads, 1, 1) and r["grid"][2] == 1, c.id
        assert r["merge"] == (want.n_splits > 1), (c.id, r)
        seen.append(got)
    coverage_claims(seen, sm)


@pytest.mark.gpu
def test_large_row_indices(torch_cuda):
    """nq 8, ndb 21 000 000, dim 26: rows above 2^24 (fp16 operand image past 2 GiB) and above 20 648 881 (float64 rows
    past 4 GiB).  Query i's 80 nearest rows lie above row 20 648 881.  The best of them, 4 q_i (exact in float32), has
    exact copies at rows 3 + i (the first split) and ndb - 1 - i (the last), so every list starts with a three-way tie
    across the whole index range: 3 + i, then the row above 2^24, then ndb - 1 - i.  All 8 queries against the oracle
    through the tensor-core filter (k 20), the FP32 filter (k 30) and the float64 kernel at 32 splits (k 60)."""
    torch = torch_cuda
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    nq, ndb, dim = 8, LARGE_NDB, 26
    g = torch.Generator(device="cuda")
    g.manual_seed(21)
    q = torch.randn((nq, dim), generator=g, device="cuda")
    db = torch.randn((ndb, dim), generator=g, device="cuda")
    best = []
    for i in range(nq):
        rows = LARGE_FROM + 1 + 40_000 * i + 500 * torch.arange(80, device="cuda")
        scale = torch.linspace(3.0, 1.0, 80, device="cuda")[:, None]
        db[rows] = q[i] * scale + 0.02 * torch.randn((80, dim), generator=g, device="cuda")
        db[rows[0]] = q[i] * 4.0                                        # no noise: the best row of query i
        db[3 + i] = db[rows[0]]
        db[ndb - 1 - i] = db[rows[0]]
        best.append(int(rows[0]))
    want_idx, want_sc = O.cosine_topk(q.cpu().numpy(), db.cpu().numpy(), 60, return_scores=True)
    for i in range(nq):                                                 # the data do what they claim
        assert want_idx[i, :3].tolist() == [3 + i, best[i], ndb - 1 - i], (i, want_idx[i, :4])
        assert want_sc[i, 0] == want_sc[i, 1] == want_sc[i, 2] > want_sc[i, 3], i
    assert (want_idx[:, 1:] > LARGE_FROM).all() and min(best) > 2**24
    for k in LARGE:
        idx, sc = R.cosine_topk(q, db, k, return_scores=True)
        assert np.array_equal(idx.cpu().numpy(), want_idx[:, :k]), k    # a stable order: top-k is a prefix of top-60
        assert np.array_equal(sc.cpu().numpy(), want_sc[:, :k]), k
        check_structure(torch, q, db, idx, sc, f"large k={k}")


# ---- GPU: cosine_similarity, hits@k, API edges ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nq,ndb,dim", [(0, 5, 26), (3, 0, 26), (1, 1, 1), (129, 257, 26), (40, 129, 33), (7, 300, 2048),
                                        (65_536, 3, 13)])
def test_cosine_similarity_bit_exact(torch_cuda, nq, ndb, dim):
    """The dense matrix equals, bit for bit, the oracle's scores of a full ranking (k = ndb) scattered back by index, in
    float32, float64 and torch; 65 536 queries take two launches."""
    torch = torch_cuda
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(nq * 31 + ndb * 7 + dim)
    q = rng.standard_normal((nq, dim), dtype=np.float32)
    db = rng.standard_normal((ndb, dim), dtype=np.float32)
    if ndb > 2:
        db[0] = 0.0
        db[-1] = db[1]
    want = np.zeros((nq, ndb))
    if nq and ndb:
        idx, sc = O.cosine_topk(q, db, ndb, return_scores=True)
        np.put_along_axis(want, idx.astype(np.int64), sc, axis=1)
    got = {"float32": R.cosine_similarity(q, db),
           "float64": R.cosine_similarity(q.astype(np.float64), db.astype(np.float64)),
           "torch": R.cosine_similarity(torch.as_tensor(q).cuda(), torch.as_tensor(db).cuda()).cpu().numpy()}
    for name, m in got.items():
        assert m.shape == (nq, ndb) and m.dtype == np.float64, name
        assert np.array_equal(m, want), name


@pytest.mark.gpu
@pytest.mark.parametrize("ndb,dim,k", [(5_000, 26, 20), (5_000, 26, 40), (5_000, 40, 10)])
def test_topk_scores_are_the_matrix(torch_cuda, ndb, dim, k):
    """cosine_topk's scores equal the dense matrix at the returned indices (one shape per kernel family)."""
    from dsp_final_b200 import retrieval as R

    rng = np.random.default_rng(ndb + dim + k)
    q = rng.standard_normal((300, dim), dtype=np.float32)
    db = rng.standard_normal((ndb, dim), dtype=np.float32)
    idx, sc = R.cosine_topk(q, db, k, return_scores=True)
    sims = R.cosine_similarity(q, db)
    assert np.array_equal(np.take_along_axis(sims, idx.astype(np.int64), axis=1), sc)


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [1, 255, 256, 257, 100_000])
def test_hits_at_k(torch_cuda, nq):
    """hits_at_k_device and hits_at_k against the oracle's count on a 20-wide index matrix, k < the row stride included;
    a k wider than the matrix raises."""
    torch = torch_cuda
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(nq)
    ndb = 3_000
    idx = rng.integers(0, ndb, (nq, 20)).astype(np.int32)
    tdb = rng.integers(0, 30, ndb).astype(np.int32)
    tq = rng.integers(0, 30, nq).astype(np.int32)
    ks = (1, 7, 20)
    dev = R.hits_at_k_device(torch.as_tensor(idx).cuda(), ks, torch.as_tensor(tdb).cuda(), torch.as_tensor(tq).cuda())
    assert dev.dtype == torch.int64 and dev.is_cuda
    want = [O.hits_at_k(idx, k, tdb, tq) for k in ks]
    assert dev.cpu().tolist() == want
    assert [R.hits_at_k(idx, k, tdb, tq) for k in ks] == want
    if nq > 1:
        assert 0 < want[0] < want[1] < want[2] < nq
    with pytest.raises(ValueError):
        R.hits_at_k_device(torch.as_tensor(idx).cuda(), [21], torch.as_tensor(tdb).cuda(), torch.as_tensor(tq).cuda())


@pytest.mark.gpu
def test_api_edges(torch_cuda):
    torch = torch_cuda
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(5)
    db = rng.standard_normal((300, 26), dtype=np.float32)
    q = rng.standard_normal((9, 26), dtype=np.float32)
    # no queries: empty (0, k) results
    idx, sc = R.cosine_topk(np.zeros((0, 26), np.float32), db, 5, return_scores=True)
    assert isinstance(idx, np.ndarray) and idx.shape == (0, 5) and sc.shape == (0, 5)
    idx, sc = R.cosine_topk(torch.zeros((0, 26), device="cuda"), torch.as_tensor(db).cuda(), 5, return_scores=True)
    assert idx.is_cuda and tuple(idx.shape) == (0, 5) and tuple(sc.shape) == (0, 5)
    # k > ndb is clipped to ndb columns
    idx, sc = R.cosine_topk(q, db[:10], 20, return_scores=True)
    want_idx, want_sc = O.cosine_topk(q, db[:10], 10, return_scores=True)
    assert np.array_equal(idx, want_idx) and np.array_equal(sc, want_sc)
    with pytest.raises(NotImplementedError):
        R.cosine_topk(q, db, MAX_K + 1)
    with pytest.raises(ValueError):
        R.cosine_topk(q, db, 0)
    # half, bfloat16 and integer tensors rank as the float64 of the same values
    for dt in (torch.float16, torch.bfloat16, torch.int32):
        if dt == torch.int32:
            qt, dbt = (torch.as_tensor(rng.integers(-40, 40, x.shape), dtype=dt).cuda() for x in (q, db))
        else:
            qt, dbt = torch.as_tensor(q).to(dt).cuda(), torch.as_tensor(db).to(dt).cuda()
        idx, sc = R.cosine_topk(qt, dbt, 24, return_scores=True)
        want_idx, want_sc = O.cosine_topk(qt.double().cpu().numpy(), dbt.double().cpu().numpy(), 24, return_scores=True)
        assert np.array_equal(idx.cpu().numpy(), want_idx) and np.array_equal(sc.cpu().numpy(), want_sc), dt
    # a NumPy query against a torch database comes back as NumPy
    idx = R.cosine_topk(q, torch.as_tensor(db).cuda(), 7)
    assert isinstance(idx, np.ndarray) and np.array_equal(idx, O.cosine_topk(q, db, 7))


@pytest.mark.gpu
def test_ranking_on_a_second_gpu(torch_cuda):
    """A tensor on cuda:1 is ranked on cuda:1."""
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(6)
    q = rng.standard_normal((300, 40), dtype=np.float32)
    db = rng.standard_normal((5_000, 40), dtype=np.float32)
    idx, sc = R.cosine_topk(torch.as_tensor(q).to("cuda:1"), torch.as_tensor(db).to("cuda:1"), 10, return_scores=True)
    assert idx.device == torch.device("cuda:1") and sc.device == torch.device("cuda:1")
    want_idx, want_sc = O.cosine_topk(q, db, 10, return_scores=True)
    assert np.array_equal(idx.cpu().numpy(), want_idx) and np.array_equal(sc.cpu().numpy(), want_sc)
