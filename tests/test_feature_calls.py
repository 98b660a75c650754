"""What a feature call runs around the feature kernel, and its scratch (csrc/feat_select.cuh: feat_steps,
feat_ws_carve), on the plans dspx_plan_create derives (plan_derive), over test_feature_space's SWEEP.  CPU only: the
library's own choice, exported by the replay library.

Every call kind of the device sweep -- device float32 on an even and an odd row stride and one sample off, PCM16 with and
without normalisation, embeddings alone, the NCHW store, host float32 and PCM16, ragged float32 and PCM16 with all
outputs and with embeddings alone -- against DESIGN's rules: which kernel path runs, whether PCM16 converts in the
kernel's loads or in a pass before it, whether embeddings fuse, whether a ragged batch runs clip by clip.  Then the
workspace of each call from every base offset 0..255: regions aligned, disjoint and as large as their step needs, inside
the sizes dspx_features_ragged_workspace, dspx_embeddings_workspace and dspx_features_pcm16_workspace report.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import pytest

from conftest import REPO  # noqa: F401  (puts the repository on sys.path)
from test_feature_space import IDS, SWEEP, Case, _struct, ragged_lengths

# W8Path (csrc/feat_warp8.cuh)
GENERIC, X2, X2_AL4, ALIGNED, SHARE, U4, PCM16_PATH, UNSUPPORTED = range(8)
F32, PCM16 = 0, 2
KERNEL_GENERIC, KERNEL_WARP8 = 1, 2
BASE = 1 << 40              # an aligned device address: only its alignment is read
N = 3                       # clips per batch, as in the device sweep
REGIONS = ("rpairs", "peaks", "eacc", "mfcc", "f32")


def embed_max_frames(n_mels: int) -> int:
    """w8_embed_max_frames: the most frames whose fixed-point embedding sums stay exact (DESIGN 4.1b)"""
    c = 2.0 * n_mels * 40.0
    return int(9223372036854775808.0 / (max(c * 2.0 ** 32, c * c * 2.0 ** 20) + 0.5)) - 1


def test_embed_frame_bound_matches_design():
    assert [embed_max_frames(m) for m in (40, 128, 256)] == [671_087, 83_885, 20_970]


@dataclass(frozen=True)
class Call:
    name: str
    dtype: int = F32
    normalize: int = 0
    base: int | None = BASE                 # None: the host pipeline's cudaMalloc'd chunk
    stride: int | None = None               # None: clip_len
    length: int | None = None               # None: case.length
    ragged: bool = False
    want_mfcc: bool = True
    want_embed: bool = True


@dataclass(frozen=True)
class Steps:
    path: int
    convert: bool
    peaks: bool
    fused: bool
    mfcc_scratch: bool
    per_clip: bool
    T: int


def calls(case: Case) -> list[Call]:
    n = case.length
    even, odd = n + (n & 1), (n | 1 if n & 1 else n + 1)
    out = [Call("device f32", stride=even), Call("odd stride", stride=odd, want_embed=False),
           Call("one sample off", base=BASE + 4, stride=even, want_embed=False),
           Call("embeddings alone", stride=even, want_mfcc=False),
           Call("nchw", stride=even, want_mfcc=False, want_embed=False),
           Call("host f32", base=None), Call("host f32 embeddings", base=None, want_mfcc=False)]
    for norm in (0, 1):
        out += [Call(f"device pcm16 normalize={norm}", PCM16, norm),
                Call(f"host pcm16 normalize={norm}", PCM16, norm, base=None),
                Call(f"host pcm16 embeddings normalize={norm}", PCM16, norm, base=None, want_mfcc=False)]
    for dtype, norm in ((F32, 0), (PCM16, 0), (PCM16, 1)):
        for alone in (False, True):
            out.append(Call(f"ragged dtype={dtype} normalize={norm} embeddings alone={alone}", dtype, norm, ragged=True,
                            want_mfcc=not alone))
    return out


@pytest.fixture(scope="module")
def lib():
    from dsp_final_b200 import build

    build.build_native()
    lib = C.CDLL(str(build.build_emu()))
    batch = [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int, C.c_int]
    lib.emu_feat_steps.argtypes = [C.c_void_p, *batch, C.c_void_p]
    lib.emu_feat_workspace.argtypes = [C.c_void_p, *batch, C.c_int64, C.c_void_p]
    lib.emu_plan_create.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
    lib.emu_plan_destroy.argtypes = [C.c_void_p]
    return lib


class Plan:
    """A plan of `case` as dspx_plan_create derives it (kernel AUTO, like the device sweep)"""

    def __init__(self, lib, case: Case):
        self.lib, self.case = lib, case
        kernel, handle = C.c_int(0), C.c_void_p()
        assert lib.emu_plan_create(C.byref(_struct(case, "auto")), C.byref(kernel), C.byref(handle)) == 0, case.id
        self.kernel, self.handle = kernel.value, handle

    def close(self):
        self.lib.emu_plan_destroy(self.handle)

    def _batch(self, call: Call):
        case = self.case
        length = call.length or case.length
        table = None
        if call.ragged:
            from dsp_final_b200.batch import ragged_layout

            lengths = [length] if call.length else ragged_lengths(case)
            _, table, _ = ragged_layout(lengths, case.cfg(), np.int16 if call.dtype == PCM16 else np.float32)
        n = len(table) if call.ragged else (1 if call.length else N)
        args = (call.base, call.dtype, call.normalize, n, length, call.stride or length,
                table.ctypes.data if call.ragged else None, int(call.want_mfcc), int(call.want_embed))
        return args, table

    def steps(self, call: Call) -> Steps:
        args, _ = self._batch(call)
        out = (C.c_int64 * 7)()
        assert self.lib.emu_feat_steps(self.handle, *args, out) == 0
        v = list(out)
        return Steps(v[0], *(bool(x) for x in v[1:6]), v[6])

    def workspace(self, call: Call) -> tuple[list, np.ndarray | None]:
        """[(region offsets, size) from base offsets 0..255], the ragged table"""
        args, table = self._batch(call)
        out = (C.c_int64 * 6)()
        res = []
        for offset in range(256):
            assert self.lib.emu_feat_workspace(self.handle, *args, offset, out) == 0
            res.append((dict(zip(REGIONS, list(out)[:5])), out[5]))
        return res, table


@pytest.fixture(scope="module")
def plans(lib):
    ps = {case.id: Plan(lib, case) for case in SWEEP}
    yield ps
    for p in ps.values():
        p.close()


def kind(case: Case) -> str:
    return case.shape if isinstance(case.shape, str) else "warp8"


def pow2(case: Case) -> int:
    return 1 << ((case.n_fft or case.fl) - 1).bit_length()


def on_grid(case: Case) -> bool:
    """every frame of an 8-byte aligned, even-stride row on the 8-byte grid and a whole transform long"""
    return case.fl == pow2(case) and case.hop % 2 == 0


def f32_path(case: Case, base: int, stride: int) -> int:
    """DESIGN 4.1 / 4.1c: the kernel of float32 rows on each kind of plan"""
    if kind(case) == "generic":
        return GENERIC
    if kind(case) == "x2":
        al4 = case.fl >= pow2(case) and case.hop % 4 == 0 and stride % 4 == 0 and base % 16 == 0
        return X2_AL4 if al4 else X2
    if not (on_grid(case) and stride % 2 == 0 and base % 8 == 0):
        return U4
    return SHARE if 2 * case.hop == pow2(case) and pow2(case) != 2048 else ALIGNED


def expected(case: Case, call: Call, T: int) -> Steps:
    """DESIGN's rules for one call"""
    warp8 = kind(case) == "warp8"
    length = call.length or case.length
    base = BASE if call.base is None else call.base
    alone = call.want_embed and not call.want_mfcc
    if call.ragged:
        per_clip = not warp8                            # generic and n_fft 4096 plans have no ragged kernel
        pcm_in_kernel = call.dtype == PCM16 and warp8
        # float32 clips of a ragged batch start on the 8-byte grid (dspx_ragged_layout)
        path = UNSUPPORTED if per_clip else PCM16_PATH if pcm_in_kernel else f32_path(case, BASE, 0)
    else:
        per_clip = False
        pcm_in_kernel = call.dtype == PCM16 and warp8
        stride = length if call.dtype == PCM16 and not pcm_in_kernel else (call.stride or length)
        path = PCM16_PATH if pcm_in_kernel else f32_path(case, base if call.dtype == F32 else BASE, stride)
    fused = alone and call.dtype == F32 and warp8 and path in (SHARE, ALIGNED) and T <= embed_max_frames(case.n_mels)
    return Steps(path, call.dtype == PCM16 and not pcm_in_kernel, pcm_in_kernel and bool(call.normalize), fused,
                 alone and not fused, per_clip, T)


@pytest.mark.parametrize("case", SWEEP, ids=IDS)
def test_steps_follow_design(plans, case):
    """PCM16 on warp8 plans at n_fft 512 / 1024 / 2048 converts in the kernel's loads, with peaks iff normalised;
    elsewhere host and ragged calls convert first and dspx_features_pcm16 refuses.  Embeddings alone fuse on aligned
    float32 frames within the frame bound, else host and ragged calls take MFCC scratch and dspx_embeddings refuses.
    Ragged batches on generic and n_fft 4096 plans run clip by clip."""
    plan = plans[case.id]
    assert plan.kernel == (KERNEL_GENERIC if case.shape == "generic" else KERNEL_WARP8), case.id
    frames = [1 + (n - case.fl) // case.hop for n in ragged_lengths(case)]
    for call in calls(case):
        got = plan.steps(call)
        T = max(frames) if call.ragged else 1 + (case.length - case.fl) // case.hop
        assert got == expected(case, call, T), (case.id, call.name, got)
    if kind(case) == "warp8" and on_grid(case):
        # both sides of the frame bound of the fused sums, on the device, the host and in a ragged batch
        bound = embed_max_frames(case.n_mels)
        for frames, fused in ((bound, True), (bound + 1, False)):
            length = case.fl + (frames - 1) * case.hop
            for call in (Call("device", length=length, want_mfcc=False), Call("host", base=None, length=length, want_mfcc=False),
                         Call("ragged", length=length, ragged=True, want_mfcc=False)):
                got = plan.steps(call)
                assert (got.fused, got.mfcc_scratch, got.T) == (fused, not fused, frames), (case.id, call.name, frames)


def align256(x: int) -> int:
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("case", SWEEP, ids=IDS)
def test_workspace_regions(plans, case):
    plan = plans[case.id]
    C_ = case.n_mfcc
    for call in calls(case):
        s = plan.steps(call)
        res, table = plan.workspace(call)
        n = len(table) if call.ragged else N
        frames = int(table[-1, 3] + table[-1, 2]) if call.ragged else N * s.T
        samples = int(table[:, 1].max()) if call.ragged else N * case.length
        need = {"rpairs": (n + 1) * 4 if call.ragged and not s.per_clip else 0, "peaks": n * 4 if s.peaks else 0,
                "eacc": n * 2 * C_ * 8 if s.fused else 0, "mfcc": frames * C_ * 4 if s.mfcc_scratch else 0,
                "f32": samples * 4 if s.convert else 0}
        for offset, (regions, total) in enumerate(res):
            what = (case.id, call.name, offset)
            for r in REGIONS:
                assert (regions[r] >= 0) == (need[r] > 0), (*what, r, regions[r], need[r])
                if need[r]:
                    assert (offset + regions[r]) % 256 == 0, (*what, r)          # aligned
            used = sorted((regions[r], need[r]) for r in REGIONS if need[r])
            for (a, na), (b, _) in zip(used, used[1:]):
                assert a + na <= b, what                                         # disjoint
            assert all(o + nb <= total for o, nb in used), what                  # inside the carve's size
            if call.ragged:                                                      # dspx_features_ragged_workspace
                assert total == sum(align256(v) for v in need.values()) + 256, what
            if call.name == "embeddings alone" and s.fused:                      # dspx_embeddings_workspace
                assert regions["eacc"] + need["eacc"] <= n * 2 * C_ * 8 + 256, what
            if call.name.startswith("device pcm16") and s.peaks:                 # dspx_features_pcm16_workspace
                assert regions["peaks"] + need["peaks"] <= n * 4 + 256, what
