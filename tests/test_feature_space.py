"""Feature kernels across the configuration space, against the float64 oracle (oracle/dsp_oracle.c).

SWEEP is an explicit list of configurations: sample rates 8-96 kHz, n_fft 512 / 1024 / 2048 / 4096 and two
generic-only transforms, frames shorter than the transform, even / odd / half-transform hops and hops longer than the
frame, 20-256 mel filters, 1-128 coefficients (across the DCT block edges 16/17, 32/33, 64/65), narrow bands, every
window with pre-emphasis 0, 0.5 and 0.97, odd and even frame counts.  Every configuration names the CTA shape its warp8
plan launches (warps per CTA); the shapes follow from the shared memory of the plan's tables (warp8_shapes).

CPU: the replay of the warp8 and generic phase functions (libdspx_emu.so) over the whole list -- feature mode on
aligned and odd row strides, STFT mode with and without pre-emphasis, the RAGGED mapping -- and the CTA shape of every
plan.  GPU (-m gpu): every entry point that applies to a configuration (device float32 on each path warp8_select can
take, the generic kernel, host buffers, PCM16, ragged batches, fused embeddings, STFT, the NCHW store, the plan's
tables), the kernels and block sizes the sweep launched, and clips long enough to overflow 64-bit fused embedding sums.

One tolerance model holds for every path (see the check_* functions): MFCC per coefficient, log-mel per frame within 60
dB of the frame's peak and by a round-off model below, embeddings mean and std per coefficient, STFT per frame.
"""
from __future__ import annotations

import ctypes as C
import json
from dataclasses import dataclass

import numpy as np
import pytest

from conftest import REPO  # noqa: F401  (puts the repository on sys.path)

TOL = 1e-4


@dataclass(frozen=True)
class Case:
    sr: int
    fl: int
    hop: int
    n_fft: int | None
    n_mels: int
    n_mfcc: int
    f_min: float
    f_max: float | None
    pre: float
    window: str
    frames: int                 # frames of the batch's clips (odd: the last frame pair is half empty)
    shape: int | str            # warps per CTA of the plan's feat_warp8_kernel, or "x2" / "generic" (see SWEEP)

    @property
    def id(self) -> str:
        band = "" if (self.f_min, self.f_max) == (0.0, None) else f"-{self.f_min:g}-{self.f_max or 'ny'}"
        nf = f"/{self.n_fft}" if self.n_fft else ""
        return (f"{self.sr}-{self.fl}{nf}-h{self.hop}-m{self.n_mels}-c{self.n_mfcc}{band}-{self.window}"
                f"-p{self.pre:g}-t{self.frames}")

    @property
    def length(self) -> int:
        return self.fl + (self.frames - 1) * self.hop + min(self.hop - 1, 7)

    def cfg(self):
        from dsp_final_b200.dsp.mfcc import MfccConfig

        return MfccConfig(self.sr, self.fl, self.hop, self.n_fft, self.n_mels, self.n_mfcc, self.f_min, self.f_max,
                          self.pre, self.window)

    def ocfg(self):
        from oracle import oracle as O

        return O.OracleConfig(self.sr, self.fl, self.hop, self.n_fft, self.n_mels, self.n_mfcc, self.f_min, self.f_max,
                              self.pre, self.window)


def _c(sr, fl, hop, n_mels, n_mfcc, pre, window, frames, shape, n_fft=None, f_min=0.0, f_max=None):
    return Case(sr, fl, hop, n_fft, n_mels, n_mfcc, f_min, f_max, pre, window, frames, shape)


# Paths (float32, contiguous clips of even length): SHARE = hop n_fft / 2 at radix 4 / 8, ALIGNED = other even hops
# with frame_length = n_fft, U4 = odd hops or frames shorter than n_fft.  Every case also runs U4 on an odd row stride
# and one sample off, PCM16, RAGGED and (aligned ones) the fused embeddings.  `shape`: the warps per CTA of the plan's
# feat_warp8_kernel -- 20 / 12 / 8 at radix 4 / 8, 10 / 8 at radix 16 (w8_launch_cfg, from the plan's shared memory)
# -- or "x2" (feat_warp8_x2_kernel) or "generic" (feat_generic_kernel).
SWEEP = [
    # radix 4 (n_fft 512)
    _c(16000, 512, 256, 40, 13, 0.97, "hann", 11, 20),                        # SHARE
    _c(8000, 512, 256, 20, 1, 0.0, "hamming", 10, 20),                        # SHARE, no pre-emphasis, one coefficient
    _c(22050, 512, 160, 128, 16, 0.5, "rect", 13, 12, f_min=20.0, f_max=8000.0),     # ALIGNED
    _c(16000, 512, 128, 128, 128, 0.0, "hann", 12, 12),                       # ALIGNED, 128 coefficients
    _c(16000, 400, 160, 64, 17, 0.97, "hann", 14, 20, n_fft=512),             # U4: 400-sample frames in 512
    _c(32000, 512, 255, 256, 32, 0.97, "hamming", 9, 8),                      # U4 (odd hop)
    _c(48000, 512, 600, 200, 33, 0.0, "hann", 8, 20, f_min=300.0, f_max=3400.0),     # hop > frame, narrow band
    _c(96000, 512, 128, 96, 65, 0.5, "hann", 16, 12),                         # ALIGNED, 65 coefficients
    _c(22050, 512, 256, 256, 20, 0.5, "hamming", 9, 8),                       # SHARE
    _c(16000, 512, 384, 256, 32, 0.97, "rect", 10, 20, f_min=1000.0, f_max=1100.0),  # 1000-1100 Hz in 256 filters
    _c(44100, 512, 1001, 80, 32, 0.97, "rect", 7, 20),                        # U4: odd hop > frame
    # radix 8 (n_fft 1024)
    _c(44100, 1024, 512, 40, 13, 0.97, "hann", 12, 20),                       # SHARE (the headline configuration)
    _c(44100, 1024, 441, 40, 20, 0.97, "hann", 11, 20),                       # U4 (odd hop)
    _c(16000, 1000, 400, 80, 32, 0.97, "hamming", 10, 12, n_fft=1024, f_min=50.0, f_max=7600.0),   # U4: short frames
    _c(22050, 1024, 256, 128, 128, 0.0, "rect", 15, 8),                       # ALIGNED, no pre-emphasis
    _c(48000, 1024, 512, 256, 13, 0.5, "hann", 9, 8),                         # SHARE
    _c(96000, 1024, 2000, 64, 64, 0.97, "hamming", 7, 12),                    # hop > frame
    _c(32000, 1024, 320, 128, 33, 0.97, "hann", 12, 12, f_min=300.0, f_max=3400.0),  # ALIGNED, narrow band
    _c(8000, 1024, 512, 20, 17, 0.0, "hann", 10, 20),                         # SHARE, no pre-emphasis, 17 coefficients
    _c(96000, 1024, 96, 64, 13, 0.5, "rect", 13, 8),                          # ALIGNED, two 8-warp CTAs per SM
    _c(22050, 1024, 221, 200, 64, 0.97, "hamming", 11, 8),                    # U4 (odd hop)
    # radix 16 (n_fft 2048; rows are never shared)
    _c(44100, 2048, 512, 40, 13, 0.97, "hann", 10, 10),                       # ALIGNED
    _c(48000, 2048, 1024, 128, 64, 0.0, "hann", 9, 8),                        # ALIGNED, no pre-emphasis
    _c(22050, 2048, 441, 64, 33, 0.5, "hamming", 11, 10),                     # U4 (odd hop)
    _c(96000, 2048, 960, 200, 13, 0.97, "rect", 8, 8, f_min=20.0, f_max=20000.0),   # ALIGNED
    _c(16000, 2048, 2560, 160, 32, 0.97, "rect", 8, 8, f_min=20.0),           # hop > frame
    _c(8000, 2048, 200, 20, 16, 0.0, "hamming", 12, 10),                      # ALIGNED, no pre-emphasis
    _c(32000, 1500, 640, 96, 64, 0.97, "hann", 9, 8, n_fft=2048),             # U4: short frames
    _c(44100, 2048, 1023, 128, 20, 0.5, "rect", 8, 8),                        # U4 (odd hop)
    # n_fft 4096 (feat_warp8_x2_kernel): 16-byte loads (AL4) or not
    _c(44100, 4096, 1024, 40, 13, 0.97, "hann", 8, "x2"),                     # AL4
    _c(16000, 4096, 1001, 128, 13, 0.5, "hamming", 9, "x2"),                  # odd hop: 8-byte loads
    _c(96000, 4000, 1000, 64, 16, 0.0, "rect", 7, "x2", n_fft=4096),          # frames shorter than 4096
    _c(48000, 4096, 2048, 20, 1, 0.0, "hann", 6, "x2"),                       # AL4, no pre-emphasis
    # warp8 tables too large for shared memory: the generic kernel
    _c(32000, 512, 255, 256, 128, 0.97, "hamming", 9, "generic"),
    _c(48000, 2048, 1024, 128, 128, 0.0, "hann", 9, "generic"),
    _c(96000, 4000, 1000, 256, 128, 0.0, "rect", 7, "generic", n_fft=4096),
    # the generic kernel only (n_fft 256, 8192)
    _c(16000, 256, 128, 20, 13, 0.97, "hann", 17, "generic"),
    _c(44100, 8192, 2048, 128, 20, 0.5, "hamming", 6, "generic"),
    _c(8000, 200, 80, 40, 13, 0.0, "rect", 21, "generic", n_fft=256),
]
IDS = [c.id for c in SWEEP]


# ---- inputs and references ------------------------------------------------------------------------------------------
def clips(case: Case) -> np.ndarray:
    """[3, length] float32: a synthetic clip, a quiet one whose second half is digital silence, and silence."""
    from dsp_final_b200 import synth

    n = case.length
    x = synth.host_clips(2, seed=case.sr + case.fl + case.hop, length=n, sample_rate=case.sr)
    x[1] *= 1e-3
    x[1, n // 2:] = 0.0
    return np.concatenate((x, np.zeros((1, n), np.float32)))


def pcm16(x: np.ndarray) -> np.ndarray:
    return (x * 20000).astype(np.int16)


def pcm16_reference_input(p: np.ndarray, normalize: bool) -> np.ndarray:
    """load_audio (int16 / 32768) + normalize_audio (x / max|x| unless silent) in float32 NumPy."""
    x = p.astype(np.float32) / np.float32(32768.0)
    if normalize:
        peak = np.max(np.abs(x), axis=1, keepdims=True)
        x = np.where(peak > 0, x / np.where(peak > 0, peak, 1), x).astype(np.float32)
    return x


def ragged_lengths(case: Case) -> list[int]:
    """three clips: the batch's length, one frame, and two frames more plus an odd remainder"""
    return [case.length, case.fl, case.length + 2 * case.hop + 3]


def ragged_clips(case: Case) -> list[np.ndarray]:
    from dsp_final_b200 import synth

    return [synth.host_clip(i, seed=7 * case.fl + case.hop, length=n, sample_rate=case.sr)
            for i, n in enumerate(ragged_lengths(case))]


def stft_reference(x: np.ndarray, case: Case, pre: float) -> np.ndarray:
    from oracle import oracle as O

    y = x.astype(np.float64)
    if pre > 0:
        y[1:] -= pre * x[:-1].astype(np.float64)
    return O.stft(y, case.fl, case.hop, case.window, case.n_fft)


# ---- the tolerance model --------------------------------------------------------------------------------------------
def check_mfcc(got, ref, what):
    """Per clip and coefficient: max_t |got - ref| <= TOL * max_t |ref[:, c]|, plus a floor for coefficients that are
    identically zero (silence): the float32 round-off of a DCT row sum over n_mels log-mel values, 2^-20 |C0|."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    for b in range(ref.shape[0]):
        err = np.max(np.abs(got[b] - ref[b]), axis=0)
        bound = TOL * np.max(np.abs(ref[b]), axis=0) + 2.0 ** -20 * np.max(np.abs(ref[b][:, 0]))
        bad = np.nonzero(~(err <= bound))[0]
        assert bad.size == 0, (f"{what}: clip {b} coefficients {bad.tolist()[:8]}: error "
                               f"{(err[bad] / np.maximum(np.max(np.abs(ref[b]), axis=0)[bad], 1e-30)).tolist()[:8]} "
                               "of the column maximum")


def check_logmel(got, ref, what):
    """Per clip: cells within 60 dB of their frame's peak band meet TOL * max|ref|; weaker cells carry the FP32
    round-off of the transform, which is relative to the frame's strongest bins: error x relative amplitude < 3e-5."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    for b in range(ref.shape[0]):
        peak = ref[b].max(axis=1, keepdims=True)
        strong = ref[b] >= peak - np.log(1e6)
        err = np.abs(got[b] - ref[b])
        assert np.all(err[strong] <= TOL * np.max(np.abs(ref[b]))), (what, b, float(err[strong].max()))
        level = np.exp(0.5 * (ref[b] - peak))
        assert float((err * level).max()) < 3e-5, (what, b, float((err * level).max()))
        assert float(err.max()) < 0.1, (what, b, float(err.max()))


def check_embed(got, ref, mfcc_ref, what):
    """Mean and std per coefficient, each against the oracle's: |d mean| <= TOL * rms_t(C) (the scale of the values
    averaged), |d std| <= TOL * std; floors: the MFCC floor for the mean, and for std the resolution of the fixed-point
    sums, whose E[x^2] - mean^2 is good to 2^-20 + 2^-30 |mean| (a constant coefficient has std 0)."""
    got, ref, mfcc_ref = (np.asarray(a, np.float64) for a in (got, ref, mfcc_ref))
    n = ref.shape[1] // 2
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    for b in range(ref.shape[0]):
        mean, std = ref[b, :n], ref[b, n:]
        floor = 2.0 ** -20 * np.max(np.abs(mfcc_ref[b][:, 0]))
        d_mean = np.abs(got[b, :n] - mean)
        bad = np.nonzero(~(d_mean <= TOL * np.sqrt(mean ** 2 + std ** 2) + floor))[0]
        assert bad.size == 0, (f"{what}: clip {b} mean of coefficients {bad.tolist()[:8]}", d_mean[bad][:8], mean[bad][:8])
        g = got[b, n:]
        d_var = np.abs(g * g - std * std)
        bad = np.nonzero(~(d_var <= 2 * TOL * std * std + 2.0 ** -20 + 2.0 ** -30 * np.abs(mean)))[0]
        assert bad.size == 0, (f"{what}: clip {b} std of coefficients {bad.tolist()[:8]}", g[bad][:8], std[bad][:8])


def check_stft(got, ref, what):
    """Per frame: ||got - ref|| <= TOL * ||ref|| (a silent frame must come out exactly zero)."""
    got, ref = np.asarray(got, np.complex128), np.asarray(ref, np.complex128)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err = np.linalg.norm(got - ref, axis=-1)
    norm = np.linalg.norm(ref, axis=-1)
    bad = np.argwhere(~(err <= TOL * norm))
    assert bad.size == 0, (what, bad[:4].tolist(), (err / np.maximum(norm, 1e-30))[tuple(bad[0])])


def oracle_features(x, case: Case) -> dict:
    from oracle import oracle as O

    return O.features_batch(x, case.ocfg(), want=("mfcc", "log_mel", "embed"))


def check_features(got: dict, ref: dict, what: str) -> None:
    if "mfcc" in got:
        check_mfcc(got["mfcc"], ref["mfcc"], what + " mfcc")
    if "log_mel" in got:
        check_logmel(got["log_mel"], ref["log_mel"], what + " log-mel")
    if "embed" in got:
        check_embed(got["embed"], ref["embed"], ref["mfcc"], what + " embed")


# ---- CPU: the replay of the phase functions over the same list -----------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    from dsp_final_b200 import build

    build.build_native()
    return C.CDLL(str(build.build_emu()))


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _struct(case: Case, kernel: str = "warp8"):
    from dsp_final_b200.plan import config_key, config_struct

    return config_struct(config_key(case.cfg()), kernel)


def emu_shapes(emu, case: Case):
    """(rc, {table bytes, shared memory of the 8 / 20 / 12 / 10-warp CTAs, 8-warp CTAs per SM, radix, x2})"""
    out = (C.c_int64 * 8)()
    rc = emu.emu_warp8_shapes(C.byref(_struct(case)), out)
    keys = ("tables", "smem8", "smem20", "smem12", "smem10", "ctas_per_sm", "radix", "x2")
    return rc, dict(zip(keys, list(out)))


def device_shape(rc: int, s: dict):
    """What the library launches for a plan: warp8_supported and tables that fit shared memory (warp8_prepare), then
    the widest CTA whose shared memory the plan found room for (w8_launch_cfg); feat_warp8_x2_kernel at n_fft 4096"""
    if rc != 0 or s["smem8"] > 227 * 1024:
        return "generic"
    if s["x2"]:
        return "x2"
    if s["radix"] != 16:
        return 20 if s["smem20"] else (12 if s["smem12"] else 8)
    return 10 if s["smem10"] else 8


def _strided(x: np.ndarray, odd: bool) -> np.ndarray:
    """x in a buffer whose row stride is even (frames on the 8-byte grid when the hop is even) or odd"""
    n = x.shape[1]
    stride = n + (n & 1) if not odd else n | 1 if n & 1 else n + 1
    buf = np.zeros((x.shape[0], stride), np.float32)
    buf[:, :n] = x
    return buf


def emu_features(emu, case: Case, x: np.ndarray, odd_stride: bool):
    buf = _strided(x, odd_stride)
    b, n = x.shape
    t = 1 + (n - case.fl) // case.hop
    lm = np.zeros((b, t, case.n_mels), np.float32)
    mf = np.zeros((b, t, case.n_mfcc), np.float32)
    rc = emu.emu_features_warp8(C.byref(_struct(case)), _fp(buf), C.c_int64(b), C.c_int64(n), C.c_int64(buf.shape[1]),
                                _fp(lm), _fp(mf), None, 0)
    return rc, {"mfcc": mf, "log_mel": lm}


def emu_generic(emu, case: Case, x: np.ndarray):
    b, n = x.shape
    t = 1 + (n - case.fl) // case.hop
    lm = np.zeros((b, t, case.n_mels), np.float32)
    mf = np.zeros((b, t, case.n_mfcc), np.float32)
    rc = emu.emu_features_generic(C.byref(_struct(case, "generic")), _fp(x), C.c_int64(b), C.c_int64(n), C.c_int64(n),
                                  0, 0, _fp(lm), _fp(mf), None, 0)
    assert rc == 0, (case.id, rc)
    return {"mfcc": mf, "log_mel": lm}


def emu_stft(emu, case: Case, x: np.ndarray, pre: bool):
    """(rc, [B, T, bins] complex) of the warp8 STFT mode, or of the generic kernel where the plan has no warp8 STFT"""
    b, n = x.shape
    t = 1 + (n - case.fl) // case.hop
    p = 1 << ((case.n_fft or case.fl) - 1).bit_length()
    out = np.zeros((b, t, p // 2 + 1, 2), np.float32)
    buf = _strided(x, False)
    rc = emu.emu_features_warp8(C.byref(_struct(case)), _fp(buf), C.c_int64(b), C.c_int64(n), C.c_int64(buf.shape[1]),
                                None, None, _fp(out), int(pre))
    if rc != 0:
        rc = emu.emu_features_generic(C.byref(_struct(case, "generic")), _fp(x), C.c_int64(b), C.c_int64(n),
                                      C.c_int64(n), 1, int(pre), None, None, _fp(out), 0)
    return rc, out[..., 0] + 1j * out[..., 1]


def emu_ragged(emu, case: Case, xs: list):
    from dsp_final_b200.batch import ragged_layout

    starts, table, total = ragged_layout([len(x) for x in xs], case.cfg())
    flat = np.zeros(int(starts[-1] + len(xs[-1])), np.float32)
    for s, x in zip(starts, xs):
        flat[s:s + len(x)] = x
    lm = np.zeros((total, case.n_mels), np.float32)
    mf = np.zeros((total, case.n_mfcc), np.float32)
    rc = emu.emu_features_warp8_ragged(C.byref(_struct(case)), C.c_void_p(flat.ctypes.data),
                                       C.c_void_p(table.ctypes.data), C.c_int64(len(xs)), C.c_void_p(lm.ctypes.data),
                                       C.c_void_p(mf.ctypes.data))
    return rc, table, lm, mf


def test_sweep_reaches_every_cta_shape(emu):
    """Every case's plan launches the kernel and CTA shape its entry names, and together they reach 20, 12 and 8 warps
    at radix 4 and 8 and 10 and 8 at radix 16."""
    seen = set()
    for case in SWEEP:
        rc, s = emu_shapes(emu, case)
        assert device_shape(rc, s) == case.shape, (case.id, rc, s)
        if isinstance(case.shape, int):
            seen.add((s["radix"], case.shape))
    assert seen == {(4, 20), (4, 12), (4, 8), (8, 20), (8, 12), (8, 8), (16, 10), (16, 8)}, sorted(seen)


@pytest.mark.parametrize("case", SWEEP, ids=IDS)
def test_replay_matches_oracle(emu, case):
    """The CPU replay of the kernel a configuration runs -- feature mode on even and odd row strides, STFT mode with
    and without pre-emphasis, the RAGGED mapping -- against the oracle under the sweep's tolerance model."""
    from oracle import oracle as O

    x = clips(case)
    ref = oracle_features(x, case)
    if case.shape == "generic":
        check_features(emu_generic(emu, case, x), ref, f"{case.id} generic replay")
    else:
        for odd in (False, True):
            rc, got = emu_features(emu, case, x, odd)
            assert rc == 0, (case.id, odd, rc)
            check_features(got, ref, f"{case.id} warp8 replay, {'odd' if odd else 'even'} row stride")
        xs = ragged_clips(case)
        rc, table, lm, mf = emu_ragged(emu, case, xs)
        assert (rc == 0) == (case.shape != "x2"), (case.id, rc)          # n_fft 4096 has no RAGGED variant
        for i, xi in enumerate(xs if rc == 0 else []):
            rows = slice(table[i, 3], table[i, 3] + table[i, 2])
            r = O.features_batch(xi[None], case.ocfg(), want=("mfcc", "log_mel"))
            check_features({"mfcc": mf[None, rows], "log_mel": lm[None, rows]}, r, f"{case.id} ragged replay clip {i}")
    for pre in (False, True):
        rc, st = emu_stft(emu, case, x[:2], pre)
        assert rc == 0, (case.id, pre, rc)
        for b in range(2):
            check_stft(st[b], stft_reference(x[b], case, case.pre if pre else 0.0), f"{case.id} stft pre={pre} clip {b}")


def test_replay_sweep_covers_the_issue_axes():
    """The list itself: every sample rate, window x pre-emphasis pair and DCT block edge is in it."""
    assert {c.sr for c in SWEEP} == {8000, 16000, 22050, 32000, 44100, 48000, 96000}
    assert {(c.window, c.pre) for c in SWEEP} == {(w, p) for w in ("hann", "hamming", "rect") for p in (0.0, 0.5, 0.97)}
    assert {1, 16, 17, 32, 33, 64, 65, 128} <= {c.n_mfcc for c in SWEEP}
    assert {20, 128, 200, 256} <= {c.n_mels for c in SWEEP}
    assert {c.frames % 2 for c in SWEEP} == {0, 1}


# ---- GPU: every entry point over the same list ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def _dev_rows(torch, x: np.ndarray, odd_stride: bool = False, offset: int = 0):
    """x on the device as a [B, n] view of rows of even (odd) stride whose first sample sits `offset` samples into
    the allocation (8-byte aligned at offset 0)"""
    b, n = x.shape
    stride = _strided(x, odd_stride).shape[1]
    flat = torch.zeros(b * stride + offset, dtype=torch.float32, device="cuda")
    view = torch.as_strided(flat, (b, n), (stride, 1), offset)
    view.copy_(torch.as_tensor(x))
    return view


def _np(d: dict) -> dict:
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)) for k, v in d.items()}


ALL = ("log_mel", "mfcc", "embed")


def run_device(torch, case: Case) -> dict:
    """Every entry point that applies to `case`, outputs copied back to NumPy."""
    from dsp_final_b200.batch import features_batch, features_ragged, log_mel_nchw, stft_batch
    from dsp_final_b200.plan import get_plan

    cfg = case.cfg()
    x = clips(case)
    even = _dev_rows(torch, x)
    r = {"plan_kernel": get_plan(cfg, 0).kernel}
    r["f32"] = _np(features_batch(even, cfg, ALL))
    r["odd stride"] = _np(features_batch(_dev_rows(torch, x, odd_stride=True), cfg, ("log_mel", "mfcc")))
    r["one sample off"] = _np(features_batch(_dev_rows(torch, x, offset=1), cfg, ("log_mel", "mfcc")))
    r["generic"] = _np(features_batch(even, cfg, ALL, kernel="generic"))
    r["host"] = _np(features_batch(x, cfg, ALL))
    r["embed device"] = features_batch(even, cfg, ("embed",))["embed"].cpu().numpy()
    r["embed host"] = features_batch(x, cfg, ("embed",))["embed"]
    p = pcm16(x)
    for norm in (True, False):
        r[f"pcm16 device normalize={norm}"] = _np(features_batch(torch.as_tensor(p).cuda(), cfg, ALL, normalize=norm))
        r[f"pcm16 host normalize={norm}"] = _np(features_batch(p, cfg, ALL, normalize=norm))
    xs = ragged_clips(case)
    xs_dev = [torch.as_tensor(v).cuda() for v in xs]
    r["ragged"] = _np(features_ragged(xs_dev, cfg, ALL))
    r["ragged embed"] = features_ragged(xs_dev, cfg, ("embed",))["embed"].cpu().numpy()
    r["alone"] = [_np(features_batch(_dev_rows(torch, v[None]), cfg, ALL)) for v in xs]
    r["alone embed"] = [features_batch(_dev_rows(torch, v[None]), cfg, ("embed",))["embed"].cpu().numpy() for v in xs]
    for pre in (0.0, case.pre or 0.97):
        r[f"stft pre={pre:g}"] = stft_batch(even[:2], case.fl, case.hop, case.window, case.n_fft,
                                            pre_emphasis=pre).cpu().numpy()
    r["nchw"] = log_mel_nchw(even, cfg).cpu().numpy()
    plan = get_plan(cfg, 0)
    r["tables"] = {k: plan.read_table(k) for k in ("window", "fbank", "dct2")}
    r["n_fft_pow2"] = plan.n_fft
    return r


@pytest.fixture(scope="module")
def device_sweep(torch_cuda, tmp_path_factory):
    """The whole sweep on the device under torch.profiler: ({case id: outputs or the exception}, kernel launches)."""
    torch = torch_cuda
    from torch.profiler import ProfilerActivity, profile

    results = {}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case in SWEEP:
            try:
                results[case.id] = run_device(torch, case)
            except Exception as e:                      # reported by the case's own test
                results[case.id] = e
        torch.cuda.synchronize()
    path = tmp_path_factory.mktemp("sweep") / "trace.json"
    prof.export_chrome_trace(str(path))
    events = json.loads(path.read_text())["traceEvents"]
    launches = [(e["name"], tuple(e["args"]["block"])) for e in events if e.get("cat") == "kernel"]
    return results, launches


@pytest.mark.gpu
@pytest.mark.parametrize("case", SWEEP, ids=IDS)
def test_device_matches_oracle(device_sweep, case):
    from dsp_final_b200.dsp.mfcc import _dct_basis, mel_filterbank
    from dsp_final_b200.dsp.stft import _get_window

    r = device_sweep[0][case.id]
    if isinstance(r, Exception):
        raise r
    assert r["plan_kernel"] == ("generic" if case.shape == "generic" else "warp8"), (case.id, r["plan_kernel"])
    x = clips(case)
    ref = oracle_features(x, case)
    for name in ("f32", "odd stride", "one sample off", "generic", "host"):
        check_features(r[name], ref, f"{case.id} {name}")
    for name in ("embed device", "embed host"):
        check_embed(r[name], ref["embed"], ref["mfcc"], f"{case.id} {name}")
    p = pcm16(x)
    for norm in (True, False):
        pref = oracle_features(pcm16_reference_input(p, norm), case)
        for where in ("device", "host"):
            check_features(r[f"pcm16 {where} normalize={norm}"], pref, f"{case.id} pcm16 {where} normalize={norm}")
    # ragged: every clip bit-identical to the clip alone, and the oracle's values
    xs = ragged_clips(case)
    off = r["ragged"]["frame_offsets"]
    for i, v in enumerate(xs):
        rows = slice(int(off[i]), int(off[i + 1]))
        alone = r["alone"][i]
        for k in ("log_mel", "mfcc"):
            assert np.array_equal(r["ragged"][k][rows], alone[k][0]), (case.id, "ragged", k, i)
        assert np.array_equal(r["ragged"]["embed"][i], alone["embed"][0]), (case.id, "ragged embed", i)
        assert np.array_equal(r["ragged embed"][i], r["alone embed"][i][0]), (case.id, "ragged fused embed", i)
        vref = oracle_features(v[None], case)
        check_features({k: alone[k] for k in ALL}, vref, f"{case.id} ragged clip {i}")
        check_embed(r["alone embed"][i], vref["embed"], vref["mfcc"], f"{case.id} ragged clip {i} embed alone")
    for pre in (0.0, case.pre or 0.97):
        st = r[f"stft pre={pre:g}"]
        for b in range(2):
            check_stft(st[b], stft_reference(x[b], case, pre), f"{case.id} stft pre={pre:g} clip {b}")
    assert np.array_equal(r["nchw"][:, 0], r["f32"]["log_mel"].transpose(0, 2, 1)), case.id
    t, n = r["tables"], r["n_fft_pow2"]
    assert np.array_equal(t["window"], _get_window(case.window, case.fl).astype(np.float32)), case.id
    assert np.array_equal(t["fbank"], mel_filterbank(case.n_mels, n, case.sr, case.f_min, case.f_max).astype(np.float32))
    assert np.array_equal(t["dct2"], (2.0 * _dct_basis(case.n_mfcc, case.n_mels)).astype(np.float32)), case.id


FEAT = "feat_warp8_kernel<"


def _template_args(name: str) -> list:
    args = name[name.index(FEAT) + len(FEAT):name.index(">")].split(",")
    return [int(a) if a.strip().lstrip("-").isdigit() else a.strip() == "true" for a in args]


@pytest.mark.gpu
def test_device_sweep_reaches_every_variant(device_sweep):
    """Which feature kernels the sweep launched, from their template arguments <R1, PRE, STFT, SHARE, NW, EMB, U4,
    PCM, RAGGED> and block sizes: every (path, radix) pair, pre-emphasis on and off, EMB / PCM / RAGGED at every radix,
    and every CTA shape of the feature path."""
    _, launches = device_sweep
    feat = set()
    for name, block in launches:
        if FEAT in name:
            a = _template_args(name)
            assert block == (a[4] * 32, 1, 1), (name, block)
            feat.add(tuple(a))
    names = {n for n, _ in launches}
    reached = sorted(feat)
    print(f"{len(reached)} feat_warp8_kernel instantiations:", *reached, sep="\n  ")
    print("other feature kernels:", sorted(n for n in names if "feat_" in n and FEAT not in n))
    plain = [a for a in feat if not a[2]]                          # not STFT
    path = {(("PCM16" if a[7] else "U4" if a[6] else "SHARE" if a[3] else "ALIGNED"), a[0]) for a in plain}
    assert path == {(p, r) for p in ("ALIGNED", "U4", "PCM16") for r in (4, 8, 16)} | {("SHARE", 4), ("SHARE", 8)}, path
    assert {a[1] for a in plain} == {True, False}
    for i, what in ((5, "EMB"), (7, "PCM"), (8, "RAGGED")):
        assert {a[0] for a in plain if a[i]} == {4, 8, 16}, what
    assert {(a[0], a[4]) for a in plain} == {(4, 20), (4, 12), (4, 8), (8, 20), (8, 12), (8, 8), (16, 10), (16, 8)}
    assert {(a[0], a[1]) for a in feat if a[2]} == {(r, p) for r in (4, 8, 16) for p in (True, False)}   # STFT mode
    x2 = {n for n in names if "feat_warp8_x2_kernel<" in n}
    assert len(x2) == 4, x2                                        # <PRE, AL4>
    assert any("feat_generic_kernel" in n for n in names)


def long_clip(frames: int, seed: int) -> np.ndarray:
    """16 kHz at 512/128: noise of amplitude 1e-6 with digital silence over its middle three fifths, where every
    log-mel value is ln 1e-10 and C0 = -46 n_mels"""
    n = 512 + (frames - 1) * 128
    x = np.random.default_rng(seed).standard_normal(n, dtype=np.float32) * np.float32(1e-6)
    x[n // 5: 4 * n // 5] = 0.0
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("n_mels, frames", ((128, 300_000), (256, 80_000)))
def test_long_clip_embeddings(torch_cuda, n_mels, frames):
    """Embeddings alone of a clip long enough that the 64-bit sums of C0^2 2^20 of the fused path would overflow
    (C0 about -5800 at 128 mels and -11600 at 256: 1.14 and 1.23 times 2^63 over these clips).  Device buffer, host
    buffer and a ragged batch that holds the clip between two short ones: the oracle's mean and std, and bit for bit
    the embeddings of the MFCC path."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import features_batch, features_ragged
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    cfg = MfccConfig(16000, 512, 128, n_mels=n_mels)
    x = long_clip(frames, n_mels)
    ref = O.features_batch(x[None], O.OracleConfig(16000, 512, 128, n_mels=n_mels), want=("mfcc", "embed"))
    dev = torch.as_tensor(x).cuda()
    via_mfcc = features_batch(dev[None], cfg, ("mfcc", "embed"))["embed"].cpu().numpy()
    short = [torch.as_tensor(synth.host_clip(i, seed=3, length=32_000 + 38 * i, sample_rate=16000)).cuda() for i in range(2)]
    got = {
        "device": features_batch(dev[None], cfg, ("embed",))["embed"].cpu().numpy(),
        "host": features_batch(x[None], cfg, ("embed",))["embed"],
        "ragged": features_ragged([short[0], dev, short[1]], cfg, ("embed",))["embed"][1:2].cpu().numpy(),
    }
    check_embed(via_mfcc, ref["embed"], ref["mfcc"], f"{frames} frames, {n_mels} mels, MFCC path")
    for name, e in got.items():
        c0 = (float(e[0, 0]), float(e[0, cfg.n_mfcc]))
        print(f"{frames} frames, {n_mels} mels, {name}: C0 mean {c0[0]:.3f} std {c0[1]:.3f} "
              f"(oracle {ref['embed'][0, 0]:.3f}, {ref['embed'][0, cfg.n_mfcc]:.3f})")
        check_embed(e, ref["embed"], ref["mfcc"], f"{frames} frames, {n_mels} mels, {name}")
        assert np.array_equal(e, via_mfcc), name
