"""CPU-only checks: host-side tables, the C ABI surface, and the CPU replay of the kernels."""
from __future__ import annotations

import ctypes as C
import hashlib
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import REPO, rel_err


def _sha12(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:12]


@pytest.fixture(scope="module")
def built():
    from dsp_final_b200 import build

    return build.build_native(), build.build_emu()


def test_host_tables_bit_exact(known_answers):
    from dsp_final_b200.dsp.mfcc import _dct_basis, mel_filterbank
    from dsp_final_b200.dsp.stft import _get_window

    for key, want in known_answers["table_sha12"].items():
        kind, a, *rest = key.split("/")
        if kind == "fbank":
            got = _sha12(mel_filterbank(int(a), int(rest[0]), 44100))
        elif kind == "dct":
            got = _sha12(_dct_basis(int(a), int(rest[0])))
        else:
            got = _sha12(_get_window(kind, int(a)))
        assert got == want, key


def test_mfcc_config_matches_reference_dataclass(known_answers):
    """Field names/order/defaults feed FeatureCache.params_hash (src/features/cache.py:24-41)."""
    import json
    from dataclasses import asdict, fields

    from dsp_final_b200.dsp.mfcc import MfccConfig

    assert [f.name for f in fields(MfccConfig)] == ["sample_rate", "frame_length", "hop_length", "n_fft", "n_mels",
                                                     "n_mfcc", "f_min", "f_max", "pre_emphasis", "window"]
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    params = {"feature_type": "mfcc", **asdict(cfg)}
    params["n_fft"] = cfg.n_fft or cfg.frame_length
    params["f_max"] = cfg.sample_rate / 2
    assert params == known_answers["cache_params_mfcc_1024_512"]
    digest = hashlib.sha1(json.dumps(params, sort_keys=True, ensure_ascii=True).encode()).hexdigest()[:12]
    assert digest == known_answers["published_digests"]["mfcc/1024/512"] == "e637fe1e8db0"


def test_abi_exports_every_declared_symbol(built):
    lib_path, _ = built
    header = (REPO / "include" / "dspx.h").read_text()
    declared = set(re.findall(r"\b(dspx_[a-z0-9_]+)\s*\(", header))
    declared -= {"dspx_plan", "dspx_config", "dspx_plan_info"}
    assert len(declared) >= 18
    nm = subprocess.run(["nm", "-D", "--defined-only", str(lib_path)], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (dspx_[a-z0-9_]+)", nm))
    assert declared <= exported, declared - exported
    from dsp_final_b200 import _lib

    assert declared == set(_lib._SIGNATURES), declared ^ set(_lib._SIGNATURES)
    lib = _lib.load()                                   # loads and binds every symbol; no compute call
    assert lib.dspx_version().startswith(b"dspx")
    assert lib.dspx_next_pow_two(1000) == 1024 and lib.dspx_next_pow_two(1) == 1


def test_struct_layout_matches_header(built):
    from dsp_final_b200 import _lib

    assert C.sizeof(_lib.DspxConfig) == 56 and _lib.DspxConfig.f_min.offset == 24
    assert _lib.DspxConfig.window.offset == 48 and _lib.DspxConfig.kernel.offset == 52
    assert C.sizeof(_lib.DspxPlanInfo) == 32


def test_product_fails_loudly_without_a_gpu(built):
    """No CPU fallback: on a machine without CUDA the compute entry points raise."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("has a GPU")
    from dsp_final_b200 import _lib
    from dsp_final_b200.dsp.mfcc import MfccConfig, mfcc

    with pytest.raises(_lib.DspxError):
        mfcc(np.zeros(4096, np.float32), MfccConfig(44100, 1024, 512))


def test_product_never_touches_the_oracle():
    """oracle/ is test infrastructure: nothing under dsp_final_b200/ may import, load or name it."""
    pkg = REPO / "dsp_final_b200"
    bad = []
    for path in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list(pkg.rglob("*.cuh")):
        text = path.read_text()
        if re.search(r"^\s*(from|import)\s+oracle\b", text, re.M) or "liborc" in text or "dsp_oracle" in text:
            bad.append(str(path))
    assert not bad, bad


# ---- CPU replay of the CUDA phase functions (csrc/emu.cu) against the golden vectors ----------
def _emu(built):
    from dsp_final_b200 import _lib

    lib = C.CDLL(str(built[1]))
    return lib, _lib.DspxConfig


def _cfg_struct(DspxConfig, m, kernel=1):
    from dsp_final_b200 import _lib

    return DspxConfig(m["sample_rate"], m["frame_length"], m["hop_length"], m["n_fft"] or 0, m["n_mels"], m["n_mfcc"],
                      m["f_min"], -1.0 if m["f_max"] is None else m["f_max"], m["pre_emphasis"],
                      _lib.WINDOWS[m["window"]], kernel)


def test_generic_kernel_replay_matches_reference(built, golden_small):
    """The very source the GPU runs (feat_generic.cuh phase functions), replayed on the CPU."""
    lib, DspxConfig = _emu(built)
    z, meta = golden_small
    clips = np.ascontiguousarray(z["clips"])
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    for ci, m in enumerate(meta):
        cfg = _cfg_struct(DspxConfig, m)
        t = z[f"c{ci}_mfcc_0"].shape[0]
        lm = np.zeros((3, t, m["n_mels"]), np.float32)
        mf = np.zeros((3, t, m["n_mfcc"]), np.float32)
        rc = lib.emu_features_generic(C.byref(cfg), fp(clips), C.c_int64(3), C.c_int64(clips.shape[1]),
                                      C.c_int64(clips.shape[1]), 0, 0, fp(lm), fp(mf), None, 5 + ci)
        assert rc == 0
        st = np.zeros((1, t, z[f"c{ci}_stft_0"].shape[1], 2), np.float32)
        rc = lib.emu_features_generic(C.byref(cfg), fp(clips), C.c_int64(1), C.c_int64(clips.shape[1]),
                                      C.c_int64(clips.shape[1]), 1, 0, None, None, fp(st), 0)
        assert rc == 0
        for b in range(3):
            assert rel_err(mf[b], z[f"c{ci}_mfcc_{b}"]) < 1e-5, (ci, b)
            assert rel_err(lm[b], z[f"c{ci}_logmel_{b}"]) < 1e-5, (ci, b)
        assert rel_err(st[0, ..., 0] + 1j * st[0, ..., 1], z[f"c{ci}_stft_0"]) < 1e-6, ci


def test_warp8_kernel_replay_matches_reference(built, golden_small):
    """feat_warp8.cuh lane-phase functions (f32x2 kernel, n_fft 512 / 1024 / 2048) replayed on the CPU."""
    lib, DspxConfig = _emu(built)
    z, meta = golden_small
    clips = np.ascontiguousarray(z["clips"])
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    covered = 0
    for ci, m in enumerate(meta):
        cfg = _cfg_struct(DspxConfig, m, kernel=2)
        t = z[f"c{ci}_mfcc_0"].shape[0]
        lm = np.zeros((3, t, m["n_mels"]), np.float32)
        mf = np.zeros((3, t, m["n_mfcc"]), np.float32)
        rc = lib.emu_features_warp8(C.byref(cfg), fp(clips), C.c_int64(3), C.c_int64(clips.shape[1]),
                                    C.c_int64(clips.shape[1]), fp(lm), fp(mf), None, 0)
        n_fft = 1 << ((m["n_fft"] or m["frame_length"]) - 1).bit_length()              # mfcc.py:89-91
        supported = n_fft in (512, 1024, 2048, 4096)      # frames shorter / longer than n_fft run the general variant;
                                                          # 4096 = even / odd halves in the packed lanes (feat_warp8_x2.cuh)
        assert (rc == 0) == supported, (ci, rc)
        if rc != 0:
            continue
        covered += 1
        for b in range(3):
            assert rel_err(mf[b], z[f"c{ci}_mfcc_{b}"]) < 1e-5, (ci, b)
            assert rel_err(lm[b], z[f"c{ci}_logmel_{b}"]) < 1e-5, (ci, b)
    assert covered >= 19


def test_pcm16_quotient_is_exact(built):
    """The PCM16 conversion fused into the feature kernel's loads -- q = s (1/m), one fma refinement -- is the
    correctly rounded (s / 32768) / (m / 32768) of load_audio + normalize_audio for EVERY sample / peak pair."""
    lib, _ = _emu(built)
    lib.emu_pcm16_quotient_mismatches.restype = C.c_longlong
    total = C.c_longlong(0)
    assert lib.emu_pcm16_quotient_mismatches(C.byref(total)) == 0
    assert total.value == sum(min(2 * m + 1, m + 32768) for m in range(1, 32769))


def test_warp8_replay_unaligned_frames(built):
    """Odd hops and odd row strides put frames off the 8-byte grid: the 4-byte-load variant of the warp8 kernel
    (U4) against the oracle, n_fft 512 / 1024 / 2048 (hop 441 = 10 ms at 44.1 kHz is a common setting)."""
    from dsp_final_b200 import synth
    from oracle import oracle as O

    lib, DspxConfig = _emu(built)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    for fl, hop, length in ((1024, 441, 12_001), (512, 147, 9_000), (2048, 441, 16_385), (1024, 512, 12_001)):
        x = np.ascontiguousarray(synth.host_clips(2, seed=17, length=length))
        m = dict(sample_rate=44100, frame_length=fl, hop_length=hop, n_fft=None, n_mels=40, n_mfcc=13, f_min=0.0,
                 f_max=None, pre_emphasis=0.97, window="hann")
        cfg = _cfg_struct(DspxConfig, m, kernel=2)
        t = 1 + (length - fl) // hop
        lm = np.zeros((2, t, 40), np.float32)
        mf = np.zeros((2, t, 13), np.float32)
        rc = lib.emu_features_warp8(C.byref(cfg), fp(x), C.c_int64(2), C.c_int64(length), C.c_int64(length), fp(lm), fp(mf), None, 0)
        assert rc == 0, (fl, hop)
        ref = O.features_batch(x, O.OracleConfig(44100, fl, hop), want=("mfcc", "log_mel"))
        assert rel_err(mf, ref["mfcc"]) < 1e-5 and rel_err(lm, ref["log_mel"]) < 1e-5, (fl, hop)


def test_warp8_replay_full_clip(built, golden_config1):
    lib, DspxConfig = _emu(built)
    g = golden_config1
    x = np.ascontiguousarray(g["clip"][None, :])
    m = dict(sample_rate=44100, frame_length=1024, hop_length=512, n_fft=None, n_mels=40, n_mfcc=13, f_min=0.0,
             f_max=None, pre_emphasis=0.97, window="hann")
    cfg = _cfg_struct(DspxConfig, m, kernel=2)
    lm = np.zeros((1, 429, 40), np.float32)
    mf = np.zeros((1, 429, 13), np.float32)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    assert lib.emu_features_warp8(C.byref(cfg), fp(x), C.c_int64(1), C.c_int64(220500), C.c_int64(220500), fp(lm), fp(mf), None, 0) == 0
    assert rel_err(mf[0], g["mfcc"]) < 1e-5 and rel_err(lm[0], g["logmel"]) < 1e-5


def test_warp8_table_layouts_are_conflict_aware(built):
    """The plan-time layouts of feat_warp8_kernel's tables (csrc/feat_warp8.cuh: w8_edge_colour, w8_seg_layout): no two
    bins share a tile slot, the filter-sum loads are conflict-free under the bank model, and the modelled wavefronts of
    the power stores stay below the round-1 layout's (59 for the headline configuration, measured by ncu)."""
    lib, DspxConfig = _emu(built)
    seen = {}
    for fl in (512, 1024, 2048):
        for n_mels in (40, 64, 128):
            m = dict(sample_rate=44100, frame_length=fl, hop_length=fl // 2, n_fft=None, n_mels=n_mels, n_mfcc=13, f_min=0.0,
                     f_max=None, pre_emphasis=0.97, window="hann")
            cfg = _cfg_struct(DspxConfig, m, kernel=2)
            out = (C.c_int32 * 8)()
            assert lib.emu_warp8_layout(C.byref(cfg), out) == 0, (fl, n_mels)
            pw, pw_min, sw, sw_min, fl_wf, fl_min, rounds, shared = list(out)
            seen[(fl, n_mels)] = list(out)
            assert shared == 0, (fl, n_mels)                     # every bin has its own slot
            assert fl_wf == fl_min, (fl, n_mels, fl_wf, fl_min)   # 128-bit filter-sum loads: one wavefront per quarter-warp
            assert pw_min <= pw <= 2 * pw_min and sw >= sw_min, (fl, n_mels, list(out))
    assert seen[(1024, 40)][0] <= 52 and seen[(1024, 40)][6] == 3, seen[(1024, 40)]
    assert seen[(512, 40)][6] == 2, seen[(512, 40)]              # even round counts are allowed (row swap for odd lanes)


def test_kernel_replay_is_addresssanitizer_clean(tmp_path):
    """Out-of-bounds check of the kernels' index arithmetic: the CPU replay of both feature kernels
    (exact-size shared-memory tiles and outputs) under AddressSanitizer, 11 configurations.
    compute-sanitizer is closed on the GPU pool, so this is the memcheck we have."""
    import shutil

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = tmp_path / "emu_asan"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-g", "-std=c++17", "-Xcompiler",
           "-fsanitize=address,-fno-omit-frame-pointer,-ffp-contract=off", "-o", str(exe),
           str(REPO / "tests" / "replay_asan_main.cu"), str(REPO / "dsp_final_b200" / "csrc" / "emu.cu"), "-lasan"]
    build = subprocess.run(cmd, capture_output=True, text=True)
    out = build.stderr + build.stdout
    if build.returncode != 0 and ("-lasan" in out or "libasan" in out):      # not "asan": the source file name has it
        pytest.skip("libasan not available")
    assert build.returncode == 0, build.stderr[-2000:]
    run = subprocess.run([str(exe)], capture_output=True, text=True,
                         env={"ASAN_OPTIONS": "protect_shadow_gap=0:detect_leaks=0", "PATH": "/usr/bin:/bin"})
    assert run.returncode == 0 and "AddressSanitizer" not in run.stderr, run.stderr[-3000:]
    lines = [l for l in run.stdout.splitlines() if l.startswith("fl ")]
    assert len(lines) == 11 and all(l.endswith("finite 1") for l in lines)
