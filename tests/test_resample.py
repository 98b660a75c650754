"""Polyphase resampling bit-identical to scipy.signal.resample_poly (dspx_resample, batch.resample_poly) and the
feature paths that use it for clips at another rate than the config's.

CPU: the replay of the kernel's tile decomposition (emu_resample) against scipy over ratios, lengths, dtypes and
normalisation; dspx_resample_layout; an AddressSanitizer run; argument errors.  GPU (-m gpu): the same grid through
dspx_resample (strided, batched, ragged), features_batch / features_ragged / BatchFeatureCache / compute_embeddings
against the host path, and a profiler check that the resample kernel runs only when the rates differ.

The contract is pinned on scipy 1.18.1, which filters float32 input in float32 (DESIGN.md 4.5).  scipy is imported
at run time, so a release that computes differently fails these tests rather than passing silently.
"""
from __future__ import annotations

import ctypes as C
import math
import shutil
import struct
import subprocess

import numpy as np
import pytest

from conftest import REPO

RATES = [(44100, 22050), (44100, 16000), (44100, 32000), (44100, 48000), (44100, 8000), (16000, 44100),
         (22050, 44100), (48000, 44100), (44100, 96000), (3, 7), (7, 3)]          # (rate in, rate out)
LENGTHS = (1, 5, 37, 1000, 22050, 220500)
BIG = (44100, 44099)       # 882 001 taps, a 3.7 MB phase table


def _scipy():
    from scipy.signal import resample_poly

    return resample_poly


def _reference(x, sr_in, sr_out, normalize):
    """load_audio's resample (on int16 / 32768 for PCM16), then normalize_audio."""
    from dsp_final_b200.audio import normalize_audio

    xf = x.astype(np.float32) / np.float32(32768.0) if x.dtype == np.int16 else x
    y = _scipy()(xf, sr_out, sr_in)
    assert y.dtype == np.float32
    return normalize_audio(y) if normalize else y


def _same_bits(a, b) -> bool:
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype == np.float32 and a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _signal(n, pcm, seed):
    rng = np.random.default_rng(seed)
    if pcm:
        return (rng.standard_normal(n) * 6000).clip(-32768, 32767).astype(np.int16)
    return (rng.standard_normal(n) * 0.3).astype(np.float32)


@pytest.fixture(scope="module")
def emu():
    from dsp_final_b200 import build

    build.build_native()
    lib = C.CDLL(str(build.build_emu()))
    lib.emu_resample.restype = C.c_int
    lib.emu_resample.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int64, C.c_int64,
                                 C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]
    lib.emu_resample_shape.restype = C.c_int
    lib.emu_resample_shape.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    return lib


def _window(up, down):
    from dsp_final_b200.plan import default_window, reduce_ratio

    up, down = reduce_ratio(up, down)
    return default_window(up, down) if (up, down) != (1, 1) else np.zeros(1, np.float32)


def _emu_resample(lib, x, up, down, normalize):
    w = _window(up, down)
    g = math.gcd(up, down)
    n_out = -(-len(x) * (up // g) // (down // g))
    out = np.full(n_out, np.nan, np.float32)
    rc = lib.emu_resample(up, down, w.ctypes.data, len(w), x.ctypes.data, 2 if x.dtype == np.int16 else 0, 1, len(x), len(x),
                          int(normalize), out.ctypes.data, n_out, None)
    assert rc == 0
    return out


def _edge_lengths(lib, sr_in, sr_out):
    """Input lengths whose outputs end one short of, on, and one past a column chunk, a row and a whole tile."""
    up, down = sr_out // math.gcd(sr_in, sr_out), sr_in // math.gcd(sr_in, sr_out)
    w = _window(up, down)
    shape = (C.c_int64 * 8)()
    assert lib.emu_resample_shape(up, down, w.ctypes.data, len(w), shape) == 0
    s, nr, u = shape[1], shape[2], shape[6]
    lengths = set()
    for o in (s, u, u * nr):
        for n_out in (o - 1, o, o + 1):
            if 1 <= n_out <= 2_000_000:
                n = -(-n_out * down // up)
                lengths.update((n, max(1, n - 1), n + 1))
    return sorted(lengths)


# ---- CPU: the kernel's tile decomposition against scipy -------------------------------------------------------------
@pytest.mark.parametrize("sr_in,sr_out", RATES)
def test_emu_bit_identical_to_scipy(emu, sr_in, sr_out):
    for n in list(LENGTHS) + _edge_lengths(emu, sr_in, sr_out):
        for pcm in (False, True):
            x = _signal(n, pcm, seed=n)
            for normalize in (False, True):
                got = _emu_resample(emu, x, sr_out, sr_in, normalize)
                assert _same_bits(got, _reference(x, sr_in, sr_out, normalize)), (sr_in, sr_out, n, pcm, normalize)


def test_emu_large_table_and_identity(emu):
    for sr_in, sr_out in (BIG, (44100, 44100), (3, 3)):
        for n in (1, 37, 22050, 100_000):
            for pcm in (False, True):
                x = _signal(n, pcm, seed=n + 1)
                for normalize in (False, True):
                    got = _emu_resample(emu, x, sr_out, sr_in, normalize)
                    assert _same_bits(got, _reference(x, sr_in, sr_out, normalize)), (sr_in, sr_out, n, pcm, normalize)
    x = np.array([-0.0, 0.5, -0.0], np.float32)              # a copy keeps the sign of zero
    assert _same_bits(_emu_resample(emu, x, 5, 5, False), x)


def test_emu_all_zero_clip_is_left_as_is(emu):
    x = np.zeros(1000, np.int16)
    assert _same_bits(_emu_resample(emu, x, 16000, 44100, True), _reference(x, 44100, 16000, True))


def test_resample_layout(emu):
    from dsp_final_b200 import _lib

    lib = _lib.load()

    def layout(up, down, starts, lengths):
        starts = np.ascontiguousarray(starts, np.int64)
        lengths = np.ascontiguousarray(lengths, np.int64)
        table = np.zeros((len(lengths), 4), np.int64)
        total = lib.dspx_resample_layout(up, down, starts.ctypes.data, lengths.ctypes.data, len(lengths), table.ctypes.data)
        return int(total), table

    rng = np.random.default_rng(5)
    lengths = np.concatenate(([1, 2, 3, 5, 220500], rng.integers(1, 300_000, 50)))
    starts = np.concatenate(([0], np.cumsum(lengths)[:-1]))
    for up, down in ((16000, 44100), (160, 441), (48000, 44100), (2, 2), (44099, 44100)):
        total, table = layout(up, down, starts, lengths)
        g = math.gcd(up, down)
        n_out = -(-lengths * (up // g) // (down // g))
        assert np.array_equal(table[:, 0], starts) and np.array_equal(table[:, 1], lengths)
        assert np.array_equal(table[:, 3], n_out)
        assert np.all(table[:, 2] % 4 == 0) and table[0, 2] == 0
        assert np.array_equal(table[1:, 2], table[:-1, 2] + (n_out[:-1] + 3) // 4 * 4)
        assert total == table[-1, 2] + table[-1, 3]
    assert layout(1, 1, [], [])[0] == 0
    for up, down, s, n in ((0, 1, [0], [5]), (1, -2, [0], [5]), (2, 1, [0], [0]), (2, 1, [-1], [5]), (2, 1, [0, 5], [5, -3])):
        assert layout(up, down, s, n)[0] == _lib.EINVAL, (up, down, s, n)


def test_resample_replay_is_addresssanitizer_clean(tmp_path):
    """Tiles stage exactly the kernel's shared-memory size, and read and write only their own clips, at tile-edge
    lengths and on the large-table ratio."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = tmp_path / "resample_asan"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-g", "-std=c++17", "-Xcompiler",
           "-fsanitize=address,-fno-omit-frame-pointer,-ffp-contract=off", "-o", str(exe),
           str(REPO / "tests" / "replay_resample_asan_main.cu"), str(REPO / "dsp_final_b200" / "csrc" / "emu.cu"), "-lasan"]
    build = subprocess.run(cmd, capture_output=True, text=True)
    out = build.stderr + build.stdout
    if build.returncode != 0 and ("-lasan" in out or "libasan" in out):
        pytest.skip("libasan not available")
    assert build.returncode == 0, build.stderr[-2000:]
    run = subprocess.run([str(exe)], capture_output=True, text=True,
                         env={"ASAN_OPTIONS": "protect_shadow_gap=0:detect_leaks=0", "PATH": "/usr/bin:/bin"})
    assert run.returncode == 0 and "AddressSanitizer" not in run.stderr, run.stderr[-3000:]
    lines = [l for l in run.stdout.splitlines() if l.startswith("resample ")]
    assert len(lines) == 7 and all(l.endswith("rc 0 finite 1") for l in lines), run.stdout


def test_bad_arguments_raise_valueerror():
    from dsp_final_b200.batch import resample_poly

    x = np.zeros(100, np.float32)
    for up, down in ((0, 1), (1, 0), (-2, 3), (1.5, 2), (2, 2.5)):
        with pytest.raises(ValueError):
            resample_poly(x, up, down)
    for bad in (np.zeros(100), np.zeros(100, np.int32), [np.zeros(5, np.float32), np.zeros(5)], np.zeros((2, 3, 4), np.float32)):
        with pytest.raises(ValueError):
            resample_poly(bad, 2, 1)


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def _strided(torch, x2d):
    """The rows of x2d on the device at an odd row stride, one sample past an aligned start."""
    b, n = x2d.shape
    stride = n + 2 + (n % 2 == 0)
    buf = torch.zeros((b, stride), dtype=torch.int16 if x2d.dtype == np.int16 else torch.float32, device="cuda")
    buf[:, 1:n + 1] = torch.as_tensor(x2d).cuda()
    return buf[:, 1:n + 1]


@pytest.mark.gpu
@pytest.mark.parametrize("sr_in,sr_out", RATES + [BIG, (44100, 44100)])
def test_device_bit_identical_to_scipy(torch_cuda, emu, sr_in, sr_out):
    torch = torch_cuda
    from dsp_final_b200.batch import resample_poly

    lengths = list(LENGTHS) + (_edge_lengths(emu, sr_in, sr_out) if sr_in != sr_out else [])
    if sr_in == BIG[0] and sr_out == BIG[1]:
        lengths = [1, 37, 22050, 100_000]
    for n in lengths:
        for pcm in (False, True):
            x = _signal(n, pcm, seed=n + 7)
            for normalize in (False, True):
                want = _reference(x, sr_in, sr_out, normalize)
                assert _same_bits(resample_poly(x, sr_out, sr_in, normalize), want), (n, pcm, normalize)
                got = resample_poly(_strided(torch, x[None]), sr_out, sr_in, normalize)
                assert _same_bits(got[0].cpu().numpy(), want), ("strided", n, pcm, normalize)
    for n in (1000, 22050):                                   # 300 clips in one launch, strided
        for pcm in (False, True):
            xs = np.stack([_signal(n, pcm, seed=1000 * i + n) for i in range(300)])
            xs[17] = 0                                        # an all-zero clip stays as it is
            for normalize in (False, True):
                got = resample_poly(_strided(torch, xs), sr_out, sr_in, normalize).cpu().numpy()
                for i in range(300):
                    assert _same_bits(got[i], _reference(xs[i], sr_in, sr_out, normalize)), (n, pcm, normalize, i)


@pytest.mark.gpu
@pytest.mark.parametrize("sr_in,sr_out", [(44100, 16000), (44100, 22050), (22050, 44100), (3, 7), BIG])
def test_ragged_equals_single_clip(torch_cuda, sr_in, sr_out):
    torch = torch_cuda
    from dsp_final_b200.batch import resample_poly

    rng = np.random.default_rng(sr_out)
    lengths = [1, 5, 37, 1000, 22050, 220500] + list(rng.integers(1, 100_000, 30))
    for pcm in (False, True):
        xs = [_signal(int(n), pcm, seed=i) for i, n in enumerate(lengths)]
        for normalize in (False, True):
            got = resample_poly([torch.as_tensor(x).cuda() for x in xs], sr_out, sr_in, normalize)
            host = resample_poly(xs, sr_out, sr_in, normalize)
            for i, x in enumerate(xs):
                alone = resample_poly(x, sr_out, sr_in, normalize)
                assert _same_bits(got[i].cpu().numpy(), alone) and _same_bits(host[i], alone), (pcm, normalize, i)
                if len(x) in (37, 22050):
                    assert _same_bits(alone, _reference(x, sr_in, sr_out, normalize))


def _cfg(sr):
    from dsp_final_b200.dsp.mfcc import MfccConfig

    return MfccConfig(sample_rate=sr, frame_length=1024 if sr > 16000 else 512, hop_length=512 if sr > 16000 else 256)


@pytest.mark.gpu
@pytest.mark.parametrize("target", [16000, 22050])
def test_features_at_another_rate_match_the_host_path(torch_cuda, target):
    """int16 at 44.1 kHz with sample_rate=44100: the same bits as features on normalize_audio(resample_poly(x/32768))."""
    torch = torch_cuda
    from dsp_final_b200.batch import features_batch, features_ragged, split_ragged

    cfg = _cfg(target)
    want = ("log_mel", "mfcc", "embed")
    xs = np.stack([_signal(5 * 44100, True, seed=i) for i in range(6)])
    ref_f = np.stack([_reference(x, 44100, target, True) for x in xs])
    ref = features_batch(torch.as_tensor(ref_f).cuda(), cfg, want)
    got = features_batch(torch.as_tensor(xs).cuda(), cfg, want, sample_rate=44100)
    for k in want:
        assert torch.equal(got[k], ref[k]), k
    host = features_batch(xs, cfg, want, sample_rate=44100)
    for k in want:
        assert np.array_equal(host[k], ref[k].cpu().numpy()), k
    # float32 input keeps its meaning: resampled as it is, never normalised
    flt = xs.astype(np.float32) / np.float32(32768.0)
    got_f = features_batch(torch.as_tensor(flt).cuda(), cfg, ("mfcc",), sample_rate=44100)["mfcc"]
    ref_ff = np.stack([_reference(x, 44100, target, False) for x in flt])
    assert torch.equal(got_f, features_batch(torch.as_tensor(ref_ff).cuda(), cfg, ("mfcc",))["mfcc"])
    # ragged: clips of different lengths, one resample launch and one feature launch
    lens = [44100, 3 * 44100 + 17, 2 * 44100 - 5, 4 * 44100]
    clips = [_signal(n, True, seed=n) for n in lens]
    for src in (clips, [torch.as_tensor(c).cuda() for c in clips]):
        r = features_ragged(src, cfg, ("log_mel", "mfcc"), sample_rate=44100)
        for i, c in enumerate(clips):
            # features_batch on the clip alone, in a row of even stride: ragged float32 clips start at even samples
            y = _reference(c, 44100, target, True)
            row = torch.zeros((1, len(y) + (len(y) & 1)), dtype=torch.float32, device="cuda")
            row[0, :len(y)] = torch.as_tensor(y).cuda()
            one = features_batch(row[:, :len(y)], cfg, ("log_mel", "mfcc"))
            for k in ("log_mel", "mfcc"):
                part = split_ragged(r[k], r["frame_offsets"])[i]
                part = part if isinstance(part, np.ndarray) else part.cpu().numpy()
                assert np.array_equal(part, one[k][0].cpu().numpy()), (k, i)


def _write_wav16(path, x, sr):
    data = np.ascontiguousarray(x, dtype="<i2").tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 1, 1, sr, sr * 2, 2, 16)
    path.write_bytes(hdr + b"data" + struct.pack("<I", len(data)) + data)


def _wav_items(tmp_path, lengths):
    from dsp_final_b200.datasets import Esc50Item

    items = []
    for i, n in enumerate(lengths):
        path = tmp_path / "audio" / f"clip{i}.wav"
        path.parent.mkdir(exist_ok=True)
        _write_wav16(path, _signal(int(n), True, seed=50 + i), 44100)
        items.append(Esc50Item(f"clip{i}.wav", 1 + i % 5, i % 7, f"class{i % 7}", path))
    return items


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", [False, True])
def test_cache_and_embeddings_byte_identical_to_host_path(torch_cuda, tmp_path, mixed):
    from dsp_final_b200 import retrieval as R
    from dsp_final_b200.audio import load_audio, normalize_audio, read_pcm16
    from dsp_final_b200.cache import BatchFeatureCache

    cfg = _cfg(22050)
    rng = np.random.default_rng(9)
    lengths = list(rng.integers(44100 // 2, 4 * 44100, 12)) if mixed else [5 * 44100] * 12
    items = _wav_items(tmp_path, lengths)
    assert read_pcm16(items[0].path)[1] == 44100
    host = BatchFeatureCache(tmp_path / "host")
    gpu = BatchFeatureCache(tmp_path / "gpu")
    loader = lambda it: normalize_audio(load_audio(it.path, cfg.sample_rate)[0])      # noqa: E731
    for ft in ("mfcc", "log_mel"):
        host.get_features(items, ft, cfg, loader=loader)
        gpu.get_features(items, ft, cfg)
        for it in items:
            a = host.feature_path(it, ft, cfg).read_bytes()
            assert a == gpu.feature_path(it, ft, cfg).read_bytes(), (ft, it.filename)
    emb_host = R.compute_embeddings(items, cfg, feature_cache=BatchFeatureCache(tmp_path / "eh"), loader=loader)
    emb_gpu = R.compute_embeddings(items, cfg, feature_cache=BatchFeatureCache(tmp_path / "eg"))
    assert np.array_equal(emb_host, emb_gpu)
    for it in items:
        assert (tmp_path / "eh").exists() and BatchFeatureCache(tmp_path / "eh").feature_path(it, "mfcc", cfg).read_bytes() == \
            BatchFeatureCache(tmp_path / "eg").feature_path(it, "mfcc", cfg).read_bytes()
    # precompute from int16 clips at their own rate writes the same files
    pre = BatchFeatureCache(tmp_path / "pre")
    pre.precompute(items, cfg, ("mfcc",), clips=[read_pcm16(it.path)[0] for it in items], sample_rate=44100)
    for it in items:
        assert pre.feature_path(it, "mfcc", cfg).read_bytes() == host.feature_path(it, "mfcc", cfg).read_bytes()


def _profiled_kernels(out_dir):
    """{call: CUDA kernel names} of four calls, each profiled in its own torch.profiler session after a warm-up run.
    Runs in a fresh process (see the test below); prints the result as JSON."""
    import json
    from pathlib import Path

    import torch
    from torch.profiler import ProfilerActivity, profile

    from dsp_final_b200 import retrieval as R
    from dsp_final_b200.batch import features_batch

    torch.cuda.set_device(0)
    out_dir = Path(out_dir)
    items = _wav_items(out_dir, [2 * 44100] * 4)
    x = torch.as_tensor(np.stack([_signal(44100, True, seed=i) for i in range(3)])).cuda()
    calls = {
        "embeddings_16000": lambda: R.compute_embeddings(items, _cfg(16000)),
        "embeddings_44100": lambda: R.compute_embeddings(items, _cfg(44100)),
        "batch_44100": lambda: features_batch(x, _cfg(44100), ("mfcc",), sample_rate=44100),
        "batch_22050": lambda: features_batch(x, _cfg(22050), ("mfcc",), sample_rate=44100),
    }
    names = {}
    for name, fn in calls.items():
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        trace = out_dir / f"{name}.json"
        prof.export_chrome_trace(str(trace))
        names[name] = [e["name"] for e in json.loads(trace.read_text())["traceEvents"] if e.get("cat") == "kernel"]
    print(json.dumps(names))


@pytest.mark.gpu
def test_resample_kernel_runs_only_when_rates_differ(torch_cuda, tmp_path):
    """The resample kernel runs for clips at another rate, and not when the rates match.  The calls are profiled in a
    fresh process: a torch.profiler session that an earlier test opened in this one can leave later sessions empty."""
    import json
    import sys

    code = f"import sys; sys.path[:0] = [{str(REPO)!r}, {str(REPO / 'tests')!r}]; " \
           f"import test_resample; test_resample._profiled_kernels({str(tmp_path)!r})"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    run = subprocess.run(cmd, capture_output=True, text=True, cwd=str(REPO), timeout=600)
    assert run.returncode == 0, run.stderr[-3000:]
    names = json.loads(run.stdout.strip().splitlines()[-1])
    for call, kernels in names.items():
        assert any("feat_" in k for k in kernels), (call, kernels)        # the session recorded the feature kernel
    assert any("resample_poly_kernel" in k for k in names["embeddings_16000"]), names["embeddings_16000"]
    assert any("resample_poly_kernel" in k for k in names["batch_22050"]), names["batch_22050"]
    assert not any("resample" in k for k in names["embeddings_44100"]), names["embeddings_44100"]
    assert not any("resample" in k for k in names["batch_44100"]), names["batch_44100"]
