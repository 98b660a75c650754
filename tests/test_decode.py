"""WAV decoding and channel downmix on the GPU, bit-identical to load_audio (+ normalize_audio): dspx_decode_layout,
dspx_decode_ragged, audio.read_wav_data, batch.load_audio_batch and the retrieval / cache paths that use them.

CPU: the layout; the replay of the kernel's tile decomposition (emu_decode) against read_wav + np.mean over every
encoding, channel counts 1 ... 32, tile-edge lengths and special values, compared as bit patterns; normalisation;
the numpy summation order the contract pins; WAV files with WAVE_FORMAT_EXTENSIBLE and odd chunks; an AddressSanitizer
run.  GPU (-m gpu): the device against the replay, a heterogeneous batch against per-clip calls, load_audio_batch
against load_audio at six rates, compute_embeddings / BatchFeatureCache against the host loader, and a profiler check.

The contract (DESIGN.md 4.6) repeats numpy's float32 pairwise sum; the order test imports the installed numpy, so a
release that sums differently fails here rather than drifting.
"""
from __future__ import annotations

import ctypes as C
import shutil
import struct
import subprocess

import numpy as np
import pytest

from conftest import REPO

ENCODINGS = ("pcm8", "pcm16", "pcm24", "pcm32", "f32", "f64")
# encoding -> (WAV format code, bits, dtype code of include/dspx.h, bytes per sample)
FORMAT = {"pcm8": (1, 8, 3, 1), "pcm16": (1, 16, 2, 2), "pcm24": (1, 24, 4, 3), "pcm32": (1, 32, 5, 4),
          "f32": (3, 32, 0, 4), "f64": (3, 64, 1, 8)}
CHANNELS = (1, 2, 3, 5, 6, 7, 8, 9, 12, 15, 16, 17, 24, 31, 32)
DECODE_CLIP = np.dtype([("in_offset", "<i8"), ("n_frames", "<i8"), ("channels", "<i4"), ("dtype", "<i4"),
                        ("out_start", "<i8"), ("out_length", "<i8")])


def _tile_frames(enc, c):
    """decode.cuh's dec_tile_frames."""
    return min(2048, (16384 // (c * FORMAT[enc][3])) & ~15)


def _lengths(enc, c):
    tf = _tile_frames(enc, c)
    return sorted({1, 2, 15, 16, 17, tf - 1, tf, tf + 1, 2 * tf + 3})


def _same_bits(a, b) -> bool:
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype == np.float32 and a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _samples(enc, n, rng, specials=True) -> bytes:
    """n random samples of an encoding as stored, with its special values sprinkled in."""
    pick = rng.random(n) < (0.02 if specials else 0.0)
    if enc == "pcm8":
        x = rng.integers(0, 256, n).astype(np.uint8)
        x[pick] = rng.choice(np.array([0, 255, 128], np.uint8), pick.sum())
        return x.tobytes()
    if enc == "pcm16":
        x = rng.integers(-32768, 32768, n).astype("<i2")
        x[pick] = rng.choice(np.array([-32768, 32767, 0], "<i2"), pick.sum())
        return x.tobytes()
    if enc == "pcm24":
        x = rng.integers(-(1 << 23), 1 << 23, n).astype(np.int32)
        x[pick] = rng.choice(np.array([-(1 << 23), (1 << 23) - 1, 0], np.int32), pick.sum())
        return x.astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    if enc == "pcm32":
        x = rng.integers(-(1 << 31), 1 << 31, n).astype("<i4")
        x[pick] = rng.choice(np.array([-(1 << 31), (1 << 31) - 1, 0, 255, 257], "<i4"), pick.sum())
        return x.tobytes()
    if enc == "f32":
        x = (rng.standard_normal(n) * np.exp(rng.uniform(-20, 20, n))).astype("<f4").view("<u4")
        special = np.array([0x00000000, 0x80000000, 0x00000001, 0x807fffff, 0x00400000, 0x7f800000, 0xff800000,
                            0x7fc00000, 0xffc12345, 0x7f800001, 0x7f7fffff], "<u4")
        x[pick] = rng.choice(special, pick.sum())
        return x.tobytes()
    x = (rng.standard_normal(n) * np.exp(rng.uniform(-30, 30, n))).astype("<f8")
    special = np.array([0.0, -0.0, 1e39, -3.5e38, 3.4028235e38, 1e-46, -1e-47, 1e-40, -1.4e-45, 7e-46,
                        np.inf, -np.inf], "<f8")
    x[pick] = rng.choice(special, pick.sum())
    u = x.view("<u8")
    nan = rng.random(n) < (0.004 if specials else 0.0)
    u[nan] = rng.choice(np.array([0x7ff8000000000000, 0xfff0000000000001, 0x7ff123456789abcd], "<u8"), nan.sum())
    return u.tobytes()


def _wav_bytes(data: bytes, rate, channels, enc, extensible=False, odd_chunk=False) -> bytes:
    code, bits, _, size = FORMAT[enc]
    if extensible:
        guid = struct.pack("<H", code) + b"\x00\x00\x00\x00\x10\x00\x80\x00\x00\xaa\x00\x38\x9b\x71"
        fmt = struct.pack("<HHIIHHHHI", 0xFFFE, channels, rate, rate * channels * size, channels * size, bits, 22, bits,
                          0) + guid
    else:
        fmt = struct.pack("<HHIIHH", code, channels, rate, rate * channels * size, channels * size, bits)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt
    if odd_chunk:
        body += b"LIST" + struct.pack("<I", 3) + b"abc\x00"           # odd size, then RIFF's pad byte
    body += b"data" + struct.pack("<I", len(data)) + data + (b"\x00" if len(data) & 1 else b"")
    return b"RIFF" + struct.pack("<I", len(body)) + body


def write_wav(path, data: bytes, rate, channels, enc, **kw):
    path.write_bytes(_wav_bytes(data, rate, channels, enc, **kw))
    return path


def _reference(path, normalize=False):
    """load_audio(path)[0] computed with this package's decoder (read_wav), then normalize_audio."""
    from dsp_final_b200.audio import normalize_audio, read_wav

    audio, _ = read_wav(path)
    if audio.ndim > 1:
        audio = np.mean(audio, axis=1)
    audio = audio.astype(np.float32)
    return normalize_audio(audio) if normalize else audio


@pytest.fixture(scope="module")
def emu():
    from dsp_final_b200 import build

    build.build_native()
    lib = C.CDLL(str(build.build_emu()))
    lib.emu_decode.restype = C.c_int
    lib.emu_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
    return lib


def _layout(parsed):
    """(input bytes at 16-byte offsets, dspx_decode_layout table, packed output length)."""
    from dsp_final_b200 import _lib

    sizes = np.array([len(p[0]) for p in parsed], np.int64)
    offsets = np.zeros(len(parsed), np.int64)
    offsets[1:] = np.cumsum((sizes + 15) // 16 * 16)[:-1]
    buf = np.zeros(int(offsets[-1] + sizes[-1]) if len(parsed) else 0, np.uint8)
    for o, p in zip(offsets, parsed):
        buf[o:o + len(p[0])] = p[0]
    cols = [np.ascontiguousarray(v) for v in (offsets, np.array([p[4] for p in parsed], np.int64),
                                              np.array([p[2] for p in parsed], np.int32),
                                              np.array([p[3] for p in parsed], np.int32))]
    table = np.zeros(len(parsed), DECODE_CLIP)
    total = _lib.load().dspx_decode_layout(*(c.ctypes.data for c in cols), len(parsed), table.ctypes.data)
    assert total >= 0, _lib.last_error()
    return buf, table, int(total)


def _emu_decode(lib, parsed, normalize):
    buf, table, total = _layout(parsed)
    out = np.full(max(total, 1), np.nan, np.float32)
    assert lib.emu_decode(buf.ctypes.data, table.ctypes.data, len(table), int(normalize), out.ctypes.data) == 0
    return [out[s:s + n] for s, n in zip(table["out_start"], table["out_length"])]


def _grid_files(tmp_path, enc, specials=True):
    """One file per (channels, tile-edge length) of an encoding."""
    rng = np.random.default_rng(FORMAT[enc][1] * 7 + FORMAT[enc][0])
    paths = []
    for c in CHANNELS:
        for n in _lengths(enc, c):
            paths.append(write_wav(tmp_path / f"{enc}_{c}_{n}.wav", _samples(enc, n * c, rng, specials), 44100, c, enc))
    return paths


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_decode_layout():
    from dsp_final_b200 import _lib

    lib = _lib.load()

    def layout(offsets, frames, chans, dtypes):
        cols = [np.ascontiguousarray(v, dt) for v, dt in ((offsets, np.int64), (frames, np.int64), (chans, np.int32),
                                                          (dtypes, np.int32))]
        table = np.zeros(len(cols[0]), DECODE_CLIP)
        return int(lib.dspx_decode_layout(*(c.ctypes.data for c in cols), len(cols[0]), table.ctypes.data)), table

    rng = np.random.default_rng(3)
    frames = np.concatenate(([1, 2, 3, 4, 5, 220500], rng.integers(1, 300_000, 40)))
    chans = rng.integers(1, 33, len(frames))
    dtypes = rng.integers(0, 6, len(frames))
    offsets = np.arange(len(frames)) * 4096
    total, table = layout(offsets, frames, chans, dtypes)
    assert np.array_equal(table["in_offset"], offsets) and np.array_equal(table["n_frames"], frames)
    assert np.array_equal(table["channels"], chans) and np.array_equal(table["dtype"], dtypes)
    assert np.array_equal(table["out_length"], frames)
    assert table["out_start"][0] == 0 and np.all(table["out_start"] % 4 == 0)
    assert np.array_equal(table["out_start"][1:], table["out_start"][:-1] + (frames[:-1] + 3) // 4 * 4)
    assert total == table["out_start"][-1] + frames[-1]
    assert layout([], [], [], [])[0] == 0
    good = ([0, 16], [5, 5], [2, 2], [2, 2])          # columns: in_offset, n_frames, channels, dtype
    for col, value in ((3, 6), (3, -1), (2, 0), (2, 33), (1, 0), (1, (1 << 40) + 1), (0, -16), (0, 8)):
        args = [list(v) for v in good]
        args[col][1] = value
        assert layout(*args)[0] == _lib.EINVAL, (col, value)
        assert "clip 1" in _lib.last_error(), _lib.last_error()
    assert layout([0], [1 << 40], [32], [1])[0] == 1 << 40


@pytest.mark.parametrize("enc", ENCODINGS)
def test_replay_bit_identical_to_read_wav_and_mean(emu, tmp_path, enc):
    """Every encoding x C in CHANNELS x tile-edge lengths, with special values, in one replayed batch per encoding."""
    from dsp_final_b200.audio import read_wav_data

    paths = _grid_files(tmp_path, enc)
    parsed = [read_wav_data(p) for p in paths]
    assert all(p is not None for p in parsed)
    for normalize in (False, True):
        got = _emu_decode(emu, parsed, normalize)
        for p, g in zip(paths, got):
            assert _same_bits(g, _reference(p, normalize)), (p.name, normalize)


def test_replay_special_values(emu, tmp_path):
    from dsp_final_b200.audio import read_wav_data

    cases = {
        "pcm8": (np.array([0, 255, 128], np.uint8), [-1.0, 127 / 128, 0.0]),
        "pcm16": (np.array([-32768, 32767], "<i2"), [-1.0, 32767 / 32768]),
        "pcm24": (np.array([-(1 << 23), (1 << 23) - 1], np.int32), [-1.0, ((1 << 23) - 1) / (1 << 23)]),
        "pcm32": (np.array([-(1 << 31), (1 << 31) - 1, 1], "<i4"), [-1.0, 1.0, 2.0 ** -31]),
    }
    for enc, (x, want) in cases.items():
        raw = x.astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes() if enc == "pcm24" else x.tobytes()
        parsed = read_wav_data(write_wav(tmp_path / f"{enc}.wav", raw, 8000, 1, enc))
        assert _same_bits(_emu_decode(emu, [parsed], False)[0], np.array(want, np.float32)), enc
    f64 = np.array([1e39, -1e39, 1e-46, -1e-46, 1e-40, np.inf, -np.inf], "<f8")
    parsed = read_wav_data(write_wav(tmp_path / "f64.wav", f64.tobytes(), 8000, 1, "f64"))
    assert _same_bits(_emu_decode(emu, [parsed], False)[0], f64.astype(np.float32))
    f32 = np.array([0x80000000, 0x00000001, 0x7f800000, 0xff800000, 0x7fa00001, 0xffc12345], "<u4")
    parsed = read_wav_data(write_wav(tmp_path / "f32.wav", f32.tobytes(), 8000, 1, "f32"))
    assert np.array_equal(_emu_decode(emu, [parsed], False)[0].view("<u4"), f32)     # kept as stored, payloads too
    for c in (2, 8, 9):                                                               # all-(-0) frames give +0
        raw = np.full(3 * c, 0x80000000, "<u4").tobytes()
        path = write_wav(tmp_path / f"negzero{c}.wav", raw, 8000, c, "f32")
        got = _emu_decode(emu, [read_wav_data(path)], False)[0]
        assert np.all(got.view("<u4") == 0) and _same_bits(got, _reference(path)), c


def test_replay_normalisation_leaves_zero_and_nan_clips(emu, tmp_path):
    from dsp_final_b200.audio import read_wav_data

    zero = write_wav(tmp_path / "zero.wav", np.zeros(2 * 500, "<i2").tobytes(), 8000, 2, "pcm16")
    x = np.random.default_rng(1).standard_normal(3 * 700).astype("<f4")
    x[1000] = np.nan
    nan = write_wav(tmp_path / "nan.wav", x.tobytes(), 8000, 3, "f32")
    y = np.random.default_rng(2).standard_normal(9 * 300).astype("<f4")
    y[17] = np.inf
    inf = write_wav(tmp_path / "inf.wav", y.tobytes(), 8000, 9, "f32")
    got = _emu_decode(emu, [read_wav_data(p) for p in (zero, nan, inf)], True)
    for g, p in zip(got, (zero, nan, inf)):
        assert _same_bits(g, _reference(p, True)), p.name
    assert np.all(got[0] == 0) and np.isnan(got[1]).sum() == 1


def _pairwise_mean(x):
    """The order DESIGN.md 4.6 pins: np.mean(float32 [n, C], axis=1) as numpy sums it."""
    n = x.shape[1]
    if n < 8:
        acc = np.zeros(x.shape[0], np.float32)
        for c in range(n):
            acc = acc + x[:, c]
    else:
        r = [x[:, j].copy() for j in range(8)]
        i = 8
        while i + 8 <= n:
            for j in range(8):
                r[j] = r[j] + x[:, i + j]
            i += 8
        acc = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        for c in range(i, n):
            acc = acc + x[:, c]
        acc = np.float32(0.0) + acc                  # the reduction's identity: all-(-0) frames give +0
    return (acc / np.float32(n)).astype(np.float32)


@pytest.mark.parametrize("c", range(2, 33))
def test_numpy_downmix_order(c):
    rng = np.random.default_rng(c)
    wide = (rng.standard_normal((50_000, c)) * np.exp(rng.uniform(-20, 20, (50_000, c)))).astype(np.float32)
    pcm24 = (rng.integers(-(1 << 23), 1 << 23, (50_000, c)) / (1 << 23)).astype(np.float32)
    for x in (wide, pcm24, np.full((4, c), -0.0, np.float32)):
        assert _same_bits(np.mean(x, axis=1), _pairwise_mean(x)), c


@pytest.mark.parametrize("enc", ENCODINGS)
def test_wav_files_extensible_and_odd_chunks(emu, tmp_path, enc):
    """read_wav_data + emu_decode equals load_audio on files with WAVE_FORMAT_EXTENSIBLE, an odd-sized chunk before
    data, and a data chunk that ends in a partial frame."""
    from dsp_final_b200.audio import load_audio, read_wav_data, read_wav_raw

    rng = np.random.default_rng(11)
    size = FORMAT[enc][3]
    paths = []
    for i, (c, n) in enumerate(((1, 1001), (2, 777), (6, 333), (3, 5))):
        data = _samples(enc, n * c, rng)
        if c > 1 and enc != "pcm24":                                     # a partial frame: dropped like read_wav_raw does
            data += _samples(enc, 1, rng)
        paths.append(write_wav(tmp_path / f"x{i}.wav", data, 48000, c, enc, extensible=bool(i % 2), odd_chunk=i >= 1))
    parsed = [read_wav_data(p) for p in paths]
    for p, d in zip(paths, parsed):
        raw, rate, _ = read_wav_raw(p)
        assert d[1] == rate == 48000 and d[2] == raw.shape[1] and d[3] == FORMAT[enc][2] and d[4] == raw.shape[0]
        assert len(d[0]) == d[4] * d[2] * size
    for normalize in (False, True):
        for p, g in zip(paths, _emu_decode(emu, parsed, normalize)):
            ref = load_audio(p)[0]
            from dsp_final_b200.audio import normalize_audio

            assert _same_bits(g, normalize_audio(ref) if normalize else ref), (p.name, normalize)


def test_read_wav_data_rejects_other_files(tmp_path):
    from dsp_final_b200.audio import read_wav_data

    assert read_wav_data(write_wav(tmp_path / "c33.wav", bytes(33 * 2 * 4), 8000, 33, "pcm16")) is None
    p = tmp_path / "alaw.wav"
    p.write_bytes(_wav_bytes(bytes(8), 8000, 1, "pcm8").replace(struct.pack("<HH", 1, 1), struct.pack("<HH", 6, 1), 1))
    assert read_wav_data(p) is None
    (tmp_path / "junk.wav").write_bytes(b"not a wav file at all")
    assert read_wav_data(tmp_path / "junk.wav") is None


def test_decode_replay_is_addresssanitizer_clean(tmp_path):
    """Tiles stage exactly the kernel's shared-memory size and read and write only their own clips."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = tmp_path / "decode_asan"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-g", "-std=c++17", "-Xcompiler",
           "-fsanitize=address,-fno-omit-frame-pointer,-ffp-contract=off", "-o", str(exe),
           str(REPO / "tests" / "replay_decode_asan_main.cu"), str(REPO / "dsp_final_b200" / "csrc" / "emu.cu"), "-lasan"]
    build = subprocess.run(cmd, capture_output=True, text=True)
    out = build.stderr + build.stdout
    if build.returncode != 0 and ("-lasan" in out or "libasan" in out):
        pytest.skip("libasan not available")
    assert build.returncode == 0, build.stderr[-2000:]
    run = subprocess.run([str(exe)], capture_output=True, text=True,
                         env={"ASAN_OPTIONS": "protect_shadow_gap=0:detect_leaks=0", "PATH": "/usr/bin:/bin"})
    assert run.returncode == 0 and "AddressSanitizer" not in run.stderr, run.stderr[-3000:]
    lines = [l for l in run.stdout.splitlines() if l.startswith("decode ")]
    assert len(lines) == 24 and all(l.endswith("rc 0 finite 1") for l in lines), run.stdout


def test_load_audio_batch_rejects_files_by_name(tmp_path):
    from dsp_final_b200.batch import load_audio_batch

    p = write_wav(tmp_path / "many.wav", bytes(40 * 2 * 3), 8000, 40, "pcm16")
    with pytest.raises(ValueError, match="many.wav"):
        load_audio_batch([p])


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def _device_decode(torch, parsed, normalize):
    from dsp_final_b200 import _lib

    lib = _lib.load()
    buf, table, total = _layout(parsed)
    data = torch.as_tensor(buf).cuda()
    table_dev = torch.as_tensor(table.view(np.uint8)).cuda()
    out = torch.full((max(total, 1),), float("nan"), dtype=torch.float32, device="cuda")
    ws_bytes = int(lib.dspx_decode_workspace(len(table)))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    _lib.check(lib.dspx_decode_ragged(data.data_ptr(), table_dev.data_ptr(), table.ctypes.data, len(table), int(normalize),
                                      out.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream),
               "dspx_decode_ragged")
    host = out.cpu().numpy()
    return [host[s:s + n] for s, n in zip(table["out_start"], table["out_length"])]


@pytest.mark.gpu
@pytest.mark.parametrize("enc", ENCODINGS)
def test_device_bit_identical_to_replay(torch_cuda, emu, tmp_path, enc):
    from dsp_final_b200.audio import read_wav_data

    paths = _grid_files(tmp_path, enc)
    parsed = [read_wav_data(p) for p in paths]
    for normalize in (False, True):
        got = _device_decode(torch_cuda, parsed, normalize)
        want = _emu_decode(emu, parsed, normalize)
        for p, g, w in zip(paths, got, want):
            assert _same_bits(g, w), (p.name, normalize)
            assert _same_bits(g, _reference(p, normalize)), (p.name, normalize)


@pytest.mark.gpu
def test_heterogeneous_batch_equals_single_clips(torch_cuda, tmp_path):
    from dsp_final_b200.audio import read_wav_data

    rng = np.random.default_rng(300)
    paths = []
    for i in range(300):
        enc, c = ENCODINGS[i % 6], 1 + i % 8
        n = int(rng.integers(1, 30_000))
        paths.append(write_wav(tmp_path / f"h{i}.wav", _samples(enc, n * c, rng, specials=False), 22050, c, enc))
    parsed = [read_wav_data(p) for p in paths]
    parsed[5] = read_wav_data(write_wav(tmp_path / "zero.wav", bytes(4 * 1000), 22050, 2, "pcm16"))
    for normalize in (False, True):
        batch = _device_decode(torch_cuda, parsed, normalize)
        for i, p in enumerate(parsed):
            assert _same_bits(batch[i], _device_decode(torch_cuda, [p], normalize)[0]), (i, normalize)


RATES = (8000, 16000, 22050, 44100, 48000, 96000)


@pytest.mark.gpu
def test_load_audio_batch_equals_load_audio(torch_cuda, tmp_path):
    from dsp_final_b200.audio import load_audio, normalize_audio
    from dsp_final_b200.batch import load_audio_batch

    rng = np.random.default_rng(44)
    paths = []
    for i, rate in enumerate(RATES * 3):
        enc, c = ENCODINGS[i % 6], (1, 2, 6)[i % 3]
        n = int(rng.integers(rate // 4, rate))
        paths.append(write_wav(tmp_path / f"r{i}.wav", _samples(enc, n * c, rng, specials=False), rate, c, enc))
    for target in (None, 16000, 44100):
        for normalize in (False, True):
            got = load_audio_batch(paths, target, normalize)
            for p, g in zip(paths, got):
                ref = load_audio(p, target)[0]
                ref = normalize_audio(ref) if normalize else ref
                assert g.is_cuda and _same_bits(g.cpu().numpy(), ref), (p.name, target, normalize)


def _mixed_items(tmp_path):
    """A small dataset of the kinds UrbanSound8K-style corpora mix."""
    from dsp_final_b200.datasets import Esc50Item

    rng = np.random.default_rng(8)
    kinds = [("pcm24", 2, 48000), ("pcm16", 6, 44100), ("f32", 1, 22050), ("pcm8", 1, 8000), ("pcm16", 1, 44100)]
    items = []
    for i in range(10):
        enc, c, rate = kinds[i % 5]
        n = int(rng.integers(rate, 3 * rate))
        path = tmp_path / "audio" / f"m{i}.wav"
        path.parent.mkdir(exist_ok=True)
        write_wav(path, _samples(enc, n * c, rng, specials=False), rate, c, enc)
        items.append(Esc50Item(f"m{i}.wav", 1 + i % 5, i % 4, f"class{i % 4}", path))
    return items


def _cfg(sr):
    from dsp_final_b200.dsp.mfcc import MfccConfig

    return MfccConfig(sample_rate=sr, frame_length=1024 if sr > 16000 else 512, hop_length=512 if sr > 16000 else 256)


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [16000, 44100])
def test_embeddings_and_cache_byte_identical_to_host_loader(torch_cuda, tmp_path, monkeypatch, sr):
    from dsp_final_b200 import audio
    from dsp_final_b200 import retrieval as R
    from dsp_final_b200.cache import BatchFeatureCache

    cfg = _cfg(sr)
    items = _mixed_items(tmp_path)
    loader = lambda it: audio.normalize_audio(audio.load_audio(it.path, cfg.sample_rate)[0])      # noqa: E731
    emb_host = R.compute_embeddings(items, cfg, loader=loader)
    host = BatchFeatureCache(tmp_path / "host")
    for ft in ("mfcc", "log_mel"):
        host.get_features(items, ft, cfg, loader=loader)

    def refuse(*a, **k):
        raise AssertionError("load_audio called: a file was decoded on the host")

    monkeypatch.setattr(audio, "load_audio", refuse)
    emb_gpu = R.compute_embeddings(items, cfg)
    assert emb_gpu.dtype == emb_host.dtype and emb_gpu.tobytes() == emb_host.tobytes()
    gpu = BatchFeatureCache(tmp_path / "gpu")
    for ft in ("mfcc", "log_mel"):
        gpu.get_features(items, ft, cfg)
        for it in items:
            assert host.feature_path(it, ft, cfg).read_bytes() == gpu.feature_path(it, ft, cfg).read_bytes(), (ft, it.filename)
    assert gpu.compute_feature(items[0], "mfcc", cfg).tobytes() == np.load(host.feature_path(items[0], "mfcc", cfg)).tobytes()


def _profiled_kernels(out_dir):
    """{call: CUDA kernel names} of two compute_embeddings calls, each profiled after a warm-up run; prints JSON."""
    import json
    from pathlib import Path

    import torch
    from torch.profiler import ProfilerActivity, profile

    from dsp_final_b200 import retrieval as R
    from dsp_final_b200.datasets import Esc50Item

    torch.cuda.set_device(0)
    out_dir = Path(out_dir)
    mixed = _mixed_items(out_dir)
    rng = np.random.default_rng(2)
    mono = []
    for i in range(4):
        path = write_wav(out_dir / f"mono{i}.wav", _samples("pcm16", 44100, rng, specials=False), 44100, 1, "pcm16")
        mono.append(Esc50Item(f"mono{i}.wav", 1, 0, "c", path))
    calls = {"mixed": lambda: R.compute_embeddings(mixed, _cfg(44100)),
             "mono_pcm16": lambda: R.compute_embeddings(mono, _cfg(44100))}
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
def test_decode_kernel_runs_only_for_files_off_the_pcm16_path(torch_cuda, tmp_path):
    """Profiled in a fresh process, as test_resample does: an earlier profiler session can leave later ones empty."""
    import json
    import sys

    code = f"import sys; sys.path[:0] = [{str(REPO)!r}, {str(REPO / 'tests')!r}]; " \
           f"import test_decode; test_decode._profiled_kernels({str(tmp_path)!r})"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    run = subprocess.run(cmd, capture_output=True, text=True, cwd=str(REPO), timeout=600)
    assert run.returncode == 0, run.stderr[-3000:]
    names = json.loads(run.stdout.strip().splitlines()[-1])
    for call, kernels in names.items():
        assert any("feat_" in k for k in kernels), (call, kernels)
    assert any("wav_decode_kernel" in k for k in names["mixed"]), names["mixed"]
    assert any("resample_poly_kernel" in k for k in names["mixed"]), names["mixed"]
    assert not any("decode" in k or "resample" in k for k in names["mono_pcm16"]), names["mono_pcm16"]
