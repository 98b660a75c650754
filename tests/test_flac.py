"""FLAC decoding and channel downmix on the GPU: dspx_flac_layout, dspx_flac_decode, audio.read_flac_data and the
load_audio_batch / retrieval / cache paths that use them (DESIGN.md 4.7).

The reference is FFmpeg's FLAC decoder (libavcodec, loaded from the opencv-python-headless wheel through ctypes): it
shares no code with the package.  tests/flac_ref.py writes the streams -- every subframe type and parameter the
format has -- and the first test proves that writer against FFmpeg before anything else relies on it.

CPU: writer conformance; the layout (frame discovery through sync-like data, ID3v2 and metadata skipping, variable
blocking, every error naming the file); the replay of the kernels' per-frame functions (emu_flac_decode) against the
FFmpeg integers scaled and np.mean-ed, as bit patterns; FLAC and WAV files of the same integers replaying to the same
bits; an AddressSanitizer run over the matrix and seeded corruptions.  GPU (-m gpu): the device against the replay, a
300-file FLAC + WAV batch against the host composition at six rates, embeddings and cache files byte-identical between
a corpus stored as WAV and as FLAC, corrupted files naming the file and frame, and a profiler check.
"""
from __future__ import annotations

import ctypes as C
import functools
import shutil
import struct
import subprocess

import numpy as np
import pytest

import flac_ref as F
from conftest import REPO

needs_ffmpeg = pytest.mark.skipif(F.ffmpeg() is None, reason="FFmpeg's libavcodec (opencv-python-headless) is not installed")


def _same_bits(a, b) -> bool:
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype == np.float32 and a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _reference(ints: np.ndarray, bps: int, normalize=False) -> np.ndarray:
    """load_audio's float32 clip of these integers: s / 2^(bps-1) (read_wav's scaling), then np.mean over channels."""
    from dsp_final_b200.audio import normalize_audio

    y = (ints.astype(np.float64) / float(1 << (bps - 1))).astype(np.float32)
    y = y[:, 0] if y.shape[1] == 1 else np.mean(y, axis=1)
    y = y.astype(np.float32)
    return normalize_audio(y) if normalize else y


def _smooth(rng, n, c, bps, level=0.9):
    """Band-limited noise at `level` of full scale: what LPC compresses well."""
    top = (1 << (bps - 1)) - 1
    out = []
    for _ in range(c):
        w = rng.standard_normal(n + 64)
        k = np.hanning(33)
        y = np.convolve(w, k / k.sum(), "same")[32:32 + n]
        y = y / (np.max(np.abs(y)) + 1e-12) * top * level
        out.append(np.round(y).astype(np.int64) + rng.integers(-1, 2, n))
    return np.clip(np.stack(out, 1), -top - 1, top)


def _noise(rng, n, c, bps):
    return rng.integers(-(1 << (bps - 1)), 1 << (bps - 1), (n, c), dtype=np.int64)


def _sync_like(bps_bytes=2):
    """Verbatim 16-bit samples whose bytes hold 0xFFF8 runs and a whole valid frame header (CRC-8 included) for frame
    number 7 of a mono 16-bit 44.1 kHz stream: a decoder that trusts sync codes would split the frame there."""
    head = bytes([0xFF, 0xF8, 0x69, 0x08, 0x07])
    head += bytes([F.crc8(head)])
    raw = (b"\xff\xf8" * 6 + head + b"\x00" + b"\xff\xf9\xff\xf8" * 4) * 8
    return np.frombuffer(raw, ">i2").astype(np.int64)


@functools.lru_cache(maxsize=None)
def matrix():
    """[(name, FLAC bytes, integers [n, C], bps)] over every stream feature the decoder handles."""
    rng = np.random.default_rng(2024)
    cases = []

    def add(name, x, bps, **kw):
        x = np.asarray(x, np.int64)
        x = x[:, None] if x.ndim == 1 else x
        cases.append((name, F.encode(x, kw.pop("rate", 44100), bps, **kw), x, bps))

    for bps in (4, 8, 12, 16, 20, 24, 32):
        lo = -(1 << (bps - 1))
        # 32-bit streams at a tenth of the level: coarse predictors' residuals must stay within 32 bits
        level = lambda v: v if bps < 32 else v / 10        # noqa: E731
        add(f"constant_{bps}", np.full(1000, lo), bps, blocks=1000, opts={"subframes": {"kind": "constant"}})
        add(f"verbatim_{bps}", _noise(rng, 1000, 1, bps), bps, blocks=1000, opts={"subframes": {"kind": "verbatim"}})
        for order in range(5):
            add(f"fixed{order}_{bps}", _smooth(rng, 3000, 1, bps, 0.5), bps, blocks=1024,
                opts={"subframes": {"kind": "fixed", "order": order}})
        for order, prec in ((1, 15), (2, 5), (8, 15), (8, 12), (12, 9), (31, 15), (32, 15), (32, 4)):
            add(f"lpc{order}p{prec}_{bps}", _smooth(rng, 3000, 1, bps, level(0.9)), bps, blocks=1024,
                opts={"subframes": {"kind": "lpc", "order": order, "precision": prec}})
        add(f"lpc8p1_{bps}", _smooth(rng, 2000, 1, bps, level(0.3)), bps, blocks=1000,
            opts={"subframes": {"kind": "lpc", "order": 8, "precision": 1}})
        for shift in (0, 7, 15):
            add(f"lpc_shift{shift}_{bps}", _smooth(rng, 2000, 1, bps, level(0.5)), bps, blocks=1000,
                opts={"subframes": {"kind": "lpc", "order": 4, "precision": 12, "shift": shift}})
    # predictions at their extremes: 24-bit full scale, 32 coefficients of the largest 15-bit magnitude, shift 15 --
    # partial sums of 2^42 need 64-bit accumulation -- and the same for the 33-bit side channel of a 32-bit stream
    x = _noise(rng, 4000, 1, 24)
    for name, coefs in (("pos", [16383] * 32), ("alt", [16383, -16384] * 16), ("neg", [-16384] * 32)):
        add(f"lpc_extreme_{name}_24", x, 24, blocks=1000,
            opts={"subframes": {"kind": "lpc", "order": 32, "precision": 15, "coefs": coefs, "shift": 15}})
    top = (1 << 31) - 1
    ext = np.stack([np.where(np.arange(2000) % 2, top, -top - 1), np.where(np.arange(2000) % 2, -top - 1, top)], 1)
    for asg in ("left_side", "right_side", "mid_side"):
        add(f"side33_verbatim_{asg}", ext, 32, blocks=500, opts={"assignment": asg, "subframes": {"kind": "verbatim"}})
        add(f"side33_lpc_{asg}", _smooth(rng, 4000, 2, 32, 0.99), 32, blocks=1000,
            opts={"assignment": asg, "subframes": {"kind": "lpc", "order": 8, "precision": 15}})
    # wasted bits
    add("wasted3_16", _smooth(rng, 2000, 1, 16) // 8 * 8, 16, blocks=1000,
        opts={"subframes": {"kind": "lpc", "order": 8, "wasted": 3}})
    add("wasted1_24_ls", _smooth(rng, 2000, 2, 24) // 2 * 2, 24, blocks=1000,
        opts={"assignment": "left_side", "subframes": {"kind": "fixed", "order": 2, "wasted": 1}})
    add("wasted7_8", rng.choice([-128, 0], (1000, 1)), 8, blocks=1000, opts={"subframes": {"kind": "verbatim", "wasted": 7}})
    add("wasted31_32", rng.choice([-(1 << 31), 0], (1000, 1)), 32, blocks=1000,
        opts={"subframes": {"kind": "verbatim", "wasted": 31}})
    # Rice and Rice2, partition orders 0-8, escapes, 0-bit escapes, k = 0 on noise (long unary runs), k up to 30
    s16 = _smooth(rng, 4096, 1, 16)
    for method in (0, 1):
        for po in range(9):
            add(f"rice{method}_po{po}", s16, 16, blocks=4096,
                opts={"subframes": {"kind": "lpc", "order": 8, "method": method, "porder": po}})
    add("escape", s16, 16, blocks=4096, opts={"subframes": {"kind": "fixed", "order": 2, "porder": 3, "escape": (0, 3, 7)}})
    add("escape_rice2", s16, 16, blocks=4096,
        opts={"subframes": {"kind": "fixed", "order": 2, "method": 1, "porder": 4, "escape": "all"}})
    z = s16.copy()
    z[:1024] = 0
    add("escape_0bit", z, 16, blocks=4096, opts={"subframes": {"kind": "fixed", "order": 1, "porder": 2, "escape": (0,)}})
    add("rice_k0_noise", _noise(rng, 256, 1, 16), 16, blocks=256,
        opts={"subframes": {"kind": "fixed", "order": 0, "porder": 0, "k": 0}})
    add("rice2_k30", _noise(rng, 1024, 1, 32), 32, blocks=1024,
        opts={"subframes": {"kind": "fixed", "order": 0, "method": 1, "porder": 1}})
    # channels and assignments
    for c in range(1, 9):
        add(f"independent_{c}ch", _smooth(rng, 3000, c, 16), 16, blocks=1024, opts={"subframes": {"kind": "lpc", "order": 6}})
    for bps in (8, 16, 24):
        for asg in ("left_side", "right_side", "mid_side"):
            add(f"{asg}_{bps}", _smooth(rng, 3000, 2, bps), bps, blocks=1024,
                opts={"assignment": asg, "subframes": {"kind": "lpc", "order": 8}})
    asgs = ("independent", "left_side", "right_side", "mid_side")
    add("assignment_per_frame", _smooth(rng, 4096, 2, 16), 16, blocks=512,
        opts=lambda i: {"assignment": asgs[i % 4], "subframes": {"kind": "lpc", "order": 4}})
    # every block-size code, 8- and 16-bit explicit sizes up to 65535, a short last frame; variable blocking
    sizes = [192, 576, 1152, 2304, 4608, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 1, 7, 100, 256, 257, 1000, 65535, 33]
    codes = {1: 6, 7: 6, 100: 6, 256: 6, 257: 7, 1000: 7, 65535: 7, 33: 7}
    xs = _smooth(rng, sum(sizes), 1, 16)

    def by_size(i):
        n = sizes[i]
        return {"block_code": codes.get(n, "auto") if i != 16 else 6,
                "subframes": {"kind": "verbatim"} if n < 8 else {"kind": "lpc", "order": 8}}

    add("block_codes_variable", xs, 16, blocks=sizes, variable=True, opts=by_size)
    add("block_short_last", xs[:10000], 16, blocks=4096, opts={"subframes": {"kind": "lpc", "order": 8}})
    add("block_16bit_fixed", xs[:70000], 16, blocks=65535, opts={"block_code": 7, "subframes": {"kind": "fixed", "order": 2}})
    # every sample-rate code form
    for rate in sorted(F.RATE_CODES):
        add(f"rate_{rate}", _smooth(rng, 600, 1, 16), 16, rate=rate, blocks=300, opts={"subframes": {"kind": "fixed", "order": 1}})
    for rate, code in ((44100, 0), (11000, 12), (255000, 12), (12345, 13), (65535, 13), (123450, 14), (655350, 14),
                       (1, 0), (1048575, 0), (7, 13)):
        add(f"rate_{rate}_code{code}", _smooth(rng, 600, 1, 16), 16, rate=rate, blocks=300,
            opts={"rate_code": code, "subframes": {"kind": "fixed", "order": 1}})
    add("size_code_from_streaminfo", _smooth(rng, 600, 1, 16), 16, blocks=300,
        opts={"size_code": 0, "subframes": {"kind": "fixed", "order": 1}})
    # frame / sample numbers of 1 ... 7 bytes, from streams cut out of longer ones; 2^31 and above
    for first in (0x7E, 0x7FE, 0xFFFE, 0x1FFFFE, 0x3FFFFFE, 0x7FFFFFFE - 3):
        add(f"frame_number_{first:x}", _smooth(rng, 1000, 1, 16), 16, blocks=200, first_number=first,
            opts={"subframes": {"kind": "fixed", "order": 2}})
    for first in (0, 100, 0x7FFFFFFF - 500, (1 << 31) + 12345, (1 << 36) - 5000):
        add(f"sample_number_{first:x}", _smooth(rng, 2000, 1, 16), 16, blocks=[700, 300, 1000], variable=True,
            first_number=first, opts={"subframes": {"kind": "fixed", "order": 2}})
    # sync-like runs inside the data, ID3v2 tags, other metadata blocks, an unknown total
    sy = np.concatenate([_sync_like()] * 4)
    add("sync_like", sy, 16, blocks=len(sy) // 4, opts={"subframes": {"kind": "verbatim"}})
    add("id3", _smooth(rng, 1000, 1, 16), 16, blocks=500, id3=300)
    add("id3_footer", _smooth(rng, 1000, 1, 16), 16, blocks=500, id3=17,
        metadata=[(1, bytes(50)), (4, b"\x05\x00\x00\x00dspx!\x00\x00\x00\x00"), (2, b"abcd" + bytes(9))])
    add("total_unknown", _smooth(rng, 1000, 2, 24), 24, blocks=300, total=0, opts={"assignment": "mid_side"})
    return cases


def _seven_byte(name: str) -> bool:
    """Streams whose sample numbers pass 2^31 - 1 and take 7-byte codes, which RFC 9639 allows but FFmpeg's
    GET_UTF8 refuses (a 0xFE lead byte).  They differ from the streams FFmpeg checks only in those numbers, so their
    reference is the written integers."""
    return name in ("sample_number_7ffffe0b", "sample_number_80003039", "sample_number_fffffec78")


def _ints(name, data, x, bps):
    """The reference integers of a matrix stream: FFmpeg's decode of it."""
    return x if _seven_byte(name) else F.ffmpeg_decode(data, bps, x.shape[1])


def _files(tmp_path, cases):
    paths = []
    for name, data, _, _ in cases:
        p = tmp_path / f"{name}.flac"
        p.write_bytes(data)
        paths.append(p)
    return paths


@pytest.fixture(scope="module")
def emu():
    from dsp_final_b200 import build

    build.build_native()
    lib = C.CDLL(str(build.build_emu()))
    lib.emu_flac_decode.restype = C.c_int
    lib.emu_flac_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                    C.c_void_p]
    lib.emu_decode.restype = C.c_int
    lib.emu_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
    return lib


def _layout(blobs):
    """(input buffer with the files at 16-byte offsets, file table, frame table, packed output length)."""
    from dsp_final_b200 import _lib
    from dsp_final_b200.batch import _flac_layout

    sizes = np.array([len(b) for b in blobs], np.int64)
    offsets = np.zeros(len(blobs), np.int64)
    offsets[1:] = np.cumsum((sizes + 15) // 16 * 16)[:-1]
    buf = np.zeros(int(offsets[-1] + sizes[-1]), np.uint8)
    parsed = []
    for o, b in zip(offsets, blobs):
        buf[o:o + len(b)] = np.frombuffer(b, np.uint8)
        parsed.append((np.frombuffer(b, np.uint8),))
    files, frames, total = _flac_layout(_lib.load(), offsets, parsed, list(range(len(blobs))))
    return buf, files, frames, total


def _split(out, files):
    return [out[s:s + n] for s, n in zip(files["out_start"], files["out_length"])]


def _emu(lib, blobs, normalize):
    buf, files, frames, total = _layout(blobs)
    out = np.zeros(max(total, 1), np.float32)
    status = np.full(len(frames), -1, np.int32)
    assert lib.emu_flac_decode(buf.ctypes.data, files.ctypes.data, len(files), frames.ctypes.data, len(frames),
                               int(normalize), out.ctypes.data, status.ctypes.data) == 0
    return _split(out, files), status


# ---- CPU: the writer against FFmpeg ----------------------------------------------------------------------------------

@needs_ffmpeg
def test_writer_decodes_through_ffmpeg_to_its_integers():
    """Every stream of the matrix decodes, through FFmpeg, to exactly the integers it was written from."""
    cases = matrix()
    assert sum(_seven_byte(c[0]) for c in cases) == 3
    for name, data, x, bps in cases:
        got = _ints(name, data, x, bps)
        assert got.shape == x.shape and np.array_equal(got, x), name


@needs_ffmpeg
def test_ffmpeg_binding_shifts_left_justified_samples_back():
    """Known integers at the bottom and top of every depth come back as themselves (FFmpeg stores 4-16-bit samples
    left-justified in 16 bits and 20-32-bit ones in 32 bits, planar when there are several channels)."""
    for bps in (4, 8, 12, 16, 20, 24, 32):
        x = np.array([[-(1 << (bps - 1)), (1 << (bps - 1)) - 1], [1, -1], [0, 3]], np.int64)
        for c in (1, 2):
            data = F.encode(x[:, :c], 8000, bps, blocks=3, opts={"subframes": {"kind": "verbatim"}})
            assert np.array_equal(F.ffmpeg_decode(data, bps, c), x[:, :c]), (bps, c)


# ---- CPU: layout -----------------------------------------------------------------------------------------------------

def test_layout_finds_every_frame_the_writer_wrote():
    """Frame offsets, lengths and block sizes equal the writer's, through sync-like data, ID3v2 tags, metadata blocks,
    variable blocking and numbers of every width; outputs are packed at 4-sample starts."""
    cases = matrix()
    buf, files, frames, total = _layout([c[1] for c in cases])
    at = 0
    for i, (name, data, x, bps) in enumerate(cases):
        f = files[i]
        assert (f["channels"], f["bps"], f["out_length"], f["n_frames"]) == (x.shape[1], bps, len(x), len(data.frames)), name
        assert f["out_start"] == at and f["out_start"] % 4 == 0, name
        rows = frames[f["first_frame"]:f["first_frame"] + f["n_frames"]]
        assert [(int(r["in_offset"]), int(r["in_bytes"])) for r in rows] == data.frames, name
        assert np.all(rows["file"] == i) and rows["block_size"].sum() == len(x), name
        assert np.array_equal(rows["out_start"], np.concatenate([[0], np.cumsum(rows["block_size"])[:-1]])), name
        ends = rows["ws_offset"] + (rows["block_size"] * x.shape[1] * (8 if bps == 32 else 4) + 15) // 16 * 16
        assert rows["ws_offset"][0] == 0 and np.array_equal(rows["ws_offset"][1:], ends[:-1]), name
        assert f["ws_bytes"] == ends[-1] and f["ws_start"] == (files[i - 1]["ws_start"] + files[i - 1]["ws_bytes"] if i else 0)
        at += (len(x) + 3) // 4 * 4
    assert total == files[-1]["out_start"] + files[-1]["out_length"]


def test_read_flac_data_detects_by_content(tmp_path):
    from dsp_final_b200 import _lib
    from dsp_final_b200.audio import read_flac_data, read_wav_data

    name, data, x, bps = matrix()[0]
    odd = tmp_path / "really_flac.wav"
    odd.write_bytes(data)
    d = read_flac_data(odd)
    assert d is not None and read_wav_data(odd) is None
    assert (d[1], d[2], d[3], d[4]) == (44100, 1, _lib.DTYPE_FLAC, len(x)) and d[0].tobytes() == bytes(data)
    (tmp_path / "junk.flac").write_bytes(b"not a flac file")
    assert read_flac_data(tmp_path / "junk.flac") is None


def _bad_files(tmp_path):
    """(file name, bytes, the error it must raise) for every host-side check of dspx_flac_layout."""
    rng = np.random.default_rng(5)
    x = _smooth(rng, 3000, 2, 16)
    good = F.encode(x, 44100, 16, blocks=1000)
    f0, f1 = good.frames[0], good.frames[1]
    si = 8                                                   # STREAMINFO body: after "fLaC" and its block header
    cases = []
    b = bytearray(good)
    b[4] = 0x04                                              # first block is not STREAMINFO
    cases.append(("not_streaminfo.flac", bytes(b), "byte 4: STREAMINFO is not the first"))
    cases.append(("md_past_end.flac", bytes(good[:30]), "byte 4: metadata block past the end"))
    b = bytearray(good)
    b[f0[0] + 4] ^= 0x01                                     # frame number byte: CRC-8 no longer matches
    cases.append(("header_crc8.flac", bytes(b), f"byte {f0[0]}: not a valid frame header"))
    wrong_total = F.encode(x, 44100, 16, blocks=1000, total=len(x) + 1)
    cases.append(("total.flac", bytes(wrong_total), f"byte {len(wrong_total)}: STREAMINFO total samples differ"))
    cases.append(("no_frames.flac", bytes(good[:f0[0]]), f"byte {f0[0]}: no audio frames"))
    b = bytearray(good)
    b[si + 12] = (b[si + 12] & 0xF1) | (0 << 1)              # STREAMINFO says 1 channel; the frames have 2
    cases.append(("channels.flac", bytes(b), f"byte {f0[0]}: not a valid frame header"))
    b = bytearray(good)
    b[si + 13] = (b[si + 13] & 0x0F) | (7 << 4)              # STREAMINFO says 24 bits (23 = 0b10111); frames code 16
    b[si + 12] |= 0x01
    cases.append(("bps.flac", bytes(b), f"byte {f0[0]}: not a valid frame header"))
    b = bytearray(good)
    b[si + 10:si + 13] = bytes([0, 0, b[si + 12] & 0x0F])      # sample rate 0
    cases.append(("rate0.flac", bytes(b), "STREAMINFO sample rate 0"))
    cases.append(("short_frame.flac", bytes(good[:f0[0] + 8]), f"byte {f0[0]}: frame shorter than its header"))
    return [(tmp_path / n, d, m) for n, d, m in cases]


def test_layout_errors_name_the_file_and_byte(tmp_path):
    from dsp_final_b200.audio import read_flac_data
    from dsp_final_b200.batch import load_audio_batch

    for path, data, msg in _bad_files(tmp_path):
        path.write_bytes(data)
        with pytest.raises(ValueError, match=path.name) as e:
            read_flac_data(path)
        assert msg in str(e.value), (path.name, str(e.value))
        with pytest.raises(ValueError, match=path.name):
            load_audio_batch([path])
    # an ID3v2 size with a high bit set: not recognisably FLAC to read_flac_data, refused by the layout itself
    from dsp_final_b200 import _lib
    from dsp_final_b200.batch import _flac_layout

    bad = b"ID3\x04\x00\x00\x00\x00\x80\x00" + bytes(F.encode(np.zeros(100, np.int64), 8000, 16, blocks=100))
    (tmp_path / "id3.flac").write_bytes(bad)
    assert read_flac_data(tmp_path / "id3.flac") is None
    with pytest.raises(ValueError, match="file 0: byte 0: bad ID3v2 tag size"):
        _flac_layout(_lib.load(), [0], [(np.frombuffer(bad, np.uint8),)], [0])


def test_layout_joins_per_file_tables_like_one_batch_call(tmp_path):
    """read_flac_data's own tables, joined for a batch, equal one dspx_flac_layout call over the whole batch, and
    load_audio_batch's host side parses each file once."""
    from dsp_final_b200 import _lib
    from dsp_final_b200.audio import read_flac_data
    from dsp_final_b200.batch import FLAC_FILE, FLAC_FRAME, _flac_layout

    cases = matrix()[::9]
    paths = _files(tmp_path, cases)
    lib = _lib.load()
    calls = []
    real = lib.dspx_flac_layout
    lib.dspx_flac_layout = lambda *a: calls.append(1) or real(*a)
    try:
        parsed = [read_flac_data(p) for p in paths]
    finally:
        lib.dspx_flac_layout = real
    assert len(calls) == len(paths)
    sizes = np.array([len(p[0]) for p in parsed], np.int64)
    offsets = np.concatenate([[0], np.cumsum((sizes + 15) // 16 * 16)[:-1]]).astype(np.int64)
    files, frames, total = _flac_layout(lib, offsets, parsed, list(range(len(parsed))))
    ptrs = (C.c_void_p * len(parsed))(*[p[0].ctypes.data for p in parsed])
    n = C.c_int64(0)
    want_files, want_frames = np.zeros(len(parsed), FLAC_FILE), np.zeros(len(frames), FLAC_FRAME)
    want_total = real(ptrs, sizes.ctypes.data, offsets.ctypes.data, len(parsed), want_files.ctypes.data,
                      want_frames.ctypes.data, len(want_frames), C.byref(n))
    assert n.value == len(frames) and want_total == total
    assert files.tobytes() == want_files.tobytes() and frames.tobytes() == want_frames.tobytes()


def test_trailing_id3v1_and_apev2_tags_are_not_part_of_the_last_frame(emu, tmp_path):
    """Taggers append ID3v1 ("TAG", 128 bytes) and APEv2 blocks after the last frame; the stream ends before them."""
    rng = np.random.default_rng(11)
    x = _smooth(rng, 3000, 2, 16)
    base = bytes(F.encode(x, 44100, 16, blocks=1000))
    ape_items = b"\x05\x00\x00\x00\x00\x00\x00\x00Title\x00hello"
    ape_footer = lambda flags: b"APETAGEX" + struct.pack("<IIII", 2000, len(ape_items) + 32, 1, flags) + bytes(8)  # noqa: E731
    id3v1 = b"TAG" + bytes(125)
    for name, tail in (("id3v1", id3v1), ("ape", ape_items + ape_footer(0)),
                       ("ape_header_id3v1", ape_footer(0xA0000000) + ape_items + ape_footer(0x80000000) + id3v1)):
        (out,), status = _emu(emu, [base + tail], False)
        assert not status.any() and _same_bits(out, _reference(x, 16)), name
    b = bytearray(base + id3v1)
    b[-128] = ord("X")                                       # not a tag: the bytes belong to the last frame
    _, status = _emu(emu, [bytes(b)], False)
    assert status.tolist()[-1] == 1


def test_damaged_header_mid_stream_is_named_at_its_offset(tmp_path):
    """A bit flipped in the header of frame 2 of 5 is reported at that header, with and without a STREAMINFO total."""
    from dsp_final_b200.audio import read_flac_data

    rng = np.random.default_rng(12)
    x = _smooth(rng, 5000, 1, 16)
    for total in ("auto", 0):
        good = F.encode(x, 44100, 16, blocks=1000, total=total)
        o2 = good.frames[2][0]
        for k in (4, 7):                                     # the frame number, then the header's CRC-8 byte
            b = bytearray(good)
            b[o2 + k] ^= 0x01
            p = tmp_path / f"damaged_{total}_{k}.flac"
            p.write_bytes(bytes(b))
            with pytest.raises(ValueError, match=rf"{p.name}: file 0: byte {o2}: damaged frame header"):
                read_flac_data(p)


def test_load_clips_falls_back_to_the_host_when_the_flac_path_refuses_a_file(tmp_path, monkeypatch):
    """A FLAC file the GPU decoder refuses goes to load_audio (soundfile, where installed), as it did before FLAC files
    had a GPU path; the host loader is a stub here, so no device is needed."""
    from dsp_final_b200 import audio
    from dsp_final_b200 import retrieval as R
    from dsp_final_b200.datasets import Esc50Item
    from dsp_final_b200.dsp.mfcc import MfccConfig

    rng = np.random.default_rng(13)
    good = F.encode(_smooth(rng, 3000, 1, 16), 44100, 16, blocks=1000)
    b = bytearray(good)
    b[good.frames[0][0] + 4] ^= 0x01                          # frame 0's header: refused by the host layout
    items = []
    for i, data in enumerate((bytes(good), bytes(b))):
        p = tmp_path / f"c{i}.flac"
        p.write_bytes(data)
        items.append(Esc50Item(p.name, 1, 0, "c", p))
    seen = []
    monkeypatch.setattr(audio, "load_audio", lambda path, target_sr=None: (seen.append(path) or np.ones(8, np.float32), 44100))
    clips, rate = R._load_clips(items, MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512), None)
    assert rate is None and len(clips) == 2 and [p.name for p in seen] == ["c0.flac", "c1.flac"]


# ---- CPU: replay -----------------------------------------------------------------------------------------------------

@needs_ffmpeg
def test_replay_bit_identical_to_ffmpeg_scaled_and_averaged(emu):
    """The per-frame functions of both kernels give the FFmpeg integers, scaled and np.mean-ed, bit for bit."""
    cases = matrix()
    for normalize in (False, True):
        outs, status = _emu(emu, [c[1] for c in cases], normalize)
        assert not status.any()
        for (name, data, x, bps), got in zip(cases, outs):
            want = _reference(_ints(name, data, x, bps), bps, normalize)
            assert _same_bits(got, want), (name, normalize)


def test_flac_and_wav_of_the_same_integers_replay_to_the_same_bits(emu):
    """A FLAC file and a WAV file holding the same integers decode to identical bits (1-8 channels, 8/16/24/32 bits),
    and both equal read_wav + np.mean."""
    import test_decode as TD
    from dsp_final_b200.audio import read_wav_data

    rng = np.random.default_rng(17)
    enc = {8: "pcm8", 16: "pcm16", 24: "pcm24", 32: "pcm32"}
    flacs, wavs, refs = [], [], []
    for bps in (8, 16, 24, 32):
        for c in range(1, 9):
            x = _smooth(rng, 2500, c, bps, 0.95)
            x[rng.random(len(x)) < 0.01] = -(1 << (bps - 1))
            asg = ("left_side", "right_side", "mid_side")[bps % 3] if c == 2 else "independent"
            kind = {"kind": "lpc", "order": 8} if bps < 32 else {"kind": "verbatim"}   # residuals within 32 bits
            flacs.append(bytes(F.encode(x, 22050, bps, blocks=1000, opts={"assignment": asg, "subframes": kind})))
            if bps == 8:
                raw = (x + 128).astype(np.uint8).tobytes()
            elif bps == 24:
                raw = x.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
            else:
                raw = x.astype("<i2" if bps == 16 else "<i4").tobytes()
            wavs.append(TD._wav_bytes(raw, 22050, c, enc[bps]))
            refs.append(_reference(x, bps))
    import tempfile
    from pathlib import Path

    with tempfile.TemporaryDirectory() as d:
        parsed = []
        for i, w in enumerate(wavs):
            p = Path(d) / f"w{i}.wav"
            p.write_bytes(w)
            parsed.append(read_wav_data(p))
        for normalize in (False, True):
            wav_out = TD._emu_decode(emu, parsed, normalize)
            flac_out, status = _emu(emu, flacs, normalize)
            assert not status.any()
            for i, (a, b, r) in enumerate(zip(flac_out, wav_out, refs)):
                from dsp_final_b200.audio import normalize_audio

                assert _same_bits(a, b) and _same_bits(a, normalize_audio(r) if normalize else r), (i, normalize)


def _corruptions(rng):
    """(name, bytes, statuses allowed) of seeded corruptions of matrix streams: bit flips with the CRC-16 left as it
    is (DSPX_FLAC_CRC), bit flips with the CRC-16 recomputed (the subframe walker runs on garbage: any status, None),
    frames truncated mid-frame or mid-header with the CRC-16 recomputed, streams the writer makes invalid on request,
    and frames out of order ("host": the layout refuses the file)."""
    out = []
    cases = matrix()
    picks = [c for c in cases if not c[0].startswith(("constant", "rate_"))]
    for k in range(40):
        name, data, x, bps = picks[int(rng.integers(len(picks)))]
        b = bytearray(data)
        o, n = max(data.frames, key=lambda f: f[1])
        fix = k % 2 == 1
        for _ in range(1 + k % 5):                           # past the longest header (16 bytes), before the CRC-16
            b[o + int(rng.integers(16, n - 2))] ^= 1 << int(rng.integers(8))
        if fix:
            b[o + n - 2:o + n] = struct.pack(">H", F.crc16(bytes(b[o:o + n - 2])))
        out.append((f"flip{k}_{name}", bytes(b), None if fix else {1}))
    for k, (name, data, x, bps) in enumerate(picks[::7]):
        o, n = data.frames[-1]
        for cut in (n // 2, 5, n - 3):
            body = bytearray(data[:o + cut])
            body += struct.pack(">H", F.crc16(bytes(body[o:])))
            out.append((f"cut{cut}_{name}", bytes(body), None))
    rng2 = np.random.default_rng(9)
    x = _smooth(rng2, 1000, 1, 16)
    out.append(("negative_shift", bytes(F.encode(x, 44100, 16, blocks=1000, opts={"subframes": {
        "kind": "lpc", "order": 4, "precision": 12, "coefs": [1, 0, 0, 0], "shift": -3}})), {8}))
    out.append(("reserved_type", bytes(F.encode(x, 44100, 16, blocks=1000, opts={"subframes": {"type_code": 2}})), {4}))
    out.append(("reserved_method", bytes(F.encode(x, 44100, 16, blocks=1000, opts={"subframes": {
        "kind": "fixed", "order": 1, "method_code": 2}})), {4}))
    out.append(("partition_order", bytes(F.encode(x[:999], 44100, 16, blocks=999, opts={"subframes": {
        "kind": "fixed", "order": 1, "porder": 3, "exact_porder": True}})), {16}))
    good = F.encode(x, 44100, 16, blocks=250)
    (o0, n0), (o1, n1) = good.frames[:2]
    # frame 1 first: it runs on through frame 0's bytes to frame 2, so the block sizes fall short of STREAMINFO's total
    out.append(("swapped_frames", bytes(good[:o0]) + good[o1:o1 + n1] + good[o0:o0 + n0] + good[o1 + n1:], "host"))
    return out


def test_replay_statuses_of_invalid_streams(emu):
    """Each invalid stream the writer makes ends in its status; the good frames around it decode."""
    for name, data, allowed in _corruptions(np.random.default_rng(1)):
        if allowed is None or name.startswith("flip"):
            continue
        if allowed == "host":
            with pytest.raises(ValueError, match="file 0: byte"):
                _layout([data])
            continue
        _, status = _emu(emu, [data], False)
        assert set(status.tolist()) == allowed, (name, status)


def test_flac_replay_is_addresssanitizer_clean(tmp_path):
    """Every frame of the matrix and of the seeded corruptions decodes from a buffer of exactly its bytes, with the
    bytes before it poisoned, and ends in a status: no read outside the frame, no write outside the file's output."""
    from dsp_final_b200 import _lib
    from dsp_final_b200.batch import _flac_layout

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = tmp_path / "flac_asan"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-g", "-std=c++17", "-Xcompiler",
           "-fsanitize=address,-fno-omit-frame-pointer,-ffp-contract=off", "-o", str(exe),
           str(REPO / "tests" / "replay_flac_asan_main.cu"), str(REPO / "dsp_final_b200" / "csrc" / "emu.cu"), "-lasan"]
    build = subprocess.run(cmd, capture_output=True, text=True)
    out = build.stderr + build.stdout
    if build.returncode != 0 and ("-lasan" in out or "libasan" in out):
        pytest.skip("libasan not available")
    assert build.returncode == 0, build.stderr[-2000:]
    streams = [(c[0], bytes(c[1]), {0}) for c in matrix()] + _corruptions(np.random.default_rng(1))
    rec = bytearray()
    expect = []
    lib = _lib.load()
    for i, (name, data, allowed) in enumerate(streams):
        try:
            files, frames, _ = _flac_layout(lib, [0], [(np.frombuffer(data, np.uint8),)], [0])
        except ValueError:                                    # refused on the host, e.g. a cut through a header
            assert allowed == "host" or name.startswith("cut"), name
            continue
        rec += struct.pack("<ii", i, len(frames)) + files.tobytes()
        for fr in frames:
            rec += fr.tobytes() + data[int(fr["in_offset"]):int(fr["in_offset"]) + int(fr["in_bytes"])]
        expect.append((i, name, len(frames), allowed))
    (tmp_path / "cases.bin").write_bytes(bytes(rec))
    run = subprocess.run([str(exe), str(tmp_path / "cases.bin")], capture_output=True, text=True,
                         env={"ASAN_OPTIONS": "protect_shadow_gap=0:detect_leaks=0", "PATH": "/usr/bin:/bin"})
    assert run.returncode == 0 and "AddressSanitizer" not in run.stderr, run.stderr[-3000:]
    lines = [l.split() for l in run.stdout.splitlines() if l.startswith("flac case")]
    assert len(lines) == sum(n for _, _, n, _ in expect)
    assert all(l[6] == "0" for l in lines), "emu_flac_decode refused a frame"     # flac case C frame F rc R status S
    by_case = {}
    for l in lines:
        by_case.setdefault(int(l[2]), []).append(int(l[8]))
    for i, name, n, allowed in expect:
        st = set(by_case[i])
        if allowed == {0}:
            assert st == {0}, (name, st)
        elif isinstance(allowed, set):
            assert allowed <= st, (name, st)


# ---- GPU -------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def _device(torch, blobs, normalize):
    from dsp_final_b200 import _lib
    from dsp_final_b200.batch import _flac_decode

    buf, files, frames, total = _layout(blobs)
    dev = torch.device("cuda", 0)
    data = torch.from_numpy(buf).to(dev)
    out = torch.zeros(max(total, 1), dtype=torch.float32, device=dev)
    status = _flac_decode(_lib.load(), data, (files, frames, 0, None), normalize, out, dev)
    return _split(out.cpu().numpy(), files), status.cpu().numpy()


@pytest.mark.gpu
def test_device_bit_identical_to_replay(torch_cuda, emu):
    cases = matrix()
    blobs = [c[1] for c in cases]
    for normalize in (False, True):
        got, st = _device(torch_cuda, blobs, normalize)
        want, st_emu = _emu(emu, blobs, normalize)
        assert not st.any() and not st_emu.any()
        for (name, *_), g, w in zip(cases, got, want):
            assert _same_bits(g, w), (name, normalize)


@pytest.mark.gpu
def test_device_statuses_match_replay(torch_cuda, emu):
    blobs = []
    for _, d, _ in _corruptions(np.random.default_rng(1)):
        try:
            _layout([d])
            blobs.append(d)
        except ValueError:                                    # refused on the host
            pass
    _, st = _device(torch_cuda, blobs, False)
    _, st_emu = _emu(emu, blobs, False)
    assert np.array_equal(st, st_emu)


RATES = (8000, 16000, 22050, 44100, 48000, 96000)


def _host_composition(ints, bps, rate, target, normalize):
    """FFmpeg-independent integers -> scale -> np.mean -> scipy resample_poly -> normalize_audio, as load_audio does."""
    from scipy.signal import resample_poly

    from dsp_final_b200.audio import normalize_audio

    y = _reference(ints, bps)
    if target is not None and rate != target:
        y = resample_poly(y, target, rate).astype(np.float32)
    return normalize_audio(y) if normalize else y


@needs_ffmpeg
@pytest.mark.gpu
def test_load_audio_batch_mixed_flac_and_wav_equals_host_composition(torch_cuda, tmp_path):
    import test_decode as TD
    from dsp_final_b200.audio import load_audio, normalize_audio
    from dsp_final_b200.batch import load_audio_batch

    rng = np.random.default_rng(300)
    paths, refs = [], []
    for i in range(300):
        rate = RATES[i % 6]
        n = int(rng.integers(1, 12000))
        if i % 2:
            enc, c = TD.ENCODINGS[i % 6], 1 + (i // 2) % 8
            p = TD.write_wav(tmp_path / f"w{i}.wav", TD._samples(enc, n * c, rng, specials=False), rate, c, enc)
            refs.append(None)
        else:
            bps, c = (4, 8, 12, 16, 20, 24, 32)[(i // 2) % 7], 1 + (i // 14) % 8
            x = _smooth(rng, n, c, bps) if i % 4 else _noise(rng, n, c, bps)
            kind = {"kind": "lpc", "order": 8} if i % 4 else {"kind": "verbatim"}
            data = F.encode(x, rate, bps, blocks=int(rng.integers(16, 4097)),
                            opts={"assignment": "mid_side" if c == 2 else "independent", "subframes": kind})
            p = tmp_path / f"f{i}.flac"
            p.write_bytes(data)
            refs.append((F.ffmpeg_decode(data, bps, c), bps, rate))
        paths.append(p)
    for target in (None, 16000, 44100):
        for normalize in (False, True):
            got = load_audio_batch(paths, target, normalize)
            for p, g, r in zip(paths, got, refs):
                if r is None:
                    want = load_audio(p, target)[0]
                    want = normalize_audio(want) if normalize else want
                else:
                    want = _host_composition(*r, target, normalize)
                assert g.is_cuda and _same_bits(g.cpu().numpy(), want), (p.name, target, normalize)


def _twin_items(tmp_path):
    """The same integers stored as WAV and as FLAC: (wav items, flac items)."""
    import test_decode as TD
    from dsp_final_b200.datasets import Esc50Item

    rng = np.random.default_rng(8)
    kinds = [(24, 2, 48000), (16, 6, 44100), (16, 1, 22050), (8, 1, 8000), (16, 2, 44100)]
    enc = {8: "pcm8", 16: "pcm16", 24: "pcm24"}
    wav, flac = [], []
    for d in ("wav", "flac"):
        (tmp_path / d).mkdir(exist_ok=True)
    for i in range(10):
        bps, c, rate = kinds[i % 5]
        x = _smooth(rng, int(rng.integers(rate, 3 * rate)), c, bps, 0.7)
        raw = ((x + 128).astype(np.uint8).tobytes() if bps == 8 else
               x.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes() if bps == 24 else x.astype("<i2").tobytes())
        pw = TD.write_wav(tmp_path / "wav" / f"m{i}.wav", raw, rate, c, enc[bps])
        pf = tmp_path / "flac" / f"m{i}.flac"
        pf.write_bytes(F.encode(x, rate, bps, blocks=4096, opts={"assignment": "mid_side" if c == 2 else "independent",
                                                                "subframes": {"kind": "lpc", "order": 8, "porder": 4}}))
        wav.append(Esc50Item(f"m{i}.wav", 1 + i % 5, i % 4, f"class{i % 4}", pw))
        flac.append(Esc50Item(f"m{i}.wav", 1 + i % 5, i % 4, f"class{i % 4}", pf))
    return wav, flac


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [16000, 44100])
def test_embeddings_and_cache_byte_identical_between_wav_and_flac(torch_cuda, tmp_path, monkeypatch, sr):
    import test_decode as TD
    from dsp_final_b200 import audio
    from dsp_final_b200 import retrieval as R
    from dsp_final_b200.cache import BatchFeatureCache

    cfg = TD._cfg(sr)
    wav, flac = _twin_items(tmp_path)

    def refuse(*a, **k):
        raise AssertionError("load_audio called: a file was decoded on the host")

    monkeypatch.setattr(audio, "load_audio", refuse)
    emb_wav, emb_flac = R.compute_embeddings(wav, cfg), R.compute_embeddings(flac, cfg)
    assert emb_wav.dtype == emb_flac.dtype and emb_wav.tobytes() == emb_flac.tobytes()
    cw, cf = BatchFeatureCache(tmp_path / "cw"), BatchFeatureCache(tmp_path / "cf")
    for ft in ("mfcc", "log_mel"):
        cw.get_features(wav, ft, cfg)
        cf.get_features(flac, ft, cfg)
        for a, b in zip(wav, flac):
            assert cw.feature_path(a, ft, cfg).read_bytes() == cf.feature_path(b, ft, cfg).read_bytes(), (ft, a.filename)


@pytest.mark.gpu
def test_corrupted_files_raise_naming_file_and_frame(torch_cuda, tmp_path):
    """Runs after test_flac_replay_is_addresssanitizer_clean has shown the decoder stays in bounds on these inputs."""
    from dsp_final_b200.audio import load_audio
    from dsp_final_b200.batch import load_audio_batch

    good = tmp_path / "good.flac"
    good.write_bytes([c for c in matrix() if c[0] == "independent_3ch"][0][1])
    for name, data, allowed in _corruptions(np.random.default_rng(1)):
        if allowed is None:
            continue
        p = tmp_path / f"{name}.flac"
        p.write_bytes(data)
        frame = "" if allowed == "host" else r": FLAC frame \d+ \(byte \d+\)"
        with pytest.raises(ValueError, match=rf"{p.name}{frame}"):
            load_audio_batch([good, p], 16000, True)
        with pytest.raises(ValueError, match=p.name):
            load_audio(p)
    assert load_audio_batch([good])[0].numel() > 0


@needs_ffmpeg
@pytest.mark.gpu
def test_load_audio_reads_flac_without_soundfile(torch_cuda, tmp_path):
    from dsp_final_b200 import audio

    if audio._sf is not None:
        pytest.skip("soundfile is installed: load_audio reads FLAC through it")
    name, data, x, bps = [c for c in matrix() if c[0] == "independent_3ch"][0]
    p = tmp_path / "a.flac"
    p.write_bytes(data)
    for target in (None, 16000):
        y, sr = audio.load_audio(p, target)
        assert sr == (44100 if target is None else target) and isinstance(y, np.ndarray)
        assert _same_bits(y, _host_composition(F.ffmpeg_decode(data, bps, 3), bps, 44100, target, False))


def _profiled_kernels(out_dir):
    """{call: CUDA kernel names} of compute_embeddings over a FLAC corpus and over the same corpus as WAV, each profiled
    after a warm-up run; prints JSON."""
    import json
    from pathlib import Path

    import torch
    from torch.profiler import ProfilerActivity, profile

    import test_decode as TD
    from dsp_final_b200 import retrieval as R

    torch.cuda.set_device(0)
    out_dir = Path(out_dir)
    wav, flac = _twin_items(out_dir)
    calls = {"flac": lambda: R.compute_embeddings(flac, TD._cfg(44100)),
             "wav": lambda: R.compute_embeddings(wav, TD._cfg(44100))}
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
def test_flac_kernels_run_only_for_flac_files(torch_cuda, tmp_path):
    """Profiled in a fresh process, as test_decode does: an earlier profiler session can leave later ones empty."""
    import json
    import sys

    code = f"import sys; sys.path[:0] = [{str(REPO)!r}, {str(REPO / 'tests')!r}]; " \
           f"import test_flac; test_flac._profiled_kernels({str(tmp_path)!r})"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    run = subprocess.run(cmd, capture_output=True, text=True, cwd=str(REPO), timeout=600)
    assert run.returncode == 0, run.stderr[-3000:]
    names = json.loads(run.stdout.strip().splitlines()[-1])
    for call, kernels in names.items():
        assert any("feat_" in k for k in kernels), (call, kernels)
    assert any("flac_frame_kernel" in k for k in names["flac"]) and any("flac_mix_kernel" in k for k in names["flac"])
    assert not any("flac" in k for k in names["wav"]), names["wav"]
    assert any("wav_decode_kernel" in k for k in names["wav"]), names["wav"]
