"""Audio file ingest with the reference's semantics (src/utils/audio.py:19-38).

    load_audio(path, target_sr=None) -> (float32 mono samples, sample_rate)
    normalize_audio(audio)           -> audio / max|audio|   (unchanged when the clip is all zero)

ESC-50 ships 16-bit PCM WAV files.  The reference decodes them with `soundfile.read(dtype="float32")`,
which yields int16 / 32768 exactly; `read_wav` below does the same with the standard library's RIFF
parsing (PCM 8/16/24/32-bit and IEEE float), so the package has no hard dependency on soundfile.  When
soundfile is importable it is used, like in the reference.  Decoding is host work (file I/O); the batched
GPU path takes the raw int16 samples instead (`load_pcm16`, dspx_features_host_pcm16: the conversion and
the peak normalisation then run on the device and PCIe carries half the bytes).  FLAC files are decoded on the
GPU (`read_flac_data`, batch.load_audio_batch); without soundfile, load_audio reads them that way too.
"""
from __future__ import annotations

import struct
from pathlib import Path
from typing import Tuple

import numpy as np

try:                                    # the reference's decoder, when present
    import soundfile as _sf
except ImportError:                     # pragma: no cover - depends on the image
    _sf = None


def _riff_chunks(blob: bytes):
    if len(blob) < 12 or blob[:4] != b"RIFF" or blob[8:12] != b"WAVE":
        raise ValueError("not a RIFF/WAVE file")
    pos = 12
    while pos + 8 <= len(blob):
        tag, size = blob[pos:pos + 4], struct.unpack_from("<I", blob, pos + 4)[0]
        yield tag, blob[pos + 8: pos + 8 + size]
        pos += 8 + size + (size & 1)


def _wav_chunks(path: str | Path) -> Tuple[int, int, int, int, bytes]:
    """(format code, channels, sample_rate, bits per sample, data chunk) of a WAV file."""
    fmt = data = None
    for tag, body in _riff_chunks(Path(path).read_bytes()):
        if tag == b"fmt ":
            fmt = body
        elif tag == b"data":
            data = body
    if fmt is None or data is None:
        raise ValueError(f"{path}: missing fmt or data chunk")
    code, channels, rate, _bps, _align, bits = struct.unpack_from("<HHIIHH", fmt, 0)
    if code == 0xFFFE and len(fmt) >= 26:                       # WAVE_FORMAT_EXTENSIBLE: real tag in the GUID
        code = struct.unpack_from("<H", fmt, 24)[0]
    return code, channels, rate, bits, data


def read_wav_raw(path: str | Path) -> Tuple[np.ndarray, int, int]:
    """(samples [n, channels] in the file's own dtype, sample_rate, format tag) of a WAV file."""
    code, channels, rate, bits, data = _wav_chunks(path)
    if code == 1 and bits == 16:
        x = np.frombuffer(data, dtype="<i2")
    elif code == 1 and bits == 8:
        x = np.frombuffer(data, dtype=np.uint8)
    elif code == 1 and bits == 32:
        x = np.frombuffer(data, dtype="<i4")
    elif code == 1 and bits == 24:
        b = np.frombuffer(data[: len(data) // 3 * 3], dtype=np.uint8).reshape(-1, 3).astype(np.int32)
        x = (b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16))
        x = np.where(x & 0x800000, x - (1 << 24), x).astype(np.int32)
    elif code == 3 and bits in (32, 64):
        x = np.frombuffer(data, dtype="<f4" if bits == 32 else "<f8")
    else:
        raise ValueError(f"{path}: unsupported WAV encoding (format {code}, {bits} bits)")
    n = x.size // channels
    return x[: n * channels].reshape(n, channels), int(rate), (code << 8) | bits


def read_wav(path: str | Path) -> Tuple[np.ndarray, int]:
    """float32 samples in [-1, 1) like soundfile.read(dtype="float32"): integer PCM divided by 2^(bits-1)."""
    x, rate, tag = read_wav_raw(path)
    code, bits = tag >> 8, tag & 0xFF
    if code == 3:
        y = x.astype(np.float32)
    elif bits == 8:
        y = (x.astype(np.float32) - 128.0) / 128.0
    else:
        y = (x.astype(np.float64) / float(1 << (bits - 1))).astype(np.float32)
    return (y[:, 0] if y.shape[1] == 1 else y), rate


# (format code, bits) -> (dtype code of include/dspx.h, bytes per sample)
_DEVICE_ENCODINGS = {(1, 8): (3, 1), (1, 16): (2, 2), (1, 24): (4, 3), (1, 32): (5, 4), (3, 32): (0, 4), (3, 64): (1, 8)}
MAX_DEVICE_CHANNELS = 32


def read_wav_data(path: str | Path) -> Tuple[np.ndarray, int, int, int, int] | None:
    """(data chunk as uint8, sample_rate, channels, dtype code, n_frames) with no conversion, for the device decoder.

    The dtype code is one of include/dspx.h's DSPX_DTYPE_PCM8 / PCM16 / PCM24 / PCM32 / F32 / F64.  n_frames follows
    read_wav_raw: whole samples, then whole frames, and the bytes returned are exactly those frames.  None when the
    file is not a WAV file of one of those six encodings with 1 to 32 channels.
    """
    try:
        code, channels, rate, bits, data = _wav_chunks(path)
    except (ValueError, struct.error):
        return None
    enc = _DEVICE_ENCODINGS.get((code, bits))
    if enc is None or not 1 <= channels <= MAX_DEVICE_CHANNELS:
        return None
    dtype, size = enc
    n_frames = len(data) // size // channels
    return np.frombuffer(data, np.uint8, n_frames * channels * size), int(rate), int(channels), dtype, n_frames


def _is_flac(path: str | Path) -> bool:
    """Whether the file is a native FLAC stream ("fLaC" after an optional ID3v2 tag), from its first bytes only."""
    with open(path, "rb") as f:
        head = f.read(10)
        pos = 0
        if len(head) == 10 and head[:3] == b"ID3":
            pos = 10 + (head[6] << 21 | head[7] << 14 | head[8] << 7 | head[9]) + (10 if head[5] & 0x10 else 0)
        f.seek(pos)
        return f.read(4) == b"fLaC"


def read_flac_data(path: str | Path) -> Tuple[np.ndarray, int, int, int, int, tuple] | None:
    """(the file's bytes as uint8, sample_rate, channels, DTYPE_FLAC, samples per channel, (file row, frame table)) for
    the device decoder, or None when the file is not a native FLAC stream (judged by its content, not its name).

    The stream is parsed and its frames found on the host once (batch.flac_parse: dspx_flac_layout, no device
    needed); decode_packed reuses those tables.  A FLAC file that does not parse raises batch.FlacError (a ValueError)
    naming it and the byte offset of the problem.
    """
    from . import _lib
    from .batch import flac_parse

    if not _is_flac(path):
        return None
    data = np.fromfile(path, np.uint8)
    row, frames = flac_parse(data, str(path))
    return data, int(row["sample_rate"]), int(row["channels"]), _lib.DTYPE_FLAC, int(row["out_length"]), (row, frames)


def load_audio(path: str | Path, target_sr: int | None = None) -> Tuple[np.ndarray, int]:
    """src/utils/audio.py:19-31: decode, average channels, resample when the rates differ.

    Without soundfile, a FLAC file is decoded, downmixed and resampled on the GPU (batch.decode_packed), which gives
    the same bits; there is no CPU decoder for it, so without a device that raises."""
    path = Path(path)
    if _sf is not None:
        audio, sr = _sf.read(path, dtype="float32")
    else:
        flac = read_flac_data(path)
        if flac is not None:
            from .batch import decode_packed

            target = None if target_sr is None else int(target_sr)
            packed = decode_packed([flac], target, False, names=[str(path)])
            audio = packed.samples[int(packed.starts[0]):int(packed.starts[0] + packed.lengths[0])].cpu().numpy()
            return audio, flac[1] if target is None else target
        audio, sr = read_wav(path)
    if audio.ndim > 1:
        audio = np.mean(audio, axis=1)
    if target_sr is not None and sr != target_sr:
        from scipy.signal import resample_poly                  # same resampler as the reference

        audio = resample_poly(audio, target_sr, sr)
        sr = target_sr
    return audio.astype(np.float32), sr


def normalize_audio(audio: np.ndarray) -> np.ndarray:
    """src/utils/audio.py:34-38."""
    peak = np.max(np.abs(audio)) if audio.size else 0.0
    return audio / peak if peak > 0 else audio


def load_pcm16(path: str | Path, target_sr: int | None = None) -> np.ndarray | None:
    """The file's int16 samples when it is mono 16-bit PCM at `target_sr` (the ESC-50 case), else None.

    Such clips can skip the host-side float conversion altogether: features_batch() takes int16 and
    converts / peak-normalises on the GPU, bit-identically to load_audio + normalize_audio.
    """
    try:
        x, rate, tag = read_wav_raw(path)
    except ValueError:
        return None
    if tag != ((1 << 8) | 16) or x.shape[1] != 1 or (target_sr is not None and rate != target_sr):
        return None
    return np.ascontiguousarray(x[:, 0])


def read_pcm16(path: str | Path) -> Tuple[np.ndarray, int] | None:
    """(int16 samples, sample_rate) when the file is mono 16-bit PCM at any rate, else None.

    Clips at another rate than the config's can still take the GPU path: features_batch(..., sample_rate=rate)
    resamples them on the device, bit-identically to load_audio's resample_poly.
    """
    try:
        x, rate, tag = read_wav_raw(path)
    except ValueError:
        return None
    if tag != ((1 << 8) | 16) or x.shape[1] != 1:
        return None
    return np.ascontiguousarray(x[:, 0]), rate
