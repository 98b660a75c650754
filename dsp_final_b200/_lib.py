"""ctypes binding of libdspx.so (include/dspx.h).

This is the only place the package touches native code.  There is no CPU
implementation behind it: if the library is missing, or the machine has no
CUDA device, the compute entry points raise -- loudly -- instead of falling
back (BASELINE.json north_star: "no multi-backend dispatch and no CPU
fallback").
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "_native" / "libdspx.so"

OK, EINVAL, ENOMEM, ECUDA, ENODEVICE, EUNSUPPORTED = 0, -1, -2, -3, -4, -5
WINDOWS = {"hann": 0, "hamming": 1, "rect": 2}
KERNELS = {"auto": 0, "generic": 1, "warp8": 2}
KERNEL_NAMES = {v: k for k, v in KERNELS.items()}
DTYPE_F32, DTYPE_F64, DTYPE_PCM16 = 0, 1, 2
DTYPE_PCM8, DTYPE_PCM24, DTYPE_PCM32 = 3, 4, 5
MAX_CHANNELS = 32
DTYPE_FLAC = 6                  # a FLAC stream: read_flac_data's dtype code (not a dspx.h sample type)
MAX_K = 128


class DspxConfig(C.Structure):
    """struct dspx_config: image of the reference MfccConfig (src/dsp/mfcc.py:10-21)."""

    _fields_ = [
        ("sample_rate", C.c_int32),
        ("frame_length", C.c_int32),
        ("hop_length", C.c_int32),
        ("n_fft", C.c_int32),
        ("n_mels", C.c_int32),
        ("n_mfcc", C.c_int32),
        ("f_min", C.c_double),
        ("f_max", C.c_double),
        ("pre_emphasis", C.c_double),
        ("window", C.c_int32),
        ("kernel", C.c_int32),
    ]


class DspxPlanInfo(C.Structure):
    _fields_ = [
        ("n_fft_pow2", C.c_int32),
        ("n_bins", C.c_int32),
        ("take_features", C.c_int32),
        ("take_stft", C.c_int32),
        ("mel_nnz", C.c_int32),
        ("kernel", C.c_int32),
        ("device", C.c_int32),
        ("sm_count", C.c_int32),
    ]


class DspxRaggedClip(C.Structure):
    """struct dspx_ragged_clip: one row of a ragged batch's table (dspx_ragged_layout)."""

    _fields_ = [
        ("start", C.c_int64),
        ("length", C.c_int64),
        ("n_frames", C.c_int64),
        ("first_frame", C.c_int64),
        ("first_pair", C.c_int64),
    ]


class DspxError(RuntimeError):
    pass


_lib = None

_VP, _I64, _I32, _SZ = C.c_void_p, C.c_int64, C.c_int, C.c_size_t
_SIGNATURES = {
    "dspx_version": (C.c_char_p, []),
    "dspx_last_error": (C.c_char_p, []),
    "dspx_device_count": (_I32, []),
    "dspx_plan_create": (_I32, [C.POINTER(DspxConfig), _I32, C.POINTER(_VP)]),
    "dspx_plan_destroy": (_I32, [_VP]),
    "dspx_plan_get_info": (_I32, [_VP, C.POINTER(DspxPlanInfo)]),
    "dspx_num_frames": (_I64, [_VP, _I64]),
    "dspx_plan_read_table": (_I32, [_VP, _I32, _VP, _I64]),
    "dspx_stft": (_I32, [_VP, _VP, _I64, _I64, _I64, _I32, _VP, _VP]),
    "dspx_features": (_I32, [_VP, _VP, _I64, _I64, _I64, _VP, _VP, _VP, _VP]),
    "dspx_embeddings_workspace": (_SZ, [_VP, _I64]),
    "dspx_embeddings": (_I32, [_VP, _VP, _I64, _I64, _I64, _VP, _VP, _VP, _SZ, _VP]),
    "dspx_log_mel_nchw": (_I32, [_VP, _VP, _I64, _I64, _I64, _VP, _VP]),
    "dspx_embed_stats": (_I32, [_VP, _I64, _I64, _I32, _VP, _VP]),
    "dspx_cmvn": (_I32, [_VP, _I64, _I64, _I32, C.c_double, _VP]),
    "dspx_features_host": (_I32, [_VP, _VP, _I64, _I64, _I64, _VP, _VP, _VP]),
    "dspx_pcm16_to_float": (_I32, [_VP, _I64, _I64, _I64, _I32, _VP, _I64, _VP]),
    "dspx_features_pcm16_workspace": (_SZ, [_I64]),
    "dspx_features_pcm16": (_I32, [_VP, _VP, _I64, _I64, _I64, _I32, _VP, _VP, _VP, _VP, _SZ, _VP]),
    "dspx_features_host_pcm16": (_I32, [_VP, _VP, _I64, _I64, _I64, _I32, _VP, _VP, _VP]),
    "dspx_stft_host": (_I32, [_VP, _VP, _I64, _I64, _I64, _I32, _VP]),
    "dspx_ragged_layout": (_I64, [C.POINTER(DspxConfig), _VP, _VP, _I64, _I32, _VP]),
    "dspx_features_ragged_workspace": (_SZ, [_VP, _VP, _I64, _I32, _I32, _I32, _I32, _I32]),
    "dspx_features_ragged": (_I32, [_VP, _VP, _I32, _I32, _VP, _VP, _I64, _I64, _VP, _VP, _VP, _VP, _SZ, _VP]),
    "dspx_embed_stats_ragged": (_I32, [_VP, _VP, _I64, _I32, _VP, _VP]),
    "dspx_resampler_create": (_I32, [_I64, _I64, _VP, _I64, _I32, C.POINTER(_VP)]),
    "dspx_resampler_destroy": (_I32, [_VP]),
    "dspx_resample_len": (_I64, [_VP, _I64]),
    "dspx_resample_workspace": (_SZ, [_I64]),
    "dspx_resample": (_I32, [_VP, _VP, _I32, _I64, _I64, _I64, _I32, _VP, _I64, _VP, _SZ, _VP]),
    "dspx_resample_layout": (_I64, [_I64, _I64, _VP, _VP, _I64, _VP]),
    "dspx_resample_ragged": (_I32, [_VP, _VP, _I32, _I32, _VP, _VP, _I64, _VP, _VP, _SZ, _VP]),
    "dspx_decode_layout": (_I64, [_VP, _VP, _VP, _VP, _I64, _VP]),
    "dspx_decode_workspace": (_SZ, [_I64]),
    "dspx_decode_ragged": (_I32, [_VP, _VP, _VP, _I64, _I32, _VP, _VP, _SZ, _VP]),
    "dspx_flac_layout": (_I64, [_VP, _VP, _VP, _I64, _VP, _VP, _I64, _VP]),
    "dspx_flac_workspace": (_SZ, [_VP, _I64]),
    "dspx_flac_decode": (_I32, [_VP, _VP, _VP, _I64, _VP, _VP, _I64, _I32, _VP, _VP, _VP, _SZ, _VP]),
    "dspx_next_pow_two": (_I64, [_I64]),
    "dspx_fft_c2c": (_I32, [_VP, _I64, _I64, _I64, _I32, _VP, _VP, _VP]),
    "dspx_cosine_topk_workspace": (_SZ, [_I64, _I64, _I32, _I32]),
    "dspx_cosine_topk": (_I32, [_VP, _I64, _VP, _I64, _I32, _I32, _I32, _VP, _VP, _VP, _SZ, _VP]),
    "dspx_cosine_matrix": (_I32, [_VP, _I64, _VP, _I64, _I32, _I32, _VP, _VP, _SZ, _VP]),
    "dspx_dct2": (_I32, [_VP, _I64, _I32, _I32, _VP, _VP]),
    "dspx_hits_at_k": (_I32, [_VP, _I64, _I32, _I32, _VP, _VP, _VP, _VP]),
}


def load() -> C.CDLL:
    """Load libdspx.so or raise ImportError; never substitutes another backend."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("DSPX_LIBRARY", LIB_PATH))
    if not path.exists():
        raise ImportError(
            f"{path} not found. Build it with `python -m dsp_final_b200.build` "
            "(nvcc, sm_100a). dsp_final_b200 has no CPU fallback."
        )
    lib = C.CDLL(str(path))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError here = ABI drift; do not mask it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().dspx_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "libdspx call") -> int:
    """Map a DSPX_E* code onto the exception the reference raises for that case."""
    if rc >= 0:
        return rc
    msg = f"{what}: {last_error()}"
    if rc == EINVAL:
        raise ValueError(msg)          # stft.py:15-16,24,29-30 raise ValueError on bad arguments
    if rc == ENOMEM:
        raise MemoryError(msg)
    if rc == ENODEVICE:
        raise DspxError(msg + " (a CUDA device is required; there is no CPU fallback)")
    if rc == EUNSUPPORTED:
        raise NotImplementedError(msg)
    raise DspxError(msg)


def device_count() -> int:
    return int(load().dspx_device_count())


def require_device() -> None:
    if device_count() <= 0:
        raise DspxError("no CUDA device visible: dsp_final_b200 computes on the GPU only (no CPU fallback)")
