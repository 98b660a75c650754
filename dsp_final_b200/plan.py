"""Plan cache: one immutable dspx_plan (device constant tables) per config and device.

The reference caches its tables with functools.lru_cache (src/dsp/stft.py:12,
src/dsp/mfcc.py:61,79); MfccConfig is an unfrozen dataclass and therefore
unhashable, so plans are keyed on the tuple of its fields instead.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import Any

import numpy as np

from . import _lib

_plans: dict[tuple, "Plan"] = {}
_lock = threading.Lock()


def _field(cfg: Any, name: str, default=None):
    if isinstance(cfg, dict):
        return cfg.get(name, default)
    return getattr(cfg, name, default)


def config_key(cfg: Any) -> tuple:
    window = _field(cfg, "window", "hann")
    if window not in _lib.WINDOWS:
        raise ValueError(f"Unsupported window: {window}")          # stft.py:24
    n_fft = _field(cfg, "n_fft")
    f_max = _field(cfg, "f_max")
    return (
        int(_field(cfg, "sample_rate")), int(_field(cfg, "frame_length")), int(_field(cfg, "hop_length")),
        int(n_fft) if n_fft else 0, int(_field(cfg, "n_mels", 40)), int(_field(cfg, "n_mfcc", 13)),
        float(_field(cfg, "f_min", 0.0)), -1.0 if f_max is None else float(f_max),
        float(_field(cfg, "pre_emphasis", 0.97)), window,
    )


def config_struct(key: tuple, kernel: str = "auto") -> _lib.DspxConfig:
    """struct dspx_config of a config_key tuple."""
    sr, fl, hop, n_fft, n_mels, n_mfcc, f_min, f_max, pre, window = key
    return _lib.DspxConfig(sr, fl, hop, n_fft, n_mels, n_mfcc, f_min, f_max, pre, _lib.WINDOWS[window], _lib.KERNELS[kernel])


def current_device() -> int:
    """The CUDA device of this process (torch's current device when torch has CUDA up)."""
    try:
        import torch

        if torch.cuda.is_available():
            return int(torch.cuda.current_device())
    except ImportError:                                             # pragma: no cover
        pass
    return 0


class Plan:
    """Owns a dspx_plan*.  Immutable after creation; safe to share between threads."""

    def __init__(self, key: tuple, device: int, kernel: str = "auto"):
        lib = _lib.load()
        _lib.require_device()
        sr, fl, hop, n_fft, n_mels, n_mfcc, f_min, f_max, pre, window = key
        if fl <= 0 or hop <= 0:
            raise ValueError("frame_length and hop_length must be positive")   # stft.py:29-30
        self.key, self.device, self.kernel_request = key, device, kernel
        c = config_struct(key, kernel)
        handle = C.c_void_p()
        _lib.check(lib.dspx_plan_create(C.byref(c), device, C.byref(handle)), "dspx_plan_create")
        self._h = handle
        info = _lib.DspxPlanInfo()
        _lib.check(lib.dspx_plan_get_info(self._h, C.byref(info)), "dspx_plan_get_info")
        self.n_fft = int(info.n_fft_pow2)
        self.n_bins = int(info.n_bins)
        self.mel_nnz = int(info.mel_nnz)
        self.kernel = _lib.KERNEL_NAMES.get(int(info.kernel), str(info.kernel))
        self.sm_count = int(info.sm_count)
        self.frame_length, self.hop_length, self.n_mels, self.n_mfcc = fl, hop, n_mels, n_mfcc

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def num_frames(self, clip_len: int) -> int:
        t = int(_lib.load().dspx_num_frames(self._h, int(clip_len)))
        _lib.check(t, "dspx_num_frames")
        return t

    def read_table(self, which: str) -> np.ndarray:
        shapes = {"window": (0, (self.frame_length,)), "fbank": (1, (self.n_mels, self.n_bins)),
                  "dct2": (2, (self.n_mfcc, self.n_mels))}
        idx, shape = shapes[which]
        out = np.empty(shape, np.float32)
        _lib.check(_lib.load().dspx_plan_read_table(self._h, idx, out.ctypes.data, out.size), "dspx_plan_read_table")
        return out

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.load().dspx_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):                                               # best effort
        try:
            self.close()
        except Exception:
            pass


def get_plan(cfg: Any, device: int | None = None, kernel: str = "auto") -> Plan:
    dev = current_device() if device is None else int(device)
    key = (config_key(cfg), dev, kernel)
    with _lock:
        plan = _plans.get(key)
        if plan is None:
            plan = Plan(key[0], dev, kernel)
            _plans[key] = plan
        return plan


def clear_plans() -> None:
    with _lock:
        for p in _plans.values():
            p.close()
        _plans.clear()
