"""Batched entry points: many clips per call, on the device or from host buffers.

The reference computes one clip per Python call (src/features/cache.py:65-74,
scripts/tools/precompute_features.py:96-107 fans clips out to processes).  One
call per 5 s of audio cannot feed a B200, so the batched forms below are the
throughput API; the per-clip functions in dsp_final_b200.dsp are thin wrappers
over them and keep the reference signatures.

  * torch CUDA tensor in  -> torch CUDA tensors out, enqueued on torch's current
    stream through the device-pointer C ABI (dspx_features / dspx_stft);
  * NumPy array (or CPU tensor) in -> NumPy arrays out through the host-buffer
    C ABI (dspx_features_host / dspx_stft_host: pinned staging + copy/compute
    overlap inside the library).

features_ragged takes clips of different lengths in one call (dspx_features_ragged):
outputs are stacked along the frame axis and split per clip with "frame_offsets".

resample_poly is scipy.signal.resample_poly on the GPU, bit for bit (dspx_resample).  With sample_rate= the
clips' own rate, features_batch and features_ragged resample on the device first when it differs from
cfg.sample_rate (src/utils/audio.py:27-30 resamples on the host there).

load_audio_batch is load_audio (+ normalize_audio) for many WAV and FLAC files at once: the WAV data chunks and the
FLAC files go to the GPU as stored and are decoded, downmixed and resampled there, bit for bit (dspx_decode_ragged,
dspx_flac_decode, dspx_resample_ragged).
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Iterable, NamedTuple

import numpy as np

from . import _lib
from .plan import Plan, Resampler, config_key, config_struct, get_plan, get_resampler, reduce_ratio

FEATURES = ("log_mel", "mfcc", "embed")


def _is_cuda_tensor(x) -> bool:
    return type(x).__module__.startswith("torch") and getattr(x, "is_cuda", False)


def _as_host_clips(clips) -> np.ndarray:
    if type(clips).__module__.startswith("torch"):
        clips = clips.detach().cpu().numpy()
    a = np.asarray(clips)
    if a.ndim == 1:
        a = a[None, :]
    if a.ndim != 2:
        raise ValueError("clips must be [n_clips, n_samples]")
    if a.dtype != np.float32 or a.strides[1] != 4 or a.strides[0] % 4 or a.strides[0] < 4 * a.shape[1]:
        a = np.ascontiguousarray(a, dtype=np.float32)      # also normalises the 0 stride of a[None, :]
    return a


def _want(want: Iterable[str]) -> tuple[str, ...]:
    w = tuple(want)
    for name in w:
        if name not in FEATURES:
            raise ValueError(f"Unsupported feature_type: {name}")      # cache.py:73
    if not w:
        raise ValueError("no output requested")
    return w


def _is_pcm16(clips) -> bool:
    dt = getattr(clips, "dtype", None)
    return dt is not None and str(dt) in ("int16", "torch.int16")


def _ran(rc: int, what: str) -> bool:
    """False when the entry point does not apply (DSPX_EUNSUPPORTED, nothing enqueued); raises on any other error."""
    return rc != _lib.EUNSUPPORTED and _lib.check(rc, what) >= 0


def pcm16_to_float(pcm, normalize: bool = True):
    """int16 PCM [B, L] on the GPU -> float32 [B, L]: x/32768, then x/max|x| (src/utils/audio.py:19-38)."""
    import torch

    _lib.require_device()
    x = pcm if pcm.dim() == 2 else pcm[None, :]
    if x.stride(1) != 1:
        x = x.contiguous()
    dev = x.device.index
    with torch.cuda.device(dev):
        out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().dspx_pcm16_to_float(x.data_ptr(), x.shape[0], x.shape[1], x.stride(0),
                                                   1 if normalize else 0, out.data_ptr(), out.stride(0),
                                                   torch.cuda.current_stream(dev).cuda_stream), "dspx_pcm16_to_float")
    return out


def _resample_dtype(x) -> bool:
    """True for int16 PCM, False for float32; ValueError for anything else (scipy would filter float64 in float64)."""
    if _is_pcm16(x):
        return True
    if str(getattr(x, "dtype", None)) not in ("float32", "torch.float32"):
        raise ValueError(f"resample_poly takes float32 or int16 samples, not {getattr(x, 'dtype', type(x).__name__)}")
    return False


def _resample_2d(x, rs: Resampler, normalize: bool):
    """[B, L] torch CUDA float32 / int16 (unit stride) -> [B, n_out] float32 on torch's current stream."""
    import torch

    lib = _lib.load()
    pcm = _is_pcm16(x)
    b, n_in = x.shape
    if n_in < 1:
        raise ValueError("resample_poly of an empty clip")
    n_out = rs.out_len(n_in)
    dev = x.device.index
    with torch.cuda.device(dev):
        out = torch.empty((b, n_out), dtype=torch.float32, device=x.device)
        ws_bytes = int(lib.dspx_resample_workspace(b))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        _lib.check(lib.dspx_resample(rs.handle, x.data_ptr(), _lib.DTYPE_PCM16 if pcm else _lib.DTYPE_F32, b, n_in,
                                     x.stride(0), 1 if normalize else 0, out.data_ptr(), n_out, ws.data_ptr(), ws_bytes,
                                     torch.cuda.current_stream(dev).cuda_stream), "dspx_resample")
    return out


def _resample_ragged(xs: list, rs: Resampler, normalize: bool):
    """1-D torch CUDA clips of one dtype -> (packed float32 output, table int64 [n, 4]): one launch.  Clip i is
    out[table[i, 2]:table[i, 2] + table[i, 3]]; starts are multiples of RAGGED_ALIGN and the gaps are zero."""
    import torch

    lib = _lib.load()
    pcm = _is_pcm16(xs[0])
    lengths = np.array([len(x) for x in xs], np.int64)
    starts = np.concatenate(([0], np.cumsum(lengths)[:-1])).astype(np.int64)
    table = np.zeros((len(xs), 4), np.int64)
    total = _lib.check(int(lib.dspx_resample_layout(rs.up, rs.down, starts.ctypes.data, lengths.ctypes.data, len(xs),
                                                    table.ctypes.data)), "dspx_resample_layout")
    dev = xs[0].device
    with torch.cuda.device(dev.index):
        samples = torch.cat(xs)
        table_dev = torch.from_numpy(table).to(dev)
        out = torch.zeros(total, dtype=torch.float32, device=dev)
        ws_bytes = int(lib.dspx_resample_workspace(len(xs)))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.dspx_resample_ragged(rs.handle, samples.data_ptr(), _lib.DTYPE_PCM16 if pcm else _lib.DTYPE_F32,
                                            1 if normalize else 0, table_dev.data_ptr(), table.ctypes.data, len(xs),
                                            out.data_ptr(), ws.data_ptr(), ws_bytes,
                                            torch.cuda.current_stream(dev.index).cuda_stream), "dspx_resample_ragged")
    return out, table


def _to_device(x, device: int | None):
    """A torch CUDA tensor as it is; NumPy (or a CPU tensor) uploaded with torch to `device` (default: current)."""
    import torch

    if _is_cuda_tensor(x):
        return x
    if type(x).__module__.startswith("torch"):
        x = x.detach().numpy()
    dev = torch.cuda.current_device() if device is None else int(device)
    x = np.ascontiguousarray(x)
    if not x.flags.writeable:                  # decoded WAV data is a read-only view; torch.from_numpy wants writable
        x = x.copy()
    return torch.from_numpy(x).to(torch.device("cuda", dev))


def resample_poly(x, up: int, down: int, normalize: bool = False, device: int | None = None):
    """scipy.signal.resample_poly(x, up, down) with its default filter, on the GPU, bit for bit.

    x: a 1-D array, a [B, L] array (each row resampled) or a list of 1-D arrays of any lengths (one launch), as
    NumPy or torch CUDA, float32 or int16 PCM (read as int16 / 32768, what load_audio decodes).  The result comes
    back float32 in the same kind of container.  normalize=True then divides each clip by its peak, like
    normalize_audio.  Other dtypes raise ValueError: scipy filters float64 in float64, which this does not do.
    """
    up, down = reduce_ratio(up, down)
    if isinstance(x, (list, tuple)):
        if not x:
            return []
        on_gpu = [_is_cuda_tensor(c) for c in x]
        if any(on_gpu) and not all(on_gpu):
            raise ValueError("clips must be all NumPy arrays or all torch CUDA tensors")
        if len({_resample_dtype(c) for c in x}) > 1:
            raise ValueError("clips must all be float32 or all be int16 PCM")
        _lib.require_device()
        xs = [_to_device(c, device).reshape(-1) for c in x]
        if any(len(c) < 1 for c in xs):
            raise ValueError("resample_poly of an empty clip")
        if len({c.device for c in xs}) > 1:
            raise ValueError("clips must be on one device")
        out, table = _resample_ragged(xs, get_resampler(up, down, xs[0].device.index), normalize)
        if all(on_gpu):
            return [out[s:s + n] for s, n in zip(table[:, 2], table[:, 3])]
        host = out.cpu().numpy()
        return [host[s:s + n].copy() for s, n in zip(table[:, 2], table[:, 3])]
    _resample_dtype(x)
    if len(getattr(x, "shape", ())) not in (1, 2):
        raise ValueError("resample_poly takes a 1-D array, a [B, L] array or a list of 1-D arrays")
    _lib.require_device()
    on_gpu = _is_cuda_tensor(x)
    t = _to_device(x, device)
    t2 = t if t.dim() == 2 else t[None, :]
    if t2.stride(1) != 1:
        t2 = t2.contiguous()
    out = _resample_2d(t2, get_resampler(up, down, t2.device.index), normalize)
    out = out if t.dim() == 2 else out[0]
    return out if on_gpu else out.cpu().numpy()


def _resample_ratio(cfg: Any, sample_rate) -> tuple[int, int] | None:
    """(up, down) from the clips' rate to cfg.sample_rate, or None when no rate is given or the two are equal."""
    if sample_rate is None or int(sample_rate) == config_key(cfg)[0]:
        return None
    return reduce_ratio(config_key(cfg)[0], int(sample_rate))


def _features_resampled(clips, cfg: Any, want, device, kernel: str, normalize: bool, ratio) -> dict:
    """features_batch of clips at another rate: resampled on the device first, PCM16 peak-normalised after the
    resample when `normalize` (the reference's order: load_audio, then normalize_audio)."""
    on_gpu = _is_cuda_tensor(clips)
    pcm = _resample_dtype(clips)
    t = _to_device(clips, device)
    t = t if t.dim() == 2 else t[None, :]
    if t.stride(1) != 1:
        t = t.contiguous()
    y = _resample_2d(t, get_resampler(*ratio, t.device.index), normalize and pcm)
    out = features_batch(y, cfg, want, device, kernel, normalize)
    return out if on_gpu else _as_host(out)


def _as_host(out: dict) -> dict:
    return {k: (v.cpu().numpy() if _is_cuda_tensor(v) else v) for k, v in out.items()}


def features_batch(clips, cfg: Any, want: Iterable[str] = ("mfcc",), device: int | None = None,
                   kernel: str = "auto", normalize: bool = True, sample_rate: int | None = None) -> dict:
    """log-mel / MFCC / clip embeddings of a batch of equal-length clips.

    Follows src/dsp/mfcc.py:86-109 (+ src/retrieval/retrieval.py:19-23 for "embed").
    Returns {"log_mel": [B,T,n_mels], "mfcc": [B,T,n_mfcc], "embed": [B,2*n_mfcc]} (float32)
    restricted to `want`.  int16 input is taken as PCM16 and converted on the GPU like
    load_audio (+ normalize_audio when `normalize`), src/utils/audio.py:19-38, cache.py:66-67.
    `sample_rate`: the clips' own rate.  When it differs from cfg.sample_rate the clips are first resampled on the
    GPU, bit-identically to load_audio's scipy.signal.resample_poly (int16 PCM is normalised after the resample);
    NumPy input is uploaded with torch.  float32 or int16 clips only on that path.
    """
    want = _want(want)
    ratio = _resample_ratio(cfg, sample_rate)
    if ratio is not None:
        return _features_resampled(clips, cfg, want, device, kernel, normalize, ratio)
    lib = _lib.load()
    if _is_cuda_tensor(clips):
        import torch

        x = clips if clips.dim() == 2 else clips[None, :]
        pcm = _is_pcm16(x)
        if pcm:
            x = x if x.stride(1) == 1 else x.contiguous()
        elif x.dtype != torch.float32 or x.stride(1) != 1:
            x = x.to(torch.float32).contiguous()
        dev = x.device.index if device is None else device
        plan = get_plan(cfg, dev, kernel)
        b, length = x.shape
        t = plan.num_frames(length)

        def new(*shape):
            return torch.empty(shape, dtype=torch.float32, device=x.device)

        def ptr(a):
            return a.data_ptr() if a is not None else None

        # The fused entry points return DSPX_EUNSUPPORTED, having enqueued nothing, where they do not apply (plan, batch
        # size, alignment); dspx_features then computes the same values through an MFCC tensor.
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            lm = new(b, t, plan.n_mels) if "log_mel" in want else None
            mf = new(b, t, plan.n_mfcc) if "mfcc" in want else None
            em = new(b, 2 * plan.n_mfcc) if "embed" in want else None
            done = False
            if pcm:
                # conversion and peak normalisation inside the feature kernel's loads: no float32 copy of the clips
                if em is not None and mf is None:
                    mf = new(b, t, plan.n_mfcc)
                ws_bytes = int(lib.dspx_features_pcm16_workspace(b))
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
                done = _ran(lib.dspx_features_pcm16(plan.handle, x.data_ptr(), b, length, x.stride(0), 1 if normalize else 0,
                                                    ptr(lm), ptr(mf), ptr(em), ws.data_ptr(), ws_bytes, stream),
                            "dspx_features_pcm16")
                if not done:
                    x = pcm16_to_float(x, normalize)
            elif em is not None and mf is None:
                # embeddings without MFCCs: accumulated inside the feature kernel (no [B, T, n_mfcc] tensor at all)
                ws_bytes = int(lib.dspx_embeddings_workspace(plan.handle, b))
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
                done = _ran(lib.dspx_embeddings(plan.handle, x.data_ptr(), b, length, x.stride(0), em.data_ptr(), ptr(lm),
                                                ws.data_ptr(), ws_bytes, stream), "dspx_embeddings")
            if not done:
                if em is not None and mf is None:
                    mf = new(b, t, plan.n_mfcc)
                _lib.check(lib.dspx_features(plan.handle, x.data_ptr(), b, length, x.stride(0), ptr(lm), ptr(mf), ptr(em),
                                             stream), "dspx_features")
        out = {}
        if lm is not None:
            out["log_mel"] = lm
        if "mfcc" in want:
            out["mfcc"] = mf
        if em is not None:
            out["embed"] = em
        return out

    pcm = _is_pcm16(clips)
    if pcm:
        x = np.asarray(clips.numpy() if type(clips).__module__.startswith("torch") else clips)
        x = x[None, :] if x.ndim == 1 else x
        if x.strides[1] != 2 or x.strides[0] < 2 * x.shape[1] or x.strides[0] % 2:
            x = np.ascontiguousarray(x)
    else:
        x = _as_host_clips(clips)
    plan = get_plan(cfg, device, kernel)
    b, length = x.shape
    t = plan.num_frames(length)
    lm = np.empty((b, t, plan.n_mels), np.float32) if "log_mel" in want else None
    mf = np.empty((b, t, plan.n_mfcc), np.float32) if "mfcc" in want else None
    em = np.empty((b, 2 * plan.n_mfcc), np.float32) if "embed" in want else None
    outs = (lm.ctypes.data if lm is not None else None, mf.ctypes.data if mf is not None else None,
            em.ctypes.data if em is not None else None)
    if pcm:
        _lib.check(lib.dspx_features_host_pcm16(plan.handle, x.ctypes.data, b, length, max(x.strides[0] // 2, length),
                                                1 if normalize else 0, *outs), "dspx_features_host_pcm16")
    else:
        _lib.check(lib.dspx_features_host(plan.handle, x.ctypes.data, b, length, max(x.strides[0] // 4, length),
                                          *outs), "dspx_features_host")
    out = {}
    if lm is not None:
        out["log_mel"] = lm
    if mf is not None:
        out["mfcc"] = mf
    if em is not None:
        out["embed"] = em
    return out


RAGGED_ALIGN = 4       # samples: clip starts in the packed buffer (float32 needs even ones; 4 keeps 16-byte alignment)


def ragged_layout(lengths, cfg, dtype=np.float32, starts=None) -> tuple[np.ndarray, np.ndarray, int]:
    """(starts, table, total_frames) of a ragged batch: dspx_ragged_layout on the host, no device needed.

    `starts` defaults to the clips packed back to back at multiples of RAGGED_ALIGN samples.  table is int64
    [n_clips, 5], the rows of struct dspx_ragged_clip: start, length, n_frames, first_frame, first_pair.
    """
    lengths = np.ascontiguousarray(lengths, dtype=np.int64).reshape(-1)
    if starts is None:
        padded = (lengths + RAGGED_ALIGN - 1) // RAGGED_ALIGN * RAGGED_ALIGN
        starts = np.concatenate(([0], np.cumsum(padded)[:-1])).astype(np.int64) if len(lengths) else lengths.copy()
    starts = np.ascontiguousarray(starts, dtype=np.int64).reshape(-1)
    if starts.shape != lengths.shape:
        raise ValueError("one start per clip expected")
    code = _lib.DTYPE_PCM16 if np.dtype(dtype) == np.int16 else _lib.DTYPE_F32
    table = np.zeros((len(lengths), 5), np.int64)
    c = config_struct(config_key(cfg))
    total = _lib.check(_lib.load().dspx_ragged_layout(C.byref(c), starts.ctypes.data, lengths.ctypes.data, len(lengths),
                                                      code, table.ctypes.data), "dspx_ragged_layout")
    return starts, table, int(total)


def _ragged_inputs(clips) -> tuple[list, bool, bool]:
    """-> (1-D clips, on the GPU, PCM16); all NumPy float32 / int16, or all torch CUDA tensors of one dtype."""
    clips = list(clips)
    cuda = [_is_cuda_tensor(c) for c in clips]
    if any(cuda) and not all(cuda):
        raise ValueError("clips must be all NumPy arrays or all torch CUDA tensors")
    pcm = [_is_pcm16(c) for c in clips]
    if any(pcm) and not all(pcm):
        raise ValueError("clips must all be float or all be int16 PCM")
    on_gpu, is_pcm = bool(clips) and all(cuda), bool(clips) and all(pcm)
    if on_gpu:
        import torch

        dt = torch.int16 if is_pcm else torch.float32
        out = [c.reshape(-1).to(dt) for c in clips]
        if len({c.device for c in out}) > 1:
            raise ValueError("clips must be on one device")
    else:
        if clips and type(clips[0]).__module__.startswith("torch"):
            clips = [c.detach().cpu().numpy() for c in clips]
        out = [np.asarray(c, dtype=np.int16 if is_pcm else np.float32).reshape(-1) for c in clips]
    return out, on_gpu, is_pcm


def ragged_launch(plan: Plan, samples, pcm: bool, table: np.ndarray, table_dev, total: int, want, normalize: bool = True,
                  out=None) -> tuple[dict, Any]:
    """One dspx_features_ragged call on torch's current stream: `samples` a packed torch CUDA tensor (float32 or
    int16), table / table_dev the layout on the host and on the device.  Returns ({name: torch CUDA view}, the flat
    float32 tensor that holds all of them in FEATURES order); `out`, when given, is that flat tensor."""
    import torch

    lib = _lib.load()
    n = len(table)
    sizes = {"log_mel": (total, plan.n_mels), "mfcc": (total, plan.n_mfcc), "embed": (n, 2 * plan.n_mfcc)}
    counts = [sizes[k][0] * sizes[k][1] for k in FEATURES if k in want]
    dev = samples.device
    if out is None:
        out = torch.empty(sum(counts), dtype=torch.float32, device=dev)
    res, off = {}, 0
    for k in FEATURES:
        if k in want:
            m = sizes[k][0] * sizes[k][1]
            res[k] = out[off:off + m].view(sizes[k])
            off += m
    code = _lib.DTYPE_PCM16 if pcm else _lib.DTYPE_F32
    flags = [1 if k in want else 0 for k in FEATURES]
    ws_bytes = int(lib.dspx_features_ragged_workspace(plan.handle, table.ctypes.data, n, code, 1 if normalize else 0, *flags))
    with torch.cuda.device(dev.index):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        ptr = [res[k].data_ptr() if k in res else None for k in FEATURES]
        _lib.check(lib.dspx_features_ragged(plan.handle, samples.data_ptr(), code, 1 if normalize else 0, table_dev.data_ptr(),
                                           table.ctypes.data, n, total, *ptr, ws.data_ptr(), ws_bytes,
                                           torch.cuda.current_stream(dev.index).cuda_stream), "dspx_features_ragged")
    return res, out


def features_ragged(clips, cfg: Any, want: Iterable[str] = ("mfcc",), device: int | None = None,
                    normalize: bool = True, sample_rate: int | None = None) -> dict:
    """log-mel / MFCC / clip embeddings of clips of different lengths, in one launch.

    `clips` is a sequence of 1-D arrays: all NumPy (float32, or int16 PCM converted like features_batch does), or all
    torch CUDA tensors of one dtype.  Returns {"log_mel": [total_frames, n_mels], "mfcc": [total_frames, n_mfcc],
    "embed": [B, 2*n_mfcc]} restricted to `want`, plus "frame_offsets" (int64 [B+1]): clip i owns rows
    frame_offsets[i]:frame_offsets[i+1].  Every clip gets the values features_batch gives it alone.  NumPy in ->
    NumPy out (one pinned staging buffer, one copy each way); torch CUDA in -> torch CUDA out on torch's current
    stream.  A clip shorter than frame_length raises ValueError naming its index.  `sample_rate` as in
    features_batch: clips at another rate are resampled on the GPU in one launch first.
    """
    import torch

    want = _want(want)
    ratio = _resample_ratio(cfg, sample_rate)
    if ratio is not None:
        clips = list(clips)
        if clips:
            return _features_ragged_resampled(clips, cfg, want, device, normalize, ratio)
    xs, on_gpu, pcm = _ragged_inputs(clips)
    starts, table, total = ragged_layout([len(x) for x in xs], cfg, np.int16 if pcm else np.float32)
    offsets = np.concatenate((table[:, 3], [total])).astype(np.int64) if len(xs) else np.zeros(1, np.int64)
    if not xs:
        key = config_key(cfg)
        shapes = {"log_mel": (0, key[4]), "mfcc": (0, key[5]), "embed": (0, 2 * key[5])}
        res = {k: np.zeros(shapes[k], np.float32) for k in want}
        res["frame_offsets"] = offsets
        return res
    n_samples = int(starts[-1] + len(xs[-1]))
    if on_gpu:
        dev = xs[0].device
        parts = []
        pad = torch.zeros(RAGGED_ALIGN, dtype=xs[0].dtype, device=dev)
        for i, x in enumerate(xs):
            parts.append(x)
            gap = int(starts[i + 1] - starts[i] - len(x)) if i + 1 < len(xs) else 0
            if gap:
                parts.append(pad[:gap])
        plan = get_plan(cfg, dev.index if device is None else device)
        with torch.cuda.device(dev.index):
            samples = torch.cat(parts)
            table_dev = torch.from_numpy(table).to(dev)
            res, _ = ragged_launch(plan, samples, pcm, table, table_dev, total, want, normalize)
        res["frame_offsets"] = torch.from_numpy(offsets).to(dev)
        return res
    plan = get_plan(cfg, device)
    dev = torch.device("cuda", plan.device)
    staging = torch.empty(n_samples, dtype=torch.int16 if pcm else torch.float32, pin_memory=True)
    host = staging.numpy()
    for s, x in zip(starts, xs):
        host[s:s + len(x)] = x
    with torch.cuda.device(plan.device):
        stream = torch.cuda.current_stream(plan.device)
        samples = staging.to(dev, non_blocking=True)
        table_dev = torch.from_numpy(table).to(dev)
        res, flat = ragged_launch(plan, samples, pcm, table, table_dev, total, want, normalize)
        out_host = torch.empty(flat.shape, dtype=torch.float32, pin_memory=True)
        out_host.copy_(flat, non_blocking=True)
        stream.synchronize()
    out, off = {}, 0
    host_out = out_host.numpy()
    for k in FEATURES:
        if k in res:
            m = res[k].numel()
            out[k] = host_out[off:off + m].reshape(tuple(res[k].shape))
            off += m
    out["frame_offsets"] = offsets
    return out


def _features_ragged_resampled(clips: list, cfg: Any, want, device, normalize: bool, ratio) -> dict:
    """features_ragged of clips at another rate: one resample launch into a packed buffer whose layout is a valid
    ragged feature batch, then one feature launch."""
    import torch

    on_gpu = [_is_cuda_tensor(c) for c in clips]
    if any(on_gpu) and not all(on_gpu):
        raise ValueError("clips must be all NumPy arrays or all torch CUDA tensors")
    pcm = {_resample_dtype(c) for c in clips}
    if len(pcm) > 1:
        raise ValueError("clips must all be float32 or all be int16 PCM")
    xs = [_to_device(c, device).reshape(-1) for c in clips]
    if len({c.device for c in xs}) > 1:
        raise ValueError("clips must be on one device")
    dev = xs[0].device
    samples, rtable = _resample_ragged(xs, get_resampler(*ratio, dev.index), normalize and pcm.pop())
    starts, table, total = ragged_layout(rtable[:, 3], cfg, np.float32, rtable[:, 2])
    plan = get_plan(cfg, dev.index if device is None else device)
    with torch.cuda.device(dev.index):
        table_dev = torch.from_numpy(table).to(dev)
        res, _ = ragged_launch(plan, samples, False, table, table_dev, total, want, normalize)
    offsets = np.concatenate((table[:, 3], [total])).astype(np.int64)
    if all(on_gpu):
        res["frame_offsets"] = torch.from_numpy(offsets).to(dev)
        return res
    res = _as_host(res)
    res["frame_offsets"] = offsets
    return res


# struct dspx_decode_clip
DECODE_CLIP = np.dtype([("in_offset", "<i8"), ("n_frames", "<i8"), ("channels", "<i4"), ("dtype", "<i4"),
                        ("out_start", "<i8"), ("out_length", "<i8")])


class PackedClips(NamedTuple):
    """Clips of one packed float32 torch CUDA buffer: clip i is samples[starts[i]:starts[i] + lengths[i]], every start a
    multiple of RAGGED_ALIGN, so the buffer is a valid ragged feature batch as it is."""
    samples: Any
    starts: np.ndarray
    lengths: np.ndarray


def _decode_layout(lib, offsets, parsed, idx) -> tuple[np.ndarray, int]:
    """dspx_decode_layout of the files `idx` of `parsed` (read_wav_data tuples) at byte `offsets`."""
    table = np.zeros(len(idx), DECODE_CLIP)
    cols = [np.ascontiguousarray(np.asarray(v, dt)) for v, dt in (
        ([offsets[i] for i in idx], np.int64), ([parsed[i][4] for i in idx], np.int64),
        ([parsed[i][2] for i in idx], np.int32), ([parsed[i][3] for i in idx], np.int32))]
    total = _lib.check(int(lib.dspx_decode_layout(*(c.ctypes.data for c in cols), len(idx), table.ctypes.data)),
                       "dspx_decode_layout")
    return table, int(total)


def _decode(lib, data, table: np.ndarray, normalize: bool, out, dev) -> None:
    """One dspx_decode_ragged call on torch's current stream into `out` (a float32 CUDA tensor)."""
    import torch

    if not len(table):
        return
    table_dev = torch.from_numpy(table.view(np.uint8)).to(dev)
    ws_bytes = int(lib.dspx_decode_workspace(len(table)))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.check(lib.dspx_decode_ragged(data.data_ptr(), table_dev.data_ptr(), table.ctypes.data, len(table),
                                      1 if normalize else 0, out.data_ptr(), ws.data_ptr(), ws_bytes,
                                      torch.cuda.current_stream(dev.index).cuda_stream), "dspx_decode_ragged")


# struct dspx_flac_file, struct dspx_flac_frame
FLAC_FILE = np.dtype([("in_offset", "<i8"), ("in_bytes", "<i8"), ("out_start", "<i8"), ("out_length", "<i8"),
                      ("first_frame", "<i8"), ("n_frames", "<i8"), ("ws_start", "<i8"), ("ws_bytes", "<i8"),
                      ("sample_rate", "<i4"), ("channels", "<i4"), ("bps", "<i4"), ("reserved", "<i4")])
FLAC_FRAME = np.dtype([("in_offset", "<i8"), ("out_start", "<i8"), ("ws_offset", "<i8"), ("in_bytes", "<i4"),
                       ("header_bytes", "<i4"), ("block_size", "<i4"), ("assignment", "<i4"), ("file", "<i4"),
                       ("reserved", "<i4")])
FLAC_STATUS = {1: "CRC-16 mismatch", 2: "bitstream overrun", 4: "reserved code", 8: "negative LPC shift",
               16: "invalid subframe parameters"}


class FlacError(ValueError):
    """A FLAC file the GPU decoder refuses: its stream does not parse, or a frame does not decode."""


def flac_parse(data: np.ndarray, name=None) -> tuple[np.ndarray, np.ndarray]:
    """(file row, frame table) of one FLAC file's bytes, from one dspx_flac_layout pass over them in most cases: the
    frame table is sized from the file's size first (a frame of compressed audio rarely takes less than 256 bytes) and
    only a file of more frames than that, such as digital silence, is parsed a second time."""
    lib = _lib.load()
    ptr = (C.c_void_p * 1)(data.ctypes.data)
    size, offset, n_frames = (C.c_int64 * 1)(len(data)), (C.c_int64 * 1)(0), C.c_int64(0)
    files = np.zeros(1, FLAC_FILE)
    frames = np.zeros(len(data) // 256 + 16, FLAC_FRAME)
    for _ in range(2):
        if lib.dspx_flac_layout(ptr, size, offset, 1, files.ctypes.data, frames.ctypes.data, len(frames),
                                C.byref(n_frames)) < 0:
            raise FlacError(f"{name if name is not None else 'FLAC file'}: {_lib.last_error()}")
        if n_frames.value <= len(frames):
            return files[0], frames[:n_frames.value]
        frames = np.zeros(n_frames.value, FLAC_FRAME)
    raise AssertionError("dspx_flac_layout gave two frame counts for one file")


def _flac_layout(lib, offsets, parsed, idx) -> tuple[np.ndarray, np.ndarray, int]:
    """The file and frame tables of the files `idx` of `parsed` (read_flac_data tuples, whose last element holds each
    file's own tables) at byte `offsets`, and the packed output length.  The frame rows are relative to their file, so
    joining them parses nothing again: only the file rows' offsets and the frames' `file` change."""
    files = np.zeros(len(idx), FLAC_FILE)
    parts = []
    at = nf = ws = total = 0
    for j, i in enumerate(idx):
        row, frames = parsed[i][5] if len(parsed[i]) > 5 else flac_parse(parsed[i][0], f"file {i}")
        files[j] = row
        for field, v in (("in_offset", offsets[i]), ("out_start", at), ("first_frame", nf), ("ws_start", ws)):
            files[field][j] = v
        frames = frames.copy()
        frames["file"] = j
        parts.append(frames)
        total = at + int(row["out_length"])
        at += (int(row["out_length"]) + RAGGED_ALIGN - 1) // RAGGED_ALIGN * RAGGED_ALIGN
        nf += len(frames)
        ws += int(row["ws_bytes"])
    return files, (np.concatenate(parts) if parts else np.zeros(0, FLAC_FRAME)), total


def _flac_decode(lib, data, tabs, normalize: bool, out, dev):
    """One dspx_flac_decode call on torch's current stream into out[base:]; returns the per-frame status tensor."""
    import torch

    files, frames, base, _ = tabs
    files_dev = torch.from_numpy(files.view(np.uint8)).to(dev)
    frames_dev = torch.from_numpy(frames.view(np.uint8)).to(dev)
    status = torch.empty(len(frames), dtype=torch.int32, device=dev)
    ws_bytes = int(lib.dspx_flac_workspace(files.ctypes.data, len(files)))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    _lib.check(lib.dspx_flac_decode(data.data_ptr(), files_dev.data_ptr(), files.ctypes.data, len(files),
                                    frames_dev.data_ptr(), frames.ctypes.data, len(frames), 1 if normalize else 0,
                                    out[base:].data_ptr(), status.data_ptr(), ws.data_ptr(), ws_bytes,
                                    torch.cuda.current_stream(dev.index).cuda_stream), "dspx_flac_decode")
    return status


def _flac_check(checks, status: np.ndarray, offsets, names) -> None:
    """Raise FlacError naming the first file and frame whose status is not 0."""
    at = 0
    for (files, frames, _, idx), _st in checks:
        st = status[at:at + len(frames)]
        at += len(frames)
        bad = np.flatnonzero(st)
        if not len(bad):
            continue
        f = int(bad[0])
        row = frames[f]
        i = idx[int(row["file"])]
        j = f - int(files[int(row["file"])]["first_frame"])
        what = ", ".join(v for k, v in FLAC_STATUS.items() if int(st[f]) & k)
        name = names[i] if names is not None else f"file {i}"
        raise FlacError(f"{name}: FLAC frame {j} (byte {int(row['in_offset'])}): {what}")


def pack_files(parsed: list) -> tuple[Any, np.ndarray]:
    """(pinned uint8 tensor holding the bytes of read_wav_data / read_flac_data tuples, their byte offsets: multiples
    of 16)."""
    import torch

    sizes = np.array([len(p[0]) for p in parsed], np.int64)
    offsets = np.zeros(len(parsed), np.int64)
    offsets[1:] = np.cumsum((sizes + 15) // 16 * 16)[:-1]
    staging = torch.empty(max(int(offsets[-1] + sizes[-1]) if len(parsed) else 0, 1), dtype=torch.uint8, pin_memory=True)
    host = staging.numpy()
    for o, p in zip(offsets, parsed):
        host[o:o + len(p[0])] = p[0]
    return staging, offsets


def decode_device(data, offsets: np.ndarray, parsed: list, target_sr: int | None, normalize: bool,
                  names: list | None = None) -> PackedClips:
    """The device part of decode_packed: `data` (a uint8 torch CUDA tensor) holds the files of the read_wav_data /
    read_flac_data tuples `parsed` at byte `offsets`; work is enqueued on torch's current stream of data's device.
    When FLAC files are among them, their frames' status is read back once (a synchronisation) and a bad frame raises
    ValueError naming the file (names[i], else its index) and the frame."""
    import torch

    lib = _lib.load()
    dev = data.device
    n = len(parsed)
    flac = [parsed[i][3] == _lib.DTYPE_FLAC for i in range(n)]
    at_rate = [target_sr is None or parsed[i][1] == target_sr for i in range(n)]
    starts, lengths = np.zeros(n, np.int64), np.array([p[4] for p in parsed], np.int64)

    def packed(rate_ok):
        """Layouts of the WAV files, then of the FLAC files, with at_rate == rate_ok, back to back from 0."""
        wav_idx = [i for i in range(n) if at_rate[i] == rate_ok and not flac[i]]
        flac_idx = [i for i in range(n) if at_rate[i] == rate_ok and flac[i]]
        wtab, total = _decode_layout(lib, offsets, parsed, wav_idx)
        at = np.zeros(n, np.int64)
        at[wav_idx] = wtab["out_start"]
        ftabs = None
        if flac_idx:
            base = (total + RAGGED_ALIGN - 1) // RAGGED_ALIGN * RAGGED_ALIGN
            files, frames, ftotal = _flac_layout(lib, offsets, parsed, flac_idx)
            at[flac_idx] = base + files["out_start"]
            ftabs = (files, frames, base, flac_idx)
            total = base + ftotal
        return wtab, ftabs, at, total

    dtab, dflac, dstart, at = packed(True)
    direct = [i for i in range(n) if at_rate[i]]
    others = [i for i in range(n) if not at_rate[i]]
    starts[direct] = dstart[direct]
    rtab, rflac, rstart, r_total = packed(False)
    groups = []
    for rate in sorted({parsed[i][1] for i in others}):
        idx = [i for i in others if parsed[i][1] == rate]
        up, down = reduce_ratio(target_sr, rate)
        in_starts = np.ascontiguousarray(rstart[idx])
        in_lengths = np.ascontiguousarray(lengths[idx])
        table = np.zeros((len(idx), 4), np.int64)
        total = _lib.check(int(lib.dspx_resample_layout(up, down, in_starts.ctypes.data, in_lengths.ctypes.data, len(idx),
                                                        table.ctypes.data)), "dspx_resample_layout")
        base = (at + RAGGED_ALIGN - 1) // RAGGED_ALIGN * RAGGED_ALIGN
        starts[idx] = base + table[:, 2]
        lengths[idx] = table[:, 3]
        groups.append((up, down, table, base))
        at = base + int(total)
    checks = []
    with torch.cuda.device(dev.index):
        out = torch.zeros(max(at, 1), dtype=torch.float32, device=dev)
        _decode(lib, data, dtab, normalize, out, dev)
        if dflac:
            checks.append((dflac, _flac_decode(lib, data, dflac, normalize, out, dev)))
        if groups:
            scratch = torch.empty(max(r_total, 1), dtype=torch.float32, device=dev)
            _decode(lib, data, rtab, False, scratch, dev)
            if rflac:
                checks.append((rflac, _flac_decode(lib, data, rflac, False, scratch, dev)))
            stream = torch.cuda.current_stream(dev.index).cuda_stream
            for up, down, table, base in groups:
                table_dev = torch.from_numpy(table).to(dev)
                ws_bytes = int(lib.dspx_resample_workspace(len(table)))
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                _lib.check(lib.dspx_resample_ragged(get_resampler(up, down, dev.index).handle, scratch.data_ptr(),
                                                    _lib.DTYPE_F32, 1 if normalize else 0, table_dev.data_ptr(),
                                                    table.ctypes.data, len(table), out[base:].data_ptr(), ws.data_ptr(),
                                                    ws_bytes, stream), "dspx_resample_ragged")
        if checks:
            _flac_check(checks, torch.cat([st for _, st in checks]).cpu().numpy(), offsets, names)
    return PackedClips(out, starts, lengths)


def decode_packed(parsed: list, target_sr: int | None, normalize: bool, device: int | None = None,
                  names: list | None = None) -> PackedClips:
    """load_audio(path, target_sr)[0] (normalize_audio of it when `normalize`) of every file, from its read_wav_data
    or read_flac_data tuple, into one packed buffer on the GPU.

    The WAV data chunks and FLAC files travel as stored, at 16-byte offsets of one pinned buffer, in one host-to-device
    copy.  Files at target_sr (or all of them when it is None) are decoded with the normalisation, straight into the
    output buffer (one WAV and one FLAC decode launch); the others are decoded without it into a scratch buffer (the
    same two), then resampled with it, one dspx_resample_ragged launch per rate, each group of outputs at its own
    offset of the output buffer -- the reference's order: decode, downmix, resample, normalise.  A FLAC frame that
    does not decode raises ValueError naming the file (names[i] when given) and the frame.
    """
    import torch

    _lib.require_device()
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
    staging, offsets = pack_files(parsed)
    with torch.cuda.device(dev.index):
        data = staging.to(dev, non_blocking=True)
    return decode_device(data, offsets, parsed, target_sr, normalize, names)


def load_audio_batch(paths, target_sr: int | None = None, normalize: bool = False, device: int | None = None) -> list:
    """[load_audio(p, target_sr)[0] for p in paths] (normalize_audio of each when `normalize`), decoded on the GPU.

    Returns float32 torch CUDA tensors, views into one packed buffer, bit-identical to the host functions.  The files
    may mix PCM 8/16/24/32-bit and IEEE float 32/64 WAV encodings with 1 to 32 channels, FLAC files (4 to 32 bits, 1
    to 8 channels), lengths and rates; each is decoded and downmixed on the device, then resampled there when its
    rate is not target_sr.  A file of another kind, without audio frames, or with a FLAC frame that does not decode
    raises ValueError naming it.
    """
    from .audio import read_flac_data, read_wav_data

    parsed = []
    paths = list(paths)
    for p in paths:
        d = read_wav_data(p)
        if d is None:
            d = read_flac_data(p)
        if d is None:
            raise ValueError(f"{p}: neither a FLAC file nor a WAV file of PCM 8/16/24/32-bit or IEEE float 32/64 samples "
                             "with 1 to 32 channels")
        if d[4] < 1:
            raise ValueError(f"{p}: no audio frames")
        parsed.append(d)
    if not parsed:
        return []
    packed = decode_packed(parsed, None if target_sr is None else int(target_sr), normalize, device, [str(p) for p in paths])
    return [packed.samples[s:s + n] for s, n in zip(packed.starts.tolist(), packed.lengths.tolist())]


def features_packed(packed: PackedClips, cfg: Any, want: Iterable[str] = ("mfcc",)) -> dict:
    """features_ragged of the float32 clips of a PackedClips buffer, with no copy of the samples: NumPy outputs plus
    "frame_offsets", as features_ragged returns for NumPy input."""
    import torch

    want = _want(want)
    dev = packed.samples.device
    starts, table, total = ragged_layout(packed.lengths, cfg, np.float32, packed.starts)
    plan = get_plan(cfg, dev.index)
    with torch.cuda.device(dev.index):
        table_dev = torch.from_numpy(table).to(dev)
        res, _ = ragged_launch(plan, packed.samples, False, table, table_dev, total, want)
    res = _as_host(res)
    res["frame_offsets"] = np.concatenate((table[:, 3], [total])).astype(np.int64)
    return res


def split_ragged(stacked, frame_offsets) -> list:
    """[total_frames, C] stacked features -> one [T_i, C] view per clip."""
    o = [int(v) for v in (frame_offsets.tolist() if hasattr(frame_offsets, "tolist") else frame_offsets)]
    return [stacked[o[i]:o[i + 1]] for i in range(len(o) - 1)]


def mfcc_batch(clips, cfg, **kw):
    return features_batch(clips, cfg, ("mfcc",), **kw)["mfcc"]


def log_mel_batch(clips, cfg, **kw):
    return features_batch(clips, cfg, ("log_mel",), **kw)["log_mel"]


def mfcc_embed_batch(clips, cfg, **kw):
    """[B, 2*n_mfcc] clip embeddings, src/retrieval/retrieval.py:19-23 batched."""
    return features_batch(clips, cfg, ("embed",), **kw)["embed"]


def log_mel_nchw(clips, cfg, device: int | None = None, kernel: str = "auto"):
    """log-mel as the CNN input tensor [B, 1, n_mels, n_frames] (float32, torch CUDA in and out).

    What LogMelTransform + DataLoader batching hand to ResNetAudio (src/train/transforms.py:16-18,
    scripts/models/train_cnn.py:46-55), written in that layout by the kernel's store epilogue.
    """
    import torch

    if not _is_cuda_tensor(clips):
        clips = torch.as_tensor(_as_host_clips(clips)).cuda()
    if _is_pcm16(clips):
        clips = pcm16_to_float(clips)
    x = clips if clips.dim() == 2 else clips[None, :]
    if x.dtype != torch.float32 or x.stride(1) != 1:
        x = x.to(torch.float32).contiguous()
    dev = x.device.index if device is None else device
    plan = get_plan(cfg, dev, kernel)
    b, length = x.shape
    t = plan.num_frames(length)
    with torch.cuda.device(dev):
        out = torch.empty((b, 1, plan.n_mels, t), dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().dspx_log_mel_nchw(plan.handle, x.data_ptr(), b, length, x.stride(0), out.data_ptr(),
                                                 torch.cuda.current_stream(dev).cuda_stream), "dspx_log_mel_nchw")
    return out


def stft_batch(clips, frame_length: int, hop_length: int, window: str = "hann", n_fft: int | None = None,
               device: int | None = None, pre_emphasis: float = 0.0, kernel: str = "auto"):
    """[B, T, n_fft_pow2//2+1] complex64 STFT, src/dsp/stft.py:43-56 batched.

    pre_emphasis > 0 applies the MFCC path's filter first (the reference stft() has none).
    """
    lib = _lib.load()
    cfg = dict(sample_rate=1, frame_length=frame_length, hop_length=hop_length, n_fft=n_fft, n_mels=1, n_mfcc=1,
               f_min=0.0, f_max=None, pre_emphasis=float(pre_emphasis), window=window)
    pre = 1 if pre_emphasis > 0 else 0
    if _is_cuda_tensor(clips):
        import torch

        x = clips if clips.dim() == 2 else clips[None, :]
        if x.dtype != torch.float32 or x.stride(1) != 1:
            x = x.to(torch.float32).contiguous()
        dev = x.device.index if device is None else device
        plan = get_plan(cfg, dev, kernel)
        b, length = x.shape
        t = plan.num_frames(length)
        with torch.cuda.device(dev):
            out = torch.empty((b, t, plan.n_bins), dtype=torch.complex64, device=x.device)
            _lib.check(lib.dspx_stft(plan.handle, x.data_ptr(), b, length, x.stride(0), pre, out.data_ptr(),
                                     torch.cuda.current_stream(dev).cuda_stream), "dspx_stft")
        return out
    x = _as_host_clips(clips)
    plan = get_plan(cfg, device, kernel)
    b, length = x.shape
    t = plan.num_frames(length)
    out = np.empty((b, t, plan.n_bins), np.complex64)
    _lib.check(lib.dspx_stft_host(plan.handle, x.ctypes.data, b, length, max(x.strides[0] // 4, length), pre,
                                  out.ctypes.data),
               "dspx_stft_host")
    return out


def _embed_stats_ragged(feats: list):
    """embed_stats of a list of [T_i, C] arrays (all NumPy or all torch CUDA) through dspx_embed_stats_ragged."""
    import torch

    host = not all(_is_cuda_tensor(f) for f in feats)
    fs = [torch.as_tensor(np.asarray(f, dtype=np.float32)) if host else f.to(torch.float32) for f in feats]
    if any(f.dim() != 2 or f.shape[1] != fs[0].shape[1] or f.shape[0] < 1 for f in fs):
        raise ValueError("embed_stats takes [T_i, C] arrays with T_i >= 1 and one C")
    c = int(fs[0].shape[1])
    rows = np.array([f.shape[0] for f in fs], np.int64)
    table = np.zeros((len(fs), 5), np.int64)
    table[:, 2] = rows
    table[:, 3] = np.cumsum(rows) - rows
    dev = torch.device("cuda", torch.cuda.current_device()) if host else fs[0].device
    with torch.cuda.device(dev.index):
        stacked = torch.cat(fs).to(dev).contiguous()
        table_dev = torch.from_numpy(table).to(dev)
        out = torch.empty((len(fs), 2 * c), dtype=torch.float32, device=dev)
        _lib.check(_lib.load().dspx_embed_stats_ragged(stacked.data_ptr(), table_dev.data_ptr(), len(fs), c, out.data_ptr(),
                                                       torch.cuda.current_stream(dev.index).cuda_stream),
                   "dspx_embed_stats_ragged")
    return out.cpu().numpy() if host else out


def embed_stats(feats):
    """concat(mean_t, std_t) of [B, T, C] float32 features (retrieval.py:38-41). torch CUDA in/out.

    A list or tuple of [T_i, C] arrays (clips of different lengths) is reduced in one launch, with the same
    per-clip summation order."""
    import torch

    _lib.require_device()
    if isinstance(feats, (list, tuple)):
        if not feats:
            raise ValueError("embed_stats of an empty list")
        return _embed_stats_ragged(list(feats))
    if not _is_cuda_tensor(feats):
        feats = torch.as_tensor(np.asarray(feats, dtype=np.float32)).cuda()
        to_host = True
    else:
        to_host = False
    f = feats.to(torch.float32).contiguous()
    if f.dim() == 2:
        f = f[None]
    b, t, c = f.shape
    dev = f.device.index
    with torch.cuda.device(dev):
        out = torch.empty((b, 2 * c), dtype=torch.float32, device=f.device)
        _lib.check(_lib.load().dspx_embed_stats(f.data_ptr(), b, t, c, out.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream), "dspx_embed_stats")
    return out.cpu().numpy() if to_host else out


def cmvn(feats, eps: float = 1e-10):
    """Cepstral mean / variance normalisation per clip: (x - mean_t) / (std_t + eps) over [B, T, C] features.

    Not part of the reference pipeline (src/dsp/mfcc.py:102-109 end at log and DCT); offered because
    BASELINE.json's north_star names a log/CMVN epilogue.  torch CUDA tensors are normalised in place
    and returned; NumPy input returns a new array.
    """
    import torch

    _lib.require_device()
    host = not _is_cuda_tensor(feats)
    f = torch.as_tensor(np.ascontiguousarray(np.asarray(feats, dtype=np.float32))).cuda() if host else feats
    if f.dtype != torch.float32 or not f.is_contiguous():
        raise ValueError("cmvn needs a contiguous float32 tensor")
    v = f if f.dim() == 3 else f[None]
    b, t, c = v.shape
    dev = f.device.index
    with torch.cuda.device(dev):
        _lib.check(_lib.load().dspx_cmvn(v.data_ptr(), b, t, c, float(eps), torch.cuda.current_stream(dev).cuda_stream),
                   "dspx_cmvn")
    return f.cpu().numpy() if host else f


def fft_batch(x, n: int | None = None, inverse: bool = False):
    """Batched complex FFT over the last axis with the reference's length rule (fft.py:27-42).

    x: [..., n_in] real or complex (NumPy or torch CUDA).  Returns complex64 [..., next_pow2(n)],
    same kind of container as the input.
    """
    import torch

    _lib.require_device()
    lib = _lib.load()
    host = not _is_cuda_tensor(x)
    if host:
        xt = torch.as_tensor(np.ascontiguousarray(np.asarray(x).astype(np.complex64))).cuda()
    else:
        xt = x.to(torch.complex64)
    xt = xt.contiguous()
    lead = xt.shape[:-1]
    n_in = xt.shape[-1]
    nn = n_in if n is None else int(n)
    if nn < 1:
        raise ValueError("fft length must be positive")
    p = int(lib.dspx_next_pow_two(nn))
    batch = int(np.prod(lead)) if lead else 1
    dev = xt.device.index
    with torch.cuda.device(dev):
        out = torch.empty((batch, p), dtype=torch.complex64, device=xt.device)
        work = torch.empty((batch, p), dtype=torch.complex64, device=xt.device)
        _lib.check(lib.dspx_fft_c2c(xt.data_ptr(), batch, n_in, nn, 1 if inverse else 0, out.data_ptr(),
                                    work.data_ptr(), torch.cuda.current_stream(dev).cuda_stream), "dspx_fft_c2c")
    out = out.reshape(*lead, p)
    return out.cpu().numpy() if host else out


def dct2_rows(x, n_mfcc: int):
    """dct_type_2 over the last axis on the GPU (src/dsp/mfcc.py:73-83). NumPy or torch CUDA."""
    import torch

    _lib.require_device()
    host = not _is_cuda_tensor(x)
    xt = torch.as_tensor(np.ascontiguousarray(np.asarray(x, dtype=np.float32))).cuda() if host else x.to(torch.float32)
    xt = xt.contiguous()
    lead, n = xt.shape[:-1], xt.shape[-1]
    rows = int(np.prod(lead)) if lead else 1
    dev = xt.device.index
    with torch.cuda.device(dev):
        out = torch.empty((rows, int(n_mfcc)), dtype=torch.float32, device=xt.device)
        _lib.check(_lib.load().dspx_dct2(xt.data_ptr(), rows, int(n), int(n_mfcc), out.data_ptr(),
                                         torch.cuda.current_stream(dev).cuda_stream), "dspx_dct2")
    out = out.reshape(*lead, int(n_mfcc))
    return out.cpu().numpy() if host else out
