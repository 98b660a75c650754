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
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Iterable

import numpy as np

from . import _lib
from .plan import Plan, config_key, config_struct, get_plan

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


def features_batch(clips, cfg: Any, want: Iterable[str] = ("mfcc",), device: int | None = None,
                   kernel: str = "auto", normalize: bool = True) -> dict:
    """log-mel / MFCC / clip embeddings of a batch of equal-length clips.

    Follows src/dsp/mfcc.py:86-109 (+ src/retrieval/retrieval.py:19-23 for "embed").
    Returns {"log_mel": [B,T,n_mels], "mfcc": [B,T,n_mfcc], "embed": [B,2*n_mfcc]} (float32)
    restricted to `want`.  int16 input is taken as PCM16 and converted on the GPU like
    load_audio (+ normalize_audio when `normalize`), src/utils/audio.py:19-38, cache.py:66-67.
    """
    want = _want(want)
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
                    normalize: bool = True) -> dict:
    """log-mel / MFCC / clip embeddings of clips of different lengths, in one launch.

    `clips` is a sequence of 1-D arrays: all NumPy (float32, or int16 PCM converted like features_batch does), or all
    torch CUDA tensors of one dtype.  Returns {"log_mel": [total_frames, n_mels], "mfcc": [total_frames, n_mfcc],
    "embed": [B, 2*n_mfcc]} restricted to `want`, plus "frame_offsets" (int64 [B+1]): clip i owns rows
    frame_offsets[i]:frame_offsets[i+1].  Every clip gets the values features_batch gives it alone.  NumPy in ->
    NumPy out (one pinned staging buffer, one copy each way); torch CUDA in -> torch CUDA out on torch's current
    stream.  A clip shorter than frame_length raises ValueError naming its index.
    """
    import torch

    want = _want(want)
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
