"""MFCC retrieval scoring with the reference's signatures (src/retrieval/retrieval.py).

    _mfcc_embedding, compute_embeddings, cosine_similarity, evaluate_retrieval, RetrievalResult

Scoring and selection run on the GPU (dspx_cosine_topk: float64 cosine scores,
running top-k kept on chip, the [nq, ndb] matrix never materialised).  Ranking
follows np.argsort(-sims, axis=1, kind="stable")[:, :k]: descending score, ties
to the lower database index.  (The reference calls np.argsort with the default
introsort, whose tie order is unspecified; the stable order is the one
deterministic member of that family.)
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, Iterable, List

import numpy as np

from . import _lib
from .batch import FlacError, PackedClips, _is_cuda_tensor, decode_packed, embed_stats, features_batch, features_packed, features_ragged
from .dsp.mfcc import MfccConfig


@dataclass
class RetrievalResult:
    k: int
    precision: float


def _mfcc_embedding(signal: np.ndarray, cfg: MfccConfig) -> np.ndarray:
    """concat(mean_t, std_t) of the clip's MFCCs (src/retrieval/retrieval.py:19-23)."""
    sig = np.asarray(signal, dtype=np.float32).reshape(1, -1)
    return features_batch(sig, cfg, ("embed",))["embed"][0].astype(np.float64)


def _load_clips(items: List[Any], cfg: MfccConfig, loader) -> tuple[list | PackedClips, int | None]:
    """(the clips, their sample rate; None for float32 clips, which are already at cfg.sample_rate).

    The clips are what the reference's load_audio + normalize_audio return (src/utils/audio.py:19-38 as used by
    retrieval.py:35-36), bit for bit, taken in this order:
      1. every file is mono 16-bit PCM at one common rate: the raw int16 samples and that rate.  The GPU resamples
         them when that rate is not cfg.sample_rate, converts and peak-normalises inside the feature launch;
      2. otherwise, when read_wav_data (PCM 8/16/24/32-bit or IEEE float 32/64, 1 to 32 channels) or read_flac_data
         (FLAC) accepts every file, at any rates: a PackedClips buffer, decoded, downmixed, resampled and normalised on
         the GPU (decode_packed);
      3. otherwise, or when the GPU decoder refuses a FLAC file (batch.FlacError): float32 arrays from load_audio +
         normalize_audio on the host (without soundfile, load_audio of such a file raises FlacError naming it)."""
    from .audio import load_audio, normalize_audio, read_flac_data, read_pcm16, read_wav_data

    if loader is not None:
        return [np.asarray(loader(item), dtype=np.float32).reshape(-1) for item in items], None
    pcm = [read_pcm16(item.path) for item in items]
    if all(p is not None for p in pcm) and len({rate for _, rate in pcm}) == 1:
        return [x for x, _ in pcm], pcm[0][1]
    try:
        data = [read_wav_data(item.path) for item in items]
        data = [d if d is not None else read_flac_data(item.path) for d, item in zip(data, items)]
        if all(d is not None and d[4] >= 1 for d in data):
            return decode_packed(data, int(cfg.sample_rate), True, names=[str(item.path) for item in items]), None
    except FlacError:          # a FLAC file the GPU decoder refuses: the host loader (soundfile) may still read it
        pass
    clips = []
    for item in items:
        audio, _ = load_audio(item.path, target_sr=cfg.sample_rate)
        clips.append(normalize_audio(audio).astype(np.float32))
    return clips, None


def _equal_shapes(arrays: list) -> bool:
    return len({a.shape for a in arrays}) == 1


def compute_embeddings(items: List[Any], cfg: MfccConfig, feature_cache=None, loader=None) -> np.ndarray:
    """[N, 2*n_mfcc] embeddings, concat(mean_t, std_t) of each clip's MFCCs (src/retrieval/retrieval.py:26-43).

    Reference signature (items, cfg, feature_cache=None); `loader(item) -> samples` optionally replaces the
    audio decoding.  Without a cache the clips are read from item.path (load_audio + normalize_audio
    semantics) and go through the fused kernel as one batch (one ragged launch when their lengths differ).
    With a cache the float32 MFCCs come from it (any object with the reference's get_feature; BatchFeatureCache
    fills its misses in GPU batches) and are reduced on the GPU in one launch -- the path
    scripts/tasks/run_retrieval.py takes.
    """
    items = list(items)
    if not items:
        return np.zeros((0, 2 * cfg.n_mfcc), np.float32)
    if feature_cache is not None:
        if hasattr(feature_cache, "get_features"):
            feats = feature_cache.get_features(items, "mfcc", cfg, loader=loader)
        else:
            feats = [feature_cache.get_feature(item, "mfcc", cfg) for item in items]
        feats = [np.asarray(f, dtype=np.float32) for f in feats]
        return embed_stats(np.stack(feats, axis=0) if _equal_shapes(feats) else feats)
    clips, rate = _load_clips(items, cfg, loader)
    if isinstance(clips, PackedClips):
        return features_packed(clips, cfg, ("embed",))["embed"]
    if _equal_shapes(clips):
        return features_batch(np.stack(clips, axis=0), cfg, ("embed",), sample_rate=rate)["embed"]
    return features_ragged(clips, cfg, ("embed",), sample_rate=rate)["embed"]


def _dev_matrix(x):
    """-> (torch CUDA tensor [n, d] contiguous float32|float64, dtype code)."""
    import torch

    if _is_cuda_tensor(x):
        t = x
    else:
        a = np.asarray(x)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    if t.dim() != 2:
        raise ValueError("embeddings must be [n, dim]")
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float64)
    t = t.contiguous()
    return t, (_lib.DTYPE_F32 if t.dtype == torch.float32 else _lib.DTYPE_F64)


def _dev_pair(a, b):
    """-> (a, b, dtype code): both as _dev_matrix, in float64 when their dtypes differ; their dimensions must match."""
    import torch

    q, dq = _dev_matrix(a)
    db, dd = _dev_matrix(b)
    if dq != dd:
        q, db = q.to(torch.float64), db.to(torch.float64)
        dq = _lib.DTYPE_F64
    if q.shape[1] != db.shape[1]:
        raise ValueError("query and database embeddings differ in dimension")
    return q, db, dq


def cosine_topk(query_embeddings, db_embeddings, k: int, return_scores: bool = False):
    """Indices [nq, k] (int32) of the k most similar database rows per query, best first.

    NumPy in -> NumPy out; torch CUDA in -> torch CUDA out.  k is clipped to the
    database size like the reference's slice [:, :k].
    """
    import torch

    _lib.require_device()
    lib = _lib.load()
    host = not _is_cuda_tensor(query_embeddings)
    q, db, dq = _dev_pair(query_embeddings, db_embeddings)
    nq, dim = q.shape
    ndb = db.shape[0]
    k = int(min(k, ndb))
    if k < 1:
        raise ValueError("k must be >= 1 and the database non-empty")
    if k > _lib.MAX_K:
        raise NotImplementedError(f"k > {_lib.MAX_K} not supported by dspx_cosine_topk")
    dev = q.device.index
    with torch.cuda.device(dev):
        idx = torch.empty((nq, k), dtype=torch.int32, device=q.device)
        sc = torch.empty((nq, k), dtype=torch.float64, device=q.device)
        ws_bytes = int(lib.dspx_cosine_topk_workspace(nq, ndb, dim, k))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device)
        _lib.check(lib.dspx_cosine_topk(q.data_ptr(), nq, db.data_ptr(), ndb, dim, dq, k, idx.data_ptr(),
                                        sc.data_ptr(), ws.data_ptr(), ws_bytes,
                                        torch.cuda.current_stream(dev).cuda_stream), "dspx_cosine_topk")
    if host:
        idx, sc = idx.cpu().numpy(), sc.cpu().numpy()
    return (idx, sc) if return_scores else idx


def cosine_similarity(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """a_norm @ b_norm.T with rows scaled by 1/(||row|| + 1e-10) (src/retrieval/retrieval.py:46-49).

    Dense float64 [len(a), len(b)] matrix computed on the GPU; evaluate_retrieval does
    not need it (it ranks on chip) -- this is for callers that want the scores.
    """
    import torch

    _lib.require_device()
    lib = _lib.load()
    host = not _is_cuda_tensor(a)
    q, db, dq = _dev_pair(a, b)
    nq, dim = q.shape
    ndb = db.shape[0]
    dev = q.device.index
    with torch.cuda.device(dev):
        out = torch.empty((nq, ndb), dtype=torch.float64, device=q.device)
        ws_bytes = int(lib.dspx_cosine_topk_workspace(nq, ndb, dim, 1))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device)
        st = torch.cuda.current_stream(dev).cuda_stream
        for s in range(0, nq, 65535):
            e = min(nq, s + 65535)
            _lib.check(lib.dspx_cosine_matrix(q[s:e].data_ptr(), e - s, db.data_ptr(), ndb, dim, dq,
                                              out[s:e].data_ptr(), ws.data_ptr(), ws_bytes, st), "dspx_cosine_matrix")
    return out.cpu().numpy() if host else out


def hits_at_k_device(topk_idx, k_list, targets_db, targets_query):
    """Device-side hit counts for several k at once: int64 tensor [len(k_list)] on the GPU, no host sync.

    topk_idx [nq, kmax] int32, targets_db [ndb] and targets_query [nq] int32 -- torch CUDA tensors.
    """
    import torch

    idx = topk_idx.to(torch.int32).contiguous()
    tdb = targets_db.to(torch.int32).contiguous()
    tq = targets_query.to(torch.int32).contiguous()
    dev = idx.device
    with torch.cuda.device(dev.index):
        hits = torch.zeros(len(k_list), dtype=torch.int64, device=dev)
        st = torch.cuda.current_stream(dev.index).cuda_stream
        for i, k in enumerate(k_list):
            if k > idx.shape[1]:
                raise ValueError("k exceeds the width of topk_idx")
            _lib.check(_lib.load().dspx_hits_at_k(idx.data_ptr(), idx.shape[0], idx.shape[1], int(k), tdb.data_ptr(),
                                                  tq.data_ptr(), hits[i:].data_ptr(), st), "dspx_hits_at_k")
    return hits


def hits_at_k(topk_idx, k: int, targets_db, targets_query) -> int:
    """Number of queries with at least one same-target row in their top k (retrieval.py:66-70)."""
    import torch

    _lib.require_device()
    idx = topk_idx if _is_cuda_tensor(topk_idx) else torch.as_tensor(np.ascontiguousarray(topk_idx, dtype=np.int32)).cuda()
    dev = idx.device
    tdb = torch.as_tensor(np.asarray(targets_db.cpu() if _is_cuda_tensor(targets_db) else targets_db, dtype=np.int32)).to(dev)
    tq = torch.as_tensor(np.asarray(targets_query.cpu() if _is_cuda_tensor(targets_query) else targets_query, dtype=np.int32)).to(dev)
    return int(hits_at_k_device(idx, [k], tdb, tq).item())


def evaluate_retrieval(db_items: List[Any], query_items: List[Any], db_embeddings, query_embeddings,
                       k_list: Iterable[int]) -> List[RetrievalResult]:
    """hit@k "precision" per k (src/retrieval/retrieval.py:52-72).

    One top-max(k) selection serves every k: a stable ranking's top-10 is the first
    ten columns of its top-20.
    """
    k_list = [int(k) for k in k_list]
    targets_db = np.array([item.target for item in db_items], dtype=np.int32)
    targets_query = np.array([item.target for item in query_items], dtype=np.int32)
    if not k_list:
        return []
    idx = cosine_topk(query_embeddings, db_embeddings, max(k_list))
    results = []
    for k in k_list:
        kk = min(k, idx.shape[1])
        hits = hits_at_k(idx, kk, targets_db, targets_query)
        results.append(RetrievalResult(k=k, precision=hits / len(query_items)))
    return results
