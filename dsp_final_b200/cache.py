"""Batched writer/reader of the reference's feature-cache format (SURVEY.md 8f row f1).

The reference fills its cache one clip per call (FeatureCache.get_feature, src/features/cache.py:76-87;
scripts/tools/precompute_features.py:96-107 fans that out to processes: 19 minutes for ESC-50).  This
module computes whole batches on the GPU and writes the very same files, so the reference's
run_retrieval.py / train_cnn.py read GPU-made features unchanged:

    <root>/<feature_type>/<sha1(params)[:12]>/fold<k>/<filename>.npy      float32 [n_frames, n_coef], C order
    <root>/<feature_type>/<digest>/manifest.json                          same keys as cache.py:96-112

What is kept is the on-disk contract, not the code (the functions below are organised around batches):
  * digest recipe (cache.py:24-41): sha1 of json.dumps({"feature_type": ft, **params}, sort_keys=True,
    ensure_ascii=True), first 12 hex digits.  For an MfccConfig dataclass, params = its fields with
    n_fft None -> frame_length and f_max None -> sample_rate / 2; a plain dict (what retrieval_ml.py
    passes for embedding_* caches) is hashed verbatim, with no defaulting;
  * the filename keeps its ".wav" suffix, one directory per fold (cache.py:43-49);
  * payload: np.save of a float32 C-order array, written to a unique temporary name and renamed into
    place, so readers never see a partial file (cache.py:89-94);
  * manifest keys and their order (cache.py:96-112).
"""
from __future__ import annotations

import hashlib
import json
import os
import uuid
from concurrent.futures import ThreadPoolExecutor
from dataclasses import fields, is_dataclass
from datetime import datetime, timezone
from pathlib import Path
from typing import Any, Callable, Iterable, Mapping, Sequence

import numpy as np

FEATURE_TYPES = ("mfcc", "log_mel")
MANIFEST_KEYS = ("feature_type", "hash", "params", "created_at", "num_files", "files")
_UNREADABLE = (OSError, ValueError, EOFError)      # what np.load raises on a truncated / foreign file


def cache_params(feature_type: str, cfg: Any) -> dict:
    """The dictionary whose JSON form is hashed (and stored in the manifest)."""
    if isinstance(cfg, Mapping):
        return {"feature_type": feature_type, **cfg}
    if not is_dataclass(cfg):
        raise TypeError("cfg must be an MfccConfig-like dataclass or a dict")
    values = {f.name: getattr(cfg, f.name) for f in fields(cfg)}
    if not values.get("n_fft"):
        values["n_fft"] = values["frame_length"]
    if values.get("f_max") is None:
        values["f_max"] = values["sample_rate"] / 2
    return {"feature_type": feature_type, **values}


def cache_digest(params: Mapping) -> str:
    text = json.dumps(dict(params), sort_keys=True, ensure_ascii=True)
    return hashlib.sha1(text.encode("utf-8")).hexdigest()[:12]


def write_npy_atomic(path: Path, array: np.ndarray) -> None:
    """np.save under a unique temporary name in the target directory, then rename over `path`."""
    path.parent.mkdir(parents=True, exist_ok=True)
    scratch = path.parent / f"{path.name}.{uuid.uuid4().hex}.tmp"
    try:
        with open(scratch, "wb") as handle:
            np.save(handle, array)
        os.replace(scratch, path)
    except BaseException:
        scratch.unlink(missing_ok=True)
        raise


def read_npy_shape(path: Path) -> tuple:
    """Shape from the .npy header alone (the manifest needs it for files that were already cached)."""
    with open(path, "rb") as handle:
        major, _minor = np.lib.format.read_magic(handle)
        reader = np.lib.format.read_array_header_1_0 if major == 1 else np.lib.format.read_array_header_2_0
        return tuple(reader(handle)[0])


def _features_per_clip(clips: list, cfg: Any, feature_types: tuple, normalize: bool = True) -> dict:
    """{feature_type: one [n_frames, n_coef] array per clip}: one batch when the clips have one length, else one
    ragged launch."""
    from .batch import features_batch, features_ragged, split_ragged

    if len({c.shape for c in clips}) == 1:
        out = features_batch(np.stack(clips, axis=0), cfg, feature_types, normalize=normalize)
        return {ft: list(out[ft]) for ft in feature_types}
    out = features_ragged(clips, cfg, feature_types, normalize=normalize)
    return {ft: split_ragged(out[ft], out["frame_offsets"]) for ft in feature_types}


def _record(item, path: Path, shape) -> dict:
    return {"filename": item.filename, "fold": item.fold, "path": str(path), "shape": [int(s) for s in shape]}


class BatchFeatureCache:
    """Same directory layout and files as the reference's FeatureCache, filled a batch at a time."""

    def __init__(self, root: str | Path = "outputs/features", enabled: bool = True):
        self.root = Path(root)
        self.enabled = enabled

    # ---- naming --------------------------------------------------------------------------------------
    def params_hash(self, feature_type: str, cfg: Any) -> tuple[str, dict]:
        params = cache_params(feature_type, cfg)
        return cache_digest(params), params

    def feature_dir(self, feature_type: str, cfg: Any) -> Path:
        return self.root.joinpath(feature_type, cache_digest(cache_params(feature_type, cfg)))

    def feature_path(self, item, feature_type: str, cfg: Any) -> Path:
        return self.feature_dir(feature_type, cfg).joinpath(f"fold{item.fold}", item.filename + ".npy")

    # ---- I/O -----------------------------------------------------------------------------------------
    def load_feature(self, item, feature_type: str, cfg: Any) -> np.ndarray | None:
        """The cached array, or None on a miss.  An unreadable file counts as a miss and is deleted,
        so that the next writer replaces it (cache.py:56-63)."""
        if not self.enabled:
            return None
        path = self.feature_path(item, feature_type, cfg)
        if not path.is_file():
            return None
        try:
            return np.load(path)
        except _UNREADABLE:
            path.unlink(missing_ok=True)
            return None

    def save_feature(self, path: Path, feat: np.ndarray) -> None:
        """Reference-named single-file writer (cache.py:89-94)."""
        write_npy_atomic(Path(path), np.asarray(feat))

    def compute_feature(self, item, feature_type: str, cfg: Any) -> np.ndarray:
        """One clip from item.path: load_audio + normalize_audio + the fused kernel (cache.py:65-74)."""
        return self._compute([item], feature_type, cfg, None)[0]

    def get_feature(self, item, feature_type: str, cfg: Any) -> np.ndarray:
        """Reference-named per-item access (cache.py:76-87): cache hit, else compute and store."""
        return self.get_features([item], feature_type, cfg)[0]

    def _compute(self, items: Sequence[Any], feature_type: str, cfg: Any, loader) -> list:
        from .retrieval import _load_clips

        if feature_type not in FEATURE_TYPES:
            raise ValueError(f"Unsupported feature_type: {feature_type}")
        if isinstance(cfg, Mapping):
            raise ValueError("get_feature requires MfccConfig for mfcc/log_mel")      # cache.py:83
        return _features_per_clip(_load_clips(list(items), cfg, loader), cfg, (feature_type,))[feature_type]

    def get_features(self, items: Sequence[Any], feature_type: str, cfg: Any, loader=None, batch: int = 256,
                     workers: int = 8) -> list:
        """Batched get_feature: hits are read, misses are computed `batch` clips at a time on the GPU and
        written in the reference's format.  Returns float32 [n_frames, n_coef] arrays in item order."""
        items = list(items)
        feats = [self.load_feature(it, feature_type, cfg) for it in items]
        missing = [i for i, f in enumerate(feats) if f is None]
        for s in range(0, len(missing), batch):
            rows = missing[s:s + batch]
            made = self._compute([items[i] for i in rows], feature_type, cfg, loader)
            for i, f in zip(rows, made):
                feats[i] = np.ascontiguousarray(f, dtype=np.float32)
            if self.enabled:
                base = self.feature_dir(feature_type, cfg)
                jobs = [(base.joinpath(f"fold{items[i].fold}", items[i].filename + ".npy"), feats[i]) for i in rows]
                with ThreadPoolExecutor(max_workers=max(1, workers)) as pool:
                    for _ in pool.map(lambda job: write_npy_atomic(*job), jobs):
                        pass
        return feats

    def save_features(self, items: Sequence[Any], feats: np.ndarray, feature_type: str, cfg: Any,
                      workers: int = 8) -> list[dict]:
        """Write feats[i] ([n_frames, n_coef]) for items[i]; returns the manifest records.  feats is one array
        [N, n_frames, n_coef] or a list of N arrays (clips of different lengths)."""
        if feature_type not in FEATURE_TYPES:
            raise ValueError(f"Unsupported feature_type: {feature_type}")
        if not isinstance(feats, (list, tuple)):
            feats = np.asarray(feats)
        if len(feats) != len(items):
            raise ValueError("one feature array per item expected")
        base = self.feature_dir(feature_type, cfg)                      # hash once per batch, not per file
        jobs = [(base.joinpath(f"fold{it.fold}", it.filename + ".npy"), np.ascontiguousarray(feats[i], dtype=np.float32))
                for i, it in enumerate(items)]
        if workers > 1 and len(jobs) > 1:
            with ThreadPoolExecutor(max_workers=workers) as pool:
                for _ in pool.map(lambda job: write_npy_atomic(*job), jobs):
                    pass
        else:
            for job in jobs:
                write_npy_atomic(*job)
        return [_record(it, path, arr.shape) for it, (path, arr) in zip(items, jobs)]

    def write_manifest(self, feature_type: str, cfg: Any, records: Iterable[dict]) -> Path:
        digest, params = self.params_hash(feature_type, cfg)
        files = list(records)
        stamp = datetime.now(timezone.utc).replace(tzinfo=None).isoformat() + "Z"
        body = dict(zip(MANIFEST_KEYS, (feature_type, digest, params, stamp, len(files), files)))
        target = self.root.joinpath(feature_type, digest, "manifest.json")
        target.parent.mkdir(parents=True, exist_ok=True)
        target.write_text(json.dumps(body, indent=2, ensure_ascii=True), encoding="utf-8")
        return target

    # ---- batched precompute (GPU) --------------------------------------------------------------------
    def precompute(self, items: Sequence[Any], cfg: Any, feature_types: Iterable[str] = FEATURE_TYPES,
                   clips: np.ndarray | None = None, loader: Callable[[Any], np.ndarray] | None = None,
                   batch: int = 256, workers: int = 8, normalize: bool = True, skip_existing: bool = True) -> dict:
        """Fill the cache for `items`: the batched twin of precompute_features.py:62-113.

        Audio comes from `clips` ([N, L] float32 already loaded/normalised, or int16 PCM which is
        converted and peak-normalised on the GPU; or a list of N clips of different lengths) or from
        `loader(item)` (decoding files is out of scope here).  A batch of clips of different lengths is
        one ragged launch.  Returns {feature_type: manifest path}.
        """
        feature_types = tuple(feature_types)
        for ft in feature_types:
            if ft not in FEATURE_TYPES:
                raise ValueError(f"Unsupported feature_type: {ft}")
        items = list(items)
        if clips is None and loader is None:
            raise ValueError("precompute needs clips or a loader")
        dirs = {ft: self.feature_dir(ft, cfg) for ft in feature_types}
        records = {ft: [] for ft in feature_types}
        for s in range(0, len(items), batch):
            chunk = items[s:s + batch]
            paths = {ft: [dirs[ft].joinpath(f"fold{it.fold}", it.filename + ".npy") for it in chunk] for ft in feature_types}
            todo = [i for i in range(len(chunk))
                    if not (skip_existing and all(paths[ft][i].is_file() for ft in feature_types))]
            if todo:
                if clips is not None:
                    x = [np.asarray(clips[s + i]) for i in todo]
                else:
                    x = [np.asarray(loader(chunk[i])) for i in todo]
                out = _features_per_clip(x, cfg, feature_types, normalize=normalize)
                for ft in feature_types:
                    self.save_features([chunk[i] for i in todo], out[ft], ft, cfg, workers=workers)
            for ft in feature_types:
                records[ft].extend(_record(it, p, read_npy_shape(p)) for it, p in zip(chunk, paths[ft]))
        return {ft: self.write_manifest(ft, cfg, records[ft]) for ft in feature_types}
