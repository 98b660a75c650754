"""Row f1: the batched cache writer produces the reference's cache, byte for byte."""
from __future__ import annotations

import hashlib
import json
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import GOLDEN


def _items(n):
    return [SimpleNamespace(filename=f"{1 + i // 400}-{100000 + i}-A-{i % 50}.wav", fold=1 + i // 400, target=i % 50)
            for i in range(n)]


def test_digests_and_paths_are_the_published_ones(tmp_path, known_answers):
    from dsp_final_b200.cache import BatchFeatureCache
    from dsp_final_b200.dsp.mfcc import MfccConfig

    bc = BatchFeatureCache(tmp_path)
    for key, want in known_answers["cache_digests"].items():
        ft, fl, hop, *rest = key.split("/")
        cfg = MfccConfig(44100, int(fl), int(hop), **({"n_mels": 128} if rest else {}))
        assert bc.params_hash(ft, cfg)[0] == want, key
    cfg = MfccConfig(44100, 1024, 512)
    assert bc.params_hash("mfcc", cfg)[1] == known_answers["cache_params_mfcc_1024_512"]
    it = _items(1)[0]
    assert bc.feature_path(it, "mfcc", cfg) == tmp_path / "mfcc" / "e637fe1e8db0" / "fold1" / f"{it.filename}.npy"
    # dict configs are hashed verbatim, no n_fft / f_max defaulting (cache.py:35-38; how retrieval_ml.py keys its
    # embedding_* caches): digests below were produced by the reference's FeatureCache.params_hash
    assert bc.params_hash("mfcc", {"sample_rate": 44100, "frame_length": 1024, "hop_length": 512, "n_fft": None,
                                   "n_mels": 40, "n_mfcc": 13, "f_min": 0.0, "f_max": None, "pre_emphasis": 0.97,
                                   "window": "hann"})[0] == "6f264003971b"
    assert bc.params_hash("embedding_panns", {"model": "cnn14", "sr": 32000})[0] == "b2b4aab840f8"


def test_save_load_manifest_roundtrip(tmp_path):
    from dsp_final_b200.cache import BatchFeatureCache
    from dsp_final_b200.dsp.mfcc import MfccConfig

    bc = BatchFeatureCache(tmp_path)
    cfg = MfccConfig(44100, 1024, 512)
    items = _items(5)
    feats = np.random.default_rng(0).standard_normal((5, 429, 13))            # float64 in -> float32 on disk
    recs = bc.save_features(items, feats, "mfcc", cfg, workers=3)
    for i, it in enumerate(items):
        got = bc.load_feature(it, "mfcc", cfg)
        assert got.dtype == np.float32 and got.flags["C_CONTIGUOUS"]
        assert np.array_equal(got, feats[i].astype(np.float32))
    m = json.loads(bc.write_manifest("mfcc", cfg, recs).read_text())
    assert list(m) == ["feature_type", "hash", "params", "created_at", "num_files", "files"]
    assert m["num_files"] == 5 and m["hash"] == "e637fe1e8db0" and m["files"][0]["shape"] == [429, 13]
    assert set(m["files"][0]) == {"filename", "fold", "path", "shape"}
    # corrupt file self-heals to a miss (cache.py:56-63)
    p = bc.feature_path(items[0], "mfcc", cfg)
    p.write_bytes(b"not an npy")
    assert bc.load_feature(items[0], "mfcc", cfg) is None and not p.exists()
    with pytest.raises(ValueError):
        bc.save_features(items, feats, "chroma", cfg)
    assert not list(tmp_path.rglob("*.tmp"))


def test_reference_cache_reads_our_files_and_bytes_match(tmp_path, known_answers):
    """Our cache files are the reference's, byte for byte, so its FeatureCache reads them as its own.

    tests/golden/pipeline.npz holds what the reference's FeatureCache wrote for the 40-item pipeline set
    (tests/golden/make_pipeline_golden.py): the header of its first .npy file, that file's path under the cache root
    and np.load of every file.  Header + payload is therefore the reference's file exactly; all 40 share one shape and
    so one header.  Its params dict and digest for this config are in known_answers.json."""
    from dsp_final_b200.cache import BatchFeatureCache
    from dsp_final_b200.dsp.mfcc import MfccConfig

    g = np.load(GOLDEN / "pipeline.npz")
    feats, header = g["mfcc_f32"], bytes(g["npy_header"])
    items = [SimpleNamespace(filename=f"{1 + n // 8}-{100000 + n}-A-{n % 5}.wav", fold=1 + n // 8)   # item_table()
             for n in range(feats.shape[0])]
    cfg = MfccConfig(44100, 1024, 512)
    ours = BatchFeatureCache(tmp_path)
    recs = ours.save_features(items, feats, "mfcc", cfg)
    assert str(ours.feature_path(items[0], "mfcc", cfg).relative_to(tmp_path)) == bytes(g["first_path"]).decode()
    for i, it in enumerate(items):
        blob = ours.feature_path(it, "mfcc", cfg).read_bytes()
        assert hashlib.sha1(blob).hexdigest() == hashlib.sha1(header + feats[i].tobytes()).hexdigest(), it.filename
    m = json.loads(ours.write_manifest("mfcc", cfg, recs).read_text())
    assert list(m) == ["feature_type", "hash", "params", "created_at", "num_files", "files"]
    assert m["feature_type"] == "mfcc" and m["num_files"] == len(items)
    assert m["hash"] == known_answers["cache_digests"]["mfcc/1024/512"]
    assert m["params"] == known_answers["cache_params_mfcc_1024_512"]


@pytest.mark.gpu
def test_precompute_on_gpu_writes_reference_cache(tmp_path):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dsp_final_b200 import synth
    from dsp_final_b200.cache import BatchFeatureCache
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    items = _items(20)
    clips = synth.host_clips(20, seed=9, length=30_000)
    cfg = MfccConfig(44100, 1024, 512)
    bc = BatchFeatureCache(tmp_path)
    manifests = bc.precompute(items, cfg, ("mfcc", "log_mel"), clips=clips, batch=8)
    ref = O.features_batch(clips, O.OracleConfig(44100, 1024, 512), want=("mfcc", "log_mel"))
    for i, it in enumerate(items):
        for ft in ("mfcc", "log_mel"):
            got = bc.load_feature(it, ft, cfg)
            assert got.dtype == np.float32
            assert O.relative_error(got, ref[ft][i]) < 1e-4
    m = json.loads(manifests["mfcc"].read_text())
    assert m["num_files"] == 20 and m["files"][3]["shape"] == [57, 13]
    # second call is all cache hits and rewrites only the manifest
    before = {p: p.stat().st_mtime_ns for p in tmp_path.rglob("*.npy")}
    bc.precompute(items, cfg, ("mfcc", "log_mel"), clips=clips, batch=8)
    assert before == {p: p.stat().st_mtime_ns for p in tmp_path.rglob("*.npy")}
