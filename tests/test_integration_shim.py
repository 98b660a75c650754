"""The reference's own src/features and src/retrieval run unchanged on top of our src/dsp shims.

Runs when DSP_REF_PATH names a reference checkout: a path overlay puts integration/src/dsp in place of the
reference's src/dsp while every other reference module is imported from the reference checkout.
Without a checkout the same pipeline (Esc50Meta -> FeatureCache-format files ->
compute_embeddings -> evaluate_retrieval / run_mfcc_retrieval) is exercised by tests/test_pipeline.py
against golden outputs that the reference produced here (tests/golden/make_pipeline_golden.py).
"""
from __future__ import annotations

import importlib
import sys
import types
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import REFERENCE, REPO

pytestmark = pytest.mark.needs_reference


@pytest.fixture()
def overlay():
    saved = {k: v for k, v in sys.modules.items() if k == "src" or k.startswith("src.")}
    for k in saved:
        del sys.modules[k]
    pkg = types.ModuleType("src")
    pkg.__path__ = [str(REPO / "integration" / "src"), str(REFERENCE / "src")]     # ours first: src.dsp resolves here
    sys.modules["src"] = pkg
    sys.dont_write_bytecode = True
    yield
    for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
        del sys.modules[k]
    sys.modules.update(saved)


def test_reference_cache_runs_on_our_dsp(overlay, tmp_path, known_answers):
    dsp_mfcc = importlib.import_module("src.dsp.mfcc")
    assert Path(dsp_mfcc.__file__).is_relative_to(REPO / "integration")
    cache_mod = importlib.import_module("src.features.cache")            # the reference's file, unmodified
    assert Path(cache_mod.__file__).is_relative_to(REFERENCE)
    assert cache_mod.MfccConfig is dsp_mfcc.MfccConfig                   # it picked up OUR config class
    fc = cache_mod.FeatureCache(tmp_path)
    for key, want in known_answers["cache_digests"].items():
        ft, fl, hop, *rest = key.split("/")
        kw = {"n_mels": 128} if rest else {}
        cfg = dsp_mfcc.MfccConfig(sample_rate=44100, frame_length=int(fl), hop_length=int(hop), **kw)
        assert fc.params_hash(ft, cfg)[0] == want, key
    for key, want in known_answers["published_digests"].items():
        ft, fl, hop = key.split("/")
        cfg = dsp_mfcc.MfccConfig(sample_rate=44100, frame_length=int(fl), hop_length=int(hop))
        assert fc.feature_dir(ft, cfg).name == want
    # save / load round trip of a float32 feature through the reference's own writer
    item = SimpleNamespace(filename="1-100032-A-0.wav", fold=1)
    cfg = dsp_mfcc.MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    feat = np.arange(429 * 13, dtype=np.float32).reshape(429, 13)
    path = fc.feature_path(item, "mfcc", cfg)
    fc.save_feature(path, feat)
    assert path == tmp_path / "mfcc" / "e637fe1e8db0" / "fold1" / "1-100032-A-0.wav.npy"
    assert np.array_equal(fc.load_feature(item, "mfcc", cfg), feat)


def test_reference_retrieval_module_imports_on_our_dsp(overlay):
    ret = importlib.import_module("src.retrieval.retrieval")             # reference file; imports src.dsp.mfcc
    assert Path(ret.__file__).is_relative_to(REFERENCE)
    ours = importlib.import_module("dsp_final_b200.dsp.mfcc")     # (the package re-exports the function `mfcc` too)

    assert ret.mfcc is ours.mfcc and ret.MfccConfig is ours.MfccConfig
    tr = importlib.import_module("src.train.transforms")
    assert tr.log_mel_spectrogram is ours.log_mel_spectrogram
