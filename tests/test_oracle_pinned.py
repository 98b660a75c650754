"""Pins the CPU oracle (oracle/dsp_oracle.c) to the reference.

Golden vectors are outputs of the reference itself (tests/golden/make_golden.py);
known answers are numbers the reference published (SURVEY.md section 4).  The
oracle is float64 like the reference, so the bar here is 1e-12 relative -- far
tighter than the 1e-4 the CUDA path is later held to against this oracle.
"""
from __future__ import annotations

import hashlib

import numpy as np
import pytest

from conftest import REFERENCE, rel_err
from oracle import oracle as O

TIGHT = 1e-12


def _sha12(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:12]


def _cfg(m):
    return O.OracleConfig(**m)


def test_features_small_all_cases(golden_small):
    z, meta = golden_small
    clips = z["clips"]
    for ci, m in enumerate(meta):
        cfg = _cfg(m)
        for b in range(clips.shape[0]):
            assert rel_err(O.mfcc(clips[b], cfg), z[f"c{ci}_mfcc_{b}"]) < TIGHT, (ci, b)
            assert rel_err(O.log_mel_spectrogram(clips[b], cfg), z[f"c{ci}_logmel_{b}"]) < TIGHT, (ci, b)
        s = O.stft(clips[0], m["frame_length"], m["hop_length"], m["window"], m["n_fft"])
        ref = z[f"c{ci}_stft_0"]
        assert s.shape == ref.shape
        assert rel_err(s, ref) < TIGHT, ci


def test_silence_hits_the_log_floor(golden_small):
    z, meta = golden_small
    lm = O.log_mel_spectrogram(z["clips"][2], _cfg(meta[4]))
    assert np.isclose(lm[-1], np.log(1e-10)).all()
    assert np.array_equal(lm[-1] == np.log(1e-10), z["c4_logmel_2"][-1] == np.log(1e-10))


def test_config1_full_clip(golden_config1):
    g = golden_config1
    x = g["clip"]
    cfg = O.OracleConfig(44100, 1024, 512)
    assert rel_err(O.mfcc(x, cfg), g["mfcc"]) < TIGHT
    assert rel_err(O.log_mel_spectrogram(x, cfg), g["logmel"]) < TIGHT
    s = O.stft(x, 1024, 512)
    assert tuple(g["stft_shape"]) == s.shape == (429, 513)
    assert rel_err(s[g["stft_frames"]], g["stft_sel"]) < TIGHT
    assert abs(np.linalg.norm(s) / float(g["stft_abs_fro"]) - 1) < TIGHT


def test_real_clip_excerpt(golden_real):
    g = golden_real
    x = g["pcm16"].astype(np.float32) / np.float32(32768.0)
    xn = x / np.max(np.abs(x))
    cfg = O.OracleConfig(44100, 1024, 512)
    assert rel_err(O.stft(x, 1024, 512), g["stft"]) < TIGHT
    assert rel_err(O.mfcc(xn, cfg), g["mfcc"]) < TIGHT
    assert rel_err(O.log_mel_spectrogram(xn, cfg), g["logmel"]) < TIGHT


def test_published_librosa_stft_number(golden_real, known_answers):
    """The reference's recorded stft_complex_rel_error is reproduced to 1e-12."""
    got = float(golden_real["librosa_style_stft_rel"])
    want = known_answers["librosa_compare_published_stft_complex_rel_error"]
    assert abs(got / want - 1) < 1e-12


def test_fft_family(golden_fft):
    g = golden_fft
    for i in range(int(g["n_cases"])):
        z = g[f"in_{i}"]
        n = int(g[f"n_{i}"])
        n = None if n < 0 else n
        for name, fn, arg in (("fft", O.fft, z), ("ifft", O.ifft, z), ("rfft", O.rfft, z.real)):
            y = fn(arg, n)
            assert y.shape[0] == int(g[f"{name}_len_{i}"]), (name, i)
            ref = g[f"{name}_{i}"]
            scale = float(g[f"{name}_norm_{i}"]) / np.sqrt(y.shape[0]) + 1e-300
            assert np.max(np.abs(y[g[f"{name}_sel_{i}"]] - ref)) <= 1e-11 * max(scale, 1.0), (name, i)


def test_fft_rounds_length_up_to_pow2():
    assert O.fft([1, 2, 3], n=3).shape == (4,)        # SURVEY appendix A.5
    assert O.stft(np.ones(2000), 1000, 500).shape == (3, 513)


def test_tables_bit_exact(known_answers):
    ka = known_answers["table_sha12"]
    for key, want in ka.items():
        kind, a, *rest = key.split("/")
        if kind == "fbank":
            got = _sha12(O.mel_filterbank(int(a), int(rest[0]), 44100))
        elif kind == "dct":
            got = _sha12(O.dct_basis(int(a), int(rest[0])))
        else:
            got = _sha12(O.get_window(kind, int(a)))
        assert got == want, key


def test_mel_edges_known_answer(known_answers):
    fb = O.mel_filterbank(40, 1024, 44100)
    edges = known_answers["mel_edges_1024_40"]
    for m in range(40):
        nz = np.nonzero(fb[m])[0]
        assert nz[0] >= edges[m] and nz[-1] < edges[m + 2]
        assert fb[m, edges[m + 1]] == 1.0
    assert np.count_nonzero(fb) == 940 and not fb[:, 512].any()


def test_errors():
    with pytest.raises(ValueError):
        O.get_window("blackman", 8)
    with pytest.raises(ValueError):
        O.stft(np.ones(100), 1024, 512)               # shorter than one frame
    with pytest.raises(ValueError):
        O.stft(np.ones(100), 16, 0)


def test_embedding_matches_numpy():
    f = np.random.default_rng(0).standard_normal((429, 13))
    e = O.embedding(f)
    assert np.allclose(e[:13], f.mean(0), rtol=1e-13, atol=1e-15)
    assert np.allclose(e[13:], f.std(0), rtol=1e-12)


def test_retrieval_indices_and_precision(golden_retrieval):
    g = golden_retrieval
    emb, folds, targets = g["emb"], g["folds"], g["targets"]
    db, q = emb[folds <= 4], emb[folds == 5]
    idx = O.cosine_topk(q, db, 20)
    assert np.array_equal(idx, g["top20_f64"])
    # stable argsort prefix property: top-10 is the first ten of top-20
    assert np.array_equal(O.cosine_topk(q, db, 10), g["top20_f64"][:, :10])
    res = O.evaluate_retrieval(targets[folds <= 4], targets[folds == 5], db, q, (10, 20))
    assert [r[1] for r in res] == list(g["prec_f64"])
    # float32 (cached-path) reference agrees on every query whose gap is resolvable in float32
    same = (g["top20_f32"] == g["top20_f64"]).all(axis=1).mean()
    assert same > 0.97
    assert list(g["prec_f32"]) == list(g["prec_f64"])


def test_retrieval_ties_lowest_index_first(golden_retrieval):
    g = golden_retrieval
    emb, folds = g["emb"], g["folds"]
    db = emb[folds <= 4].astype(np.float64).copy()
    r = g["tie_db_rows"]
    db[r[1]] = db[r[0]]
    db[r[2]] = db[r[0]]
    idx = O.cosine_topk(emb[folds == 5], db, 20)
    assert np.array_equal(idx, g["top20_ties_f64"])
    rows = [row for row in idx if r[0] in row and r[1] in row]
    assert rows and all(list(row).index(r[0]) + 1 == list(row).index(r[1]) for row in rows)


def test_batch_front_end_matches_single(golden_small):
    z, meta = golden_small
    cfg = _cfg(meta[4])
    out = O.features_batch(z["clips"], cfg)
    for b in range(3):
        assert np.array_equal(out["mfcc"][b], O.mfcc(z["clips"][b], cfg).astype(np.float32))
        assert np.array_equal(out["log_mel"][b], O.log_mel_spectrogram(z["clips"][b], cfg).astype(np.float32))
        e = O.embedding(out["mfcc"][b].astype(np.float64)).astype(np.float32)
        assert np.array_equal(out["embed"][b], e)


@pytest.mark.needs_reference
def test_oracle_against_live_reference():
    """A fresh random case straight against the original project (its checkout named by DSP_REF_PATH)."""
    import sys

    sys.dont_write_bytecode = True
    sys.path.insert(0, str(REFERENCE))
    try:
        from src.dsp.mfcc import MfccConfig, mfcc
    finally:
        sys.path.remove(str(REFERENCE))
    x = np.random.default_rng(99).standard_normal(6000).astype(np.float32)
    cfg = MfccConfig(sample_rate=16000, frame_length=400, hop_length=160, n_mels=23, n_mfcc=13)
    ours = O.mfcc(x, O.OracleConfig(16000, 400, 160, n_mels=23, n_mfcc=13))
    assert rel_err(ours, mfcc(x, cfg)) < TIGHT
