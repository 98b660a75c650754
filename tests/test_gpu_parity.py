"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C ABI
of libdspx.so via the ctypes binding; the checker is the CPU oracle and the committed golden
vectors (outputs of the reference itself).  Nothing here reads /root/reference.

Tolerance for floating-point features: relative Frobenius error <= 1e-4 (BASELINE.json
north_star; metric of scripts/tools/compare_librosa.py:37-38) plus an elementwise bound of
1e-4 * max|ref|.  Retrieval indices: bit-exact.
"""
from __future__ import annotations

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-4


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def _close(got, ref, what=""):
    got = np.asarray(got, dtype=np.float64) if not np.iscomplexobj(got) else np.asarray(got)
    e = rel_err(got, ref)
    assert e <= TOL, f"{what}: rel err {e:.3e}"
    assert np.max(np.abs(got - ref)) <= TOL * np.max(np.abs(ref)) + 1e-30, f"{what}: max abs err"
    return e


KERNELS = ("generic", "auto")


@pytest.mark.parametrize("kernel", KERNELS)
def test_golden_small_cases(torch_cuda, golden_small, kernel):
    from dsp_final_b200.batch import features_batch, stft_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig

    z, meta = golden_small
    clips = z["clips"]
    for ci, m in enumerate(meta):
        cfg = MfccConfig(**m)
        for src in (clips, torch_cuda.as_tensor(clips).cuda()):
            out = features_batch(src, cfg, ("log_mel", "mfcc"), kernel=kernel)
            for b in range(clips.shape[0]):
                mf = out["mfcc"][b]
                lm = out["log_mel"][b]
                mf = mf.cpu().numpy() if hasattr(mf, "cpu") else mf
                lm = lm.cpu().numpy() if hasattr(lm, "cpu") else lm
                _close(mf, z[f"c{ci}_mfcc_{b}"], f"case {ci} clip {b} mfcc [{kernel}]")
                _close(lm, z[f"c{ci}_logmel_{b}"], f"case {ci} clip {b} log-mel [{kernel}]")
        s = stft_batch(clips[:1], m["frame_length"], m["hop_length"], m["window"], m["n_fft"])[0]
        assert s.shape == z[f"c{ci}_stft_0"].shape
        _close(s, z[f"c{ci}_stft_0"], f"case {ci} stft")


def test_reference_signatures_config1(torch_cuda, golden_config1):
    """BASELINE.json configs[0]: one 5 s clip through the reference-named entry points."""
    from dsp_final_b200.dsp.mfcc import MfccConfig, log_mel_spectrogram, mfcc
    from dsp_final_b200.dsp.stft import stft

    g = golden_config1
    x = g["clip"]
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    mf, lm, s = mfcc(x, cfg), log_mel_spectrogram(x, cfg), stft(x, 1024, 512)
    assert mf.dtype == np.float64 and mf.shape == (429, 13)
    assert lm.dtype == np.float64 and lm.shape == (429, 40)
    assert s.dtype == np.complex128 and s.shape == (429, 513)
    e = {"mfcc": _close(mf, g["mfcc"], "mfcc"), "log_mel": _close(lm, g["logmel"], "log-mel"),
         "stft": _close(s[g["stft_frames"]], g["stft_sel"], "stft"),
         "stft_mag": _close(np.abs(s[g["stft_frames"]]), np.abs(g["stft_sel"]), "|stft|")}
    print("config1 rel errors", e)
    # float32 round trip of the cache (src/features/cache.py:74) is lossless
    assert np.array_equal(mf.astype(np.float32).astype(np.float64), mf)


def test_real_clip_excerpt(torch_cuda, golden_real):
    from dsp_final_b200.dsp.mfcc import MfccConfig, log_mel_spectrogram, mfcc
    from dsp_final_b200.dsp.stft import stft

    g = golden_real
    x = g["pcm16"].astype(np.float32) / np.float32(32768.0)
    xn = x / np.max(np.abs(x))
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    _close(stft(x, 1024, 512), g["stft"], "real stft")
    _close(mfcc(xn, cfg), g["mfcc"], "real mfcc")
    _close(log_mel_spectrogram(xn, cfg), g["logmel"], "real log-mel")


@pytest.mark.parametrize("kernel", KERNELS)
def test_batch_against_oracle_and_properties(torch_cuda, kernel):
    """Seeded ESC-50-shaped clips: oracle parity on a sample + size-independent properties."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    ocfg = O.OracleConfig(44100, 1024, 512)
    n = 96
    clips = synth.host_clips(n, seed=1234)
    dev = torch.as_tensor(clips).cuda()
    out = features_batch(dev, cfg, ("log_mel", "mfcc", "embed"), kernel=kernel)
    mf, lm, em = (out[k].cpu().numpy() for k in ("mfcc", "log_mel", "embed"))
    assert mf.shape == (n, 429, 13) and lm.shape == (n, 429, 40) and em.shape == (n, 26)
    sel = [0, 1, 17, 50, 95]
    ref = O.features_batch(clips[sel], ocfg)
    for j, i in enumerate(sel):
        _close(mf[i], ref["mfcc"][j], f"clip {i} mfcc")
        _close(lm[i], ref["log_mel"][j], f"clip {i} log-mel")
        _close(em[i], ref["embed"][j], f"clip {i} embed")
    # (a) batch invariance: a clip alone gives bit-identical features
    alone = features_batch(dev[17:18], cfg, ("mfcc",), kernel=kernel)["mfcc"].cpu().numpy()
    assert np.array_equal(alone[0], mf[17])
    # (b) host-buffer ABI == device-pointer ABI, bit for bit (pageable and pinned callers)
    host_out = features_batch(clips[:40], cfg, ("log_mel", "mfcc", "embed"), kernel=kernel)
    assert np.array_equal(host_out["mfcc"], mf[:40]) and np.array_equal(host_out["log_mel"], lm[:40])
    assert np.array_equal(host_out["embed"], em[:40])
    # (c) time-shift equivariance: dropping one hop of samples shifts the frames by one
    shifted = features_batch(dev[:4, 512:].contiguous(), cfg, ("mfcc",), kernel=kernel)["mfcc"].cpu().numpy()
    np.testing.assert_allclose(shifted[:, 1:], mf[:4, 2:], rtol=0, atol=2e-3)
    assert rel_err(shifted[:, 1:], mf[:4, 2:]) < 1e-5
    # (d) gain: doubling the signal adds ln 4 to every log-mel cell above the floor
    lm2 = features_batch(dev[:4] * 2.0, cfg, ("log_mel",), kernel=kernel)["log_mel"].cpu().numpy()
    above = lm[:4] > np.log(1e-10) + 2.0
    assert np.allclose((lm2 - lm[:4])[above], np.log(4.0), atol=5e-5)
    # (e) strided rows (clip_stride > clip_len) read the same samples
    wide = torch.zeros((8, 220_500 + 300), device="cuda")
    wide[:, :220_500] = dev[:8]
    strided = features_batch(wide[:, :220_500], cfg, ("mfcc",), kernel=kernel)["mfcc"].cpu().numpy()
    assert np.array_equal(strided, mf[:8])


def test_host_pipeline_many_chunks(torch_cuda):
    """More clips than one pipeline chunk, pinned and pageable: identical to the device path."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig

    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    base = synth.host_clips(8, seed=3)
    clips = np.concatenate([base * (1.0 - 0.01 * i) for i in range(25)]).astype(np.float32)   # 200 clips > 3 chunks
    ref = features_batch(torch.as_tensor(clips).cuda(), cfg, ("mfcc", "log_mel"))
    got = features_batch(clips, cfg, ("mfcc", "log_mel"))
    assert np.array_equal(got["mfcc"], ref["mfcc"].cpu().numpy())
    assert np.array_equal(got["log_mel"], ref["log_mel"].cpu().numpy())
    pinned = torch.as_tensor(clips).pin_memory()
    got2 = features_batch(pinned.numpy(), cfg, ("mfcc",))
    assert np.array_equal(got2["mfcc"], got["mfcc"])


def test_fft_family(torch_cuda, golden_fft):
    from dsp_final_b200.dsp.fft import fft, ifft, rfft

    g = golden_fft
    for i in range(int(g["n_cases"])):
        z = g[f"in_{i}"]
        n = int(g[f"n_{i}"])
        n = None if n < 0 else n
        for name, fn, arg in (("fft", fft, z), ("ifft", ifft, z), ("rfft", rfft, z.real)):
            y = fn(arg, n)
            assert y.dtype == np.complex128 and y.shape[0] == int(g[f"{name}_len_{i}"]), (name, i)
            ref = g[f"{name}_{i}"]
            got = y[g[f"{name}_sel_{i}"]]
            scale = float(g[f"{name}_norm_{i}"]) / np.sqrt(y.shape[0])
            assert np.linalg.norm(got - ref) <= 1e-5 * (scale * np.sqrt(len(ref)) + 1e-30) + 1e-30, (name, i)
    x = np.random.default_rng(0).standard_normal(300) + 1j * np.random.default_rng(1).standard_normal(300)
    back = ifft(fft(x))[:300]                       # round trip through the zero-padded length 512
    assert rel_err(back, x) < 1e-5
    assert fft([1, 2, 3], n=3).shape == (4,)


def test_errors_follow_the_reference(torch_cuda):
    from dsp_final_b200.dsp.mfcc import MfccConfig, mfcc
    from dsp_final_b200.dsp.stft import stft
    from dsp_final_b200.dsp.stft import _get_window, frame_signal

    x = np.zeros(4000, np.float32)
    with pytest.raises(ValueError):
        stft(x, 1024, 0)
    with pytest.raises(ValueError):
        stft(x, 0, 10)
    with pytest.raises(ValueError):
        stft(x, 1024, 512, window="blackman")
    with pytest.raises(ValueError):
        _get_window("hann", 0)
    with pytest.raises(ValueError):
        frame_signal(x, 8, 0)
    with pytest.raises(ValueError):
        mfcc(np.zeros(100, np.float32), MfccConfig(44100, 1024, 512))   # shorter than one frame
    with pytest.raises(ValueError):
        mfcc(x, MfccConfig(44100, 1024, 512, window="nope"))
    # digital silence is legal input and sits on the 1e-10 floor
    out = mfcc(x, MfccConfig(44100, 1024, 512))
    assert np.isfinite(out).all() and np.allclose(out[:, 1:], 0.0, atol=1e-3)


def test_tables_on_device_match_reference_tables(torch_cuda, known_answers):
    from dsp_final_b200.dsp.mfcc import MfccConfig, _dct_basis, mel_filterbank
    from dsp_final_b200.dsp.stft import _get_window
    from dsp_final_b200.plan import get_plan

    for n_mels, fl in ((40, 1024), (128, 512), (40, 2048)):
        plan = get_plan(MfccConfig(44100, fl, fl // 2, n_mels=n_mels), 0, "generic")
        assert np.array_equal(plan.read_table("fbank"), mel_filterbank(n_mels, fl, 44100).astype(np.float32))
        assert np.array_equal(plan.read_table("window"), _get_window("hann", fl).astype(np.float32))
        assert np.array_equal(plan.read_table("dct2"), (2.0 * _dct_basis(13, n_mels)).astype(np.float32))


def test_embed_stats_and_dct(torch_cuda):
    from dsp_final_b200.batch import dct2_rows, embed_stats
    from dsp_final_b200.dsp.mfcc import _dct_basis, dct_type_2
    from oracle import oracle as O

    rng = np.random.default_rng(5)
    for t, c in ((429, 13), (7, 40), (300, 128), (50, 200)):
        f = rng.standard_normal((6, t, c)).astype(np.float32) * 10 + 3
        got = embed_stats(f)
        want = np.stack([O.embedding(f[i].astype(np.float64)) for i in range(6)])
        np.testing.assert_allclose(got, want, rtol=2e-6, atol=1e-6)
    x = rng.standard_normal((11, 40)).astype(np.float32)
    np.testing.assert_allclose(dct_type_2(x, 13), 2.0 * x.astype(np.float64) @ _dct_basis(13, 40).T, rtol=1e-5, atol=1e-5)
    assert dct2_rows(x[0], 5).shape == (5,)


def test_retrieval_golden_bit_exact(torch_cuda, golden_retrieval):
    from types import SimpleNamespace

    from dsp_final_b200 import retrieval as R

    g = golden_retrieval
    emb, folds, targets = g["emb"], g["folds"], g["targets"]
    db, q = emb[folds <= 4], emb[folds == 5]
    for dt in (np.float32, np.float64):
        idx = R.cosine_topk(q.astype(dt), db.astype(dt), 20)
        assert idx.dtype == np.int32 and np.array_equal(idx, g["top20_f64"])
    assert np.array_equal(R.cosine_topk(q, db, 10), g["top20_f64"][:, :10])
    items = lambda sel: [SimpleNamespace(target=int(t)) for t in targets[sel]]   # noqa: E731
    res = R.evaluate_retrieval(items(folds <= 4), items(folds == 5), db, q, (10, 20))
    assert [r.k for r in res] == [10, 20]
    assert [r.precision for r in res] == list(g["prec_f64"])
    # ties: duplicated database rows come back lowest index first
    dbt = db.astype(np.float64).copy()
    r = g["tie_db_rows"]
    dbt[r[1]] = dbt[r[0]]
    dbt[r[2]] = dbt[r[0]]
    assert np.array_equal(R.cosine_topk(q.astype(np.float64), dbt, 20), g["top20_ties_f64"])
    # the dense matrix entry point agrees with the reference formula and with the ranked scores
    sims = R.cosine_similarity(q.astype(np.float64), db.astype(np.float64))
    qn = q / (np.linalg.norm(q.astype(np.float64), axis=1, keepdims=True) + 1e-10)
    dn = db / (np.linalg.norm(db.astype(np.float64), axis=1, keepdims=True) + 1e-10)
    np.testing.assert_allclose(sims, qn @ dn.T, rtol=0, atol=1e-14)
    idx, sc = R.cosine_topk(q.astype(np.float64), db.astype(np.float64), 20, return_scores=True)
    assert np.array_equal(np.take_along_axis(sims, idx.astype(np.int64), axis=1), sc)
    with pytest.raises(ValueError):
        R.cosine_similarity(q, db[:, :13])


@pytest.mark.parametrize("dim,k", [(26, 20), (16, 7), (32, 40)])
def test_retrieval_float32_collisions(torch_cuda, dim, k):
    """The ranking kernel filters in float32 and re-scores in float64: clusters of database rows whose scores
    differ only below float32 resolution (and exact duplicates) must still come back in the oracle's order."""
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(dim * 31 + k)
    nq, ndb = 150, 6000
    q = rng.standard_normal((nq, dim))
    db = rng.standard_normal((ndb, dim))
    for c in range(12):                                    # 12 clusters of 60 rows around a query direction
        rows = rng.choice(ndb, 60, replace=False)
        db[rows] = q[c] * rng.uniform(0.5, 2.0, (60, 1)) + 1e-9 * rng.standard_normal((60, dim))
        db[rows[:5]] = db[rows[5]]                         # plus exact duplicates
    idx, sc = R.cosine_topk(q, db, k, return_scores=True)
    want_idx, want_sc = O.cosine_topk(q, db, k, return_scores=True)
    assert np.array_equal(idx, want_idx)
    assert np.array_equal(sc, want_sc)


def test_retrieval_duplicates_across_splits(torch_cuda):
    """A large database is ranked in several splits that share a pruning threshold.  Copies of one row spread over
    the whole index range, and blocks of 64 identical rows inside one split, must come back lowest index first."""
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(99)
    nq, ndb, dim = 300, 150_000, 26
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    db = rng.standard_normal((ndb, dim)).astype(np.float32)
    for c in range(20):                                    # queries 0-19: 48 copies of a near-query row, one every ~3100 rows
        db[rng.integers(0, 3000) + np.arange(48) * 3100] = q[c] * 1.5 + 0.01 * rng.standard_normal(dim).astype(np.float32)
    for c in range(20, 30):                                # queries 20-29: 64 copies in one contiguous block
        start = 5000 + (c - 20) * 14_000
        db[start:start + 64] = q[c] * 0.7 + 0.01 * rng.standard_normal(dim).astype(np.float32)
    for k in (1, 20, 24, 28, 33):
        idx, sc = R.cosine_topk(q, db, k, return_scores=True)
        want_idx, want_sc = O.cosine_topk(q, db, k, return_scores=True)
        assert np.array_equal(idx, want_idx), k
        assert np.array_equal(sc, want_sc), k


def test_retrieval_takeover_across_waves(torch_cuda):
    """More CTAs than SMs (40 query tiles x several splits): CTAs of later waves take over the lists of the splits of their
    query tile that have already finished (retrieval_tc.cuh) and report only their own rows.  The database is ordered so
    that every later split displaces what the earlier ones found (scores grow with the index), the best row of every query
    has exact copies at both ends of the index range (ties across splits: lowest index first), and a block of queries has
    its whole top-k inside the FIRST split (later CTAs then insert nothing and must still not report the rows they took over)."""
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(2024)
    nq, ndb, dim, k = 40 * 256, 200_000, 26, 20
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    base = rng.standard_normal((ndb, dim)).astype(np.float32)
    # rows lean more and more towards a common direction the queries share: cosines rise with the index
    common = rng.standard_normal(dim).astype(np.float32)
    q += 0.8 * common
    db = base + (np.linspace(0.0, 1.5, ndb, dtype=np.float32)[:, None] * common)
    sel = np.arange(0, nq, 160)                            # 64 queries checked against the oracle (all query tiles)
    for j, qi in enumerate(sel[:24]):                      # exact copies of a near-query row at both ends and in the middle
        row = (q[qi] * 2.0 + 0.01 * rng.standard_normal(dim)).astype(np.float32)
        db[[50 + j, 100_000 + j, ndb - 50 - j]] = row
    for j, qi in enumerate(sel[24:40]):                    # whole top-k in the first 2000 rows
        rows = 200 + j * 100 + np.arange(k + 4)
        db[rows] = (q[qi][None, :] * rng.uniform(1.0, 3.0, (k + 4, 1)) + 1e-3 * rng.standard_normal((k + 4, dim))).astype(np.float32)
    idx, sc = R.cosine_topk(q, db, k, return_scores=True)
    want_idx, want_sc = O.cosine_topk(q[sel], db, k, return_scores=True)
    assert np.array_equal(np.asarray(idx)[sel], want_idx)
    assert np.array_equal(np.asarray(sc)[sel], want_sc)
    assert (np.asarray(idx) >= 0).all() and all(len(set(r)) == k for r in np.asarray(idx)[::97])   # complete lists, no row twice


def test_retrieval_fuzz_filter_kernels(torch_cuda):
    """Randomised shapes and adversarial score distributions through the tensor-core filter path (dim <= 32,
    k <= 24 on the tcgen05 kernel, k = 28 on the float32 filter): indices and scores must equal the oracle's bit for bit every time."""
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    rng = np.random.default_rng(20260)
    kinds = ("normal", "clustered", "negative", "duplicates", "all_same", "zeros", "tiny_scale")
    for case in range(42):
        kind = kinds[case % len(kinds)]
        dim = int(rng.choice([1, 2, 5, 13, 26, 31, 32]))
        ndb = int(rng.choice([1, 7, 24, 127, 128, 129, 1000, 4097, 33_000]))
        nq = int(rng.choice([1, 3, 255, 256, 257, 600]))
        k = int(min(ndb, rng.choice([1, 2, 10, 20, 28])))
        q = rng.standard_normal((nq, dim))
        db = rng.standard_normal((ndb, dim))
        if kind == "clustered":                            # every cosine close to 1 (like raw MFCC statistics)
            base = rng.standard_normal(dim) * 5.0
            q = base + 0.01 * q
            db = base + 0.01 * db
        elif kind == "negative":                           # all similarities negative
            base = np.abs(rng.standard_normal(dim)) + 0.5
            q = base + 0.05 * q
            db = -base + 0.05 * db
        elif kind == "duplicates" and ndb > 4:
            src = rng.integers(0, ndb, size=ndb // 2)
            db[rng.integers(0, ndb, size=ndb // 2)] = db[src]
        elif kind == "all_same":
            db[:] = db[0]
        elif kind == "zeros":
            db[rng.integers(0, ndb, size=max(1, ndb // 3))] = 0.0
            q[0] = 0.0
        elif kind == "tiny_scale":
            q *= 1e-12
            db *= 1e12
        dt = np.float32 if case % 2 else np.float64
        q, db = q.astype(dt), db.astype(dt)
        idx, sc = R.cosine_topk(q, db, k, return_scores=True)
        want_idx, want_sc = O.cosine_topk(q, db, k, return_scores=True)
        assert np.array_equal(idx, want_idx), (case, kind, nq, ndb, dim, k)
        assert np.array_equal(sc, want_sc), (case, kind, nq, ndb, dim, k)


def test_retrieval_full_size_clustered(torch_cuda):
    """BASELINE scale (1 M database rows) on tightly clustered, class-structured embeddings: every cosine is close to 1
    and thousands of rows lie within the filter's epsilon of the k-th score, so the result rests entirely on the exact
    float64 re-score.  Indices and scores must still equal the oracle's."""
    torch = torch_cuda
    from dsp_final_b200 import retrieval as R
    from oracle import oracle as O

    g = torch.Generator(device="cuda")
    g.manual_seed(11)
    nq, ndb, dim, classes = 384, 1_000_000, 26, 50
    centers = torch.randn((classes, dim), generator=g, device="cuda")
    offset = 4.0 * torch.randn((1, dim), generator=g, device="cuda")
    for noise in (0.02, 0.002):
        q = offset + centers[torch.arange(nq, device="cuda") % classes] + noise * torch.randn((nq, dim), generator=g, device="cuda")
        db = offset + centers[torch.arange(ndb, device="cuda") % classes] + noise * torch.randn((ndb, dim), generator=g, device="cuda")
        idx, sc = R.cosine_topk(q, db, 20, return_scores=True)
        want_idx, want_sc = O.cosine_topk(q.cpu().numpy(), db.cpu().numpy(), 20, return_scores=True)
        assert np.array_equal(idx.cpu().numpy(), want_idx)
        assert np.array_equal(sc.cpu().numpy(), want_sc)


def test_retrieval_sweep_config3(torch_cuda):
    """BASELINE.json configs[2] in miniature: frame x hop sweep, fold-5 queries vs folds 1-4,
    identical index lists and identical Top-10 / Top-20 against the oracle on the same embeddings."""
    from dsp_final_b200 import retrieval as R
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    n, length = 500, 33_075                                # 0.75 s clips keep the oracle quick
    clips = synth.host_clips(n, seed=1234, length=length)
    folds = np.array([synth.fold_of(i, n) for i in range(n)])
    targets = synth.labels(n)
    for fl in (512, 1024, 2048):
        for hop in (256, 512, 1024):
            cfg = MfccConfig(sample_rate=44100, frame_length=fl, hop_length=hop)
            emb = features_batch(clips, cfg, ("embed",))["embed"]
            ref_emb = O.features_batch(clips[:16], O.OracleConfig(44100, fl, hop), want=("embed",))["embed"]
            assert rel_err(emb[:16], ref_emb) < TOL
            db, q = emb[folds <= 4], emb[folds == 5]
            idx = R.cosine_topk(q, db, 20)
            assert np.array_equal(idx, O.cosine_topk(q, db, 20)), (fl, hop)
            for k in (10, 20):
                ours = R.hits_at_k(idx, k, targets[folds <= 4], targets[folds == 5])
                assert ours == O.hits_at_k(idx, k, targets[folds <= 4], targets[folds == 5])


def test_pcm16_ingest_matches_load_audio_semantics(torch_cuda, golden_real):
    """Row f2: int16 in -> x/32768 -> x/max|x| on the GPU == NumPy float32, bit for bit; features follow."""
    torch = torch_cuda
    from dsp_final_b200.batch import features_batch, pcm16_to_float
    from dsp_final_b200.dsp.mfcc import MfccConfig

    g = golden_real
    rng = np.random.default_rng(3)
    pcm = np.stack([g["pcm16"][:40_000], (rng.standard_normal(40_000) * 3000).astype(np.int16),
                    np.zeros(40_000, np.int16)])
    pcm[1, 123] = -32768                                          # |min int16| is the peak
    x = pcm.astype(np.float32) / np.float32(32768.0)
    peak = np.max(np.abs(x), axis=1, keepdims=True)
    xn = np.where(peak > 0, x / np.where(peak > 0, peak, 1), x).astype(np.float32)
    dev = pcm16_to_float(torch.as_tensor(pcm).cuda(), normalize=True).cpu().numpy()
    assert np.array_equal(dev, xn)
    assert np.array_equal(pcm16_to_float(torch.as_tensor(pcm).cuda(), normalize=False).cpu().numpy(), x)
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    # Round 2: the PCM16 door converts inside the feature kernel's own sample loads (general variant: 4-byte /
    # 2-byte loads, table window).  The same variant fed with the converted float32 samples -- forced here by an odd
    # row stride -- must give bit-identical features (the fused quotient is the correctly rounded one); the aligned
    # float32 variant (computed window, shared rows) differs by float32 round-off only.
    wide = torch.zeros((3, 40_001), device="cuda")
    wide[:, :40_000] = torch.as_tensor(xn).cuda()
    same_variant = features_batch(wide[:, :40_000], cfg, ("mfcc", "log_mel", "embed"))
    aligned = features_batch(xn, cfg, ("mfcc", "log_mel", "embed"))
    for src in (pcm, torch.as_tensor(pcm).cuda()):
        got = features_batch(src, cfg, ("mfcc", "log_mel", "embed"))
        for k in aligned:
            a = got[k].cpu().numpy() if hasattr(got[k], "cpu") else got[k]
            assert np.array_equal(a, same_variant[k].cpu().numpy()), k
            assert rel_err(a, aligned[k]) < 1e-6, k
    raw = features_batch(torch.as_tensor(pcm).cuda(), cfg, ("mfcc",), normalize=False)["mfcc"].cpu().numpy()
    wide[:, :40_000] = torch.as_tensor(x).cuda()
    assert np.array_equal(raw, features_batch(wide[:, :40_000], cfg, ("mfcc",))["mfcc"].cpu().numpy())
    # the real-clip golden (reference features of the normalised excerpt) through the PCM16 door
    full = features_batch(g["pcm16"][None, :], cfg, ("mfcc",))["mfcc"][0]
    _close(full, g["mfcc"], "pcm16 real clip mfcc")


@pytest.mark.parametrize("kernel,fl", [("auto", 1024), ("generic", 1024), ("auto", 512)])
def test_log_mel_cnn_layout(torch_cuda, kernel, fl):
    """Row f3: [B,1,n_mels,T] written by the store epilogue == transpose of the reference layout."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import features_batch, log_mel_nchw
    from dsp_final_b200.dsp.mfcc import MfccConfig

    cfg = MfccConfig(sample_rate=44100, frame_length=fl, hop_length=fl // 2, n_mels=128)
    dev = torch.as_tensor(synth.host_clips(5, seed=4, length=50_001)).cuda()     # odd frame count
    ref = features_batch(dev, cfg, ("log_mel",), kernel=kernel)["log_mel"]
    out = log_mel_nchw(dev, cfg, kernel=kernel)
    assert out.shape == (5, 1, 128, ref.shape[1]) and out.is_contiguous()
    assert torch.equal(out[:, 0], ref.transpose(1, 2))


@pytest.mark.parametrize("dim", [128, 512, 768, 2048])
def test_retrieval_ml_dimensions(torch_cuda, dim):
    """Row f4: model-embedding dimensions of retrieval_ml.py through the same kernels, bit-exact indices."""
    from types import SimpleNamespace

    from dsp_final_b200 import retrieval_ml as RM
    from oracle import oracle as O

    rng = np.random.default_rng(dim)
    db = rng.standard_normal((1600, dim)).astype(np.float32)
    q = rng.standard_normal((400, dim)).astype(np.float32)
    tdb, tq = rng.integers(0, 50, 1600), rng.integers(0, 50, 400)
    idx = RM.cosine_topk(q, db, 20)
    assert np.array_equal(idx, O.cosine_topk(q, db, 20))
    items = lambda t: [SimpleNamespace(target=int(v)) for v in t]   # noqa: E731
    res = RM.evaluate_retrieval(items(tdb), items(tq), db, q, (10, 20))
    want = O.evaluate_retrieval(tdb, tq, db, q, (10, 20))
    assert [(r.k, r.precision) for r in res] == want


@pytest.mark.parametrize("fl,hop", [(1024, 512), (512, 256), (2048, 512), (1024, 300)])
def test_stft_full_size_properties(torch_cuda, fl, hop):
    """stft() at ESC-50 clip length on the fast kernel: oracle parity on sampled frames plus
    size-independent properties (linearity, Parseval per frame, DC / Nyquist bins are real)."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import stft_batch
    from dsp_final_b200.dsp.stft import _get_window
    from oracle import oracle as O

    x = torch.as_tensor(synth.host_clips(12, seed=21)).cuda()
    y = torch.as_tensor(synth.host_clips(12, seed=22)).cuda()
    sx, sy = stft_batch(x, fl, hop), stft_batch(y, fl, hop)
    t = 1 + (220_500 - fl) // hop
    assert sx.shape == (12, t, fl // 2 + 1) and sx.dtype == torch.complex64
    sel = [0, 1, t // 2, t - 1]
    ref = O.stft(x[3].cpu().numpy(), fl, hop)[sel]
    _close(sx[3][sel].cpu().numpy(), ref, f"stft {fl}/{hop}")
    # linearity: stft(2x - 0.5y) == 2 stft(x) - 0.5 stft(y)
    lin = stft_batch(2.0 * x - 0.5 * y, fl, hop)
    assert rel_err(lin.cpu().numpy(), (2.0 * sx - 0.5 * sy).cpu().numpy()) < 2e-6
    # Parseval per frame: sum |frame * w|^2 = (|X0|^2 + |X_{N/2}|^2 + 2 sum_{0<k<N/2} |X_k|^2) / N
    w = torch.as_tensor(_get_window("hann", fl).astype(np.float32)).cuda()
    frames = x[0].unfold(0, fl, hop)[:t] * w
    lhs = (frames.double() ** 2).sum(dim=1)
    p = (sx[0].real.double() ** 2 + sx[0].imag.double() ** 2)
    rhs = (p[:, 0] + p[:, -1] + 2.0 * p[:, 1:-1].sum(dim=1)) / fl
    assert torch.allclose(lhs, rhs, rtol=1e-5, atol=1e-9)
    assert float(sx[..., 0].imag.abs().max()) < 1e-4 * float(sx[..., 0].real.abs().max() + 1e-30) + 1e-6
    assert float(sx[..., -1].imag.abs().max()) < 1e-4 * float(sx[..., -1].real.abs().max() + 1e-30) + 1e-6
    # the generic kernel agrees with the fast one
    g = stft_batch(x[:2], fl, hop, kernel="generic")
    assert rel_err(g.cpu().numpy(), sx[:2].cpu().numpy()) < 1e-6


def test_config2_full_size_properties(torch_cuda):
    """BASELINE.json configs[1] at full size: 2000 clips x 5 s, MFCC + log-mel + embeddings in one pass.
    Oracle parity on a sample copied back from the device, plus size-independent properties."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import embed_stats, features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    clips = synth.device_clips(2000, seed=1234, device=torch.device("cuda"))
    out = features_batch(clips, cfg, ("log_mel", "mfcc", "embed"))
    mf, lm, em = out["mfcc"], out["log_mel"], out["embed"]
    assert mf.shape == (2000, 429, 13) and lm.shape == (2000, 429, 40) and em.shape == (2000, 26)
    assert bool(torch.isfinite(mf).all()) and bool(torch.isfinite(lm).all())
    sel = [0, 399, 1000, 1999]
    ref = O.features_batch(clips[sel].cpu().numpy(), O.OracleConfig(44100, 1024, 512))
    for j, i in enumerate(sel):
        _close(mf[i].cpu().numpy(), ref["mfcc"][j], f"clip {i} mfcc")
        _close(lm[i].cpu().numpy(), ref["log_mel"][j], f"clip {i} log-mel")
        _close(em[i].cpu().numpy(), ref["embed"][j], f"clip {i} embed")
    # permutation equivariance (clips are independent units): bit-identical rows
    perm = torch.randperm(2000, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    mfp = features_batch(clips[perm].contiguous(), cfg, ("mfcc",))["mfcc"]
    assert torch.equal(mfp, mf[perm])
    # two half batches == one batch (what clip sharding across GPUs relies on)
    a = features_batch(clips[:1000], cfg, ("mfcc",))["mfcc"]
    b = features_batch(clips[1000:], cfg, ("mfcc",))["mfcc"]
    assert torch.equal(torch.cat([a, b]), mf)
    # embeddings are exactly the statistics of the MFCCs that were written
    assert torch.equal(embed_stats(mf), em)
    # log-mel never drops below the floor
    assert float(lm.min()) >= float(np.log(1e-10)) - 1e-4
