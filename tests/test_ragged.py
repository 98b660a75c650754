"""Ragged batches: clips of different lengths in one call (dspx_ragged_layout, dspx_features_ragged,
dspx_embed_stats_ragged, features_ragged and the callers that use them).

CPU: the layout against NumPy, the CPU replay of the RAGGED warp8 mapping against the oracle (also under
AddressSanitizer), and the resource usage of the ragged kernel instantiations.  GPU (-m gpu): every clip of a ragged
batch bit-identical to features_batch on that clip alone, a large mixed batch, the per-clip fallback plans and the
callers (compute_embeddings, BatchFeatureCache).
"""
from __future__ import annotations

import ctypes as C
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest

from conftest import REPO, rel_err

SR = 44100
TOL = 1e-4
# (frame_length, hop, n_fft): SHARE (hop = n_fft / 2), plain aligned, R1 = 16, odd hop (U4), frames shorter than n_fft
CONFIGS = ((1024, 512, None), (512, 256, None), (2048, 512, None), (1024, 441, None), (400, 160, 512))


def _cfg(fl, hop, n_fft=None):
    from dsp_final_b200.dsp.mfcc import MfccConfig

    return MfccConfig(sample_rate=SR, frame_length=fl, hop_length=hop, n_fft=n_fft)


def _special_lengths(fl, hop):
    """one frame exactly, an odd frame count, frame_length + hop - 1 (still one frame), 0.1 s, and a 30 s clip."""
    return [fl, fl + 2 * hop, fl + hop - 1, 4410, 30 * SR, 4410 + 3, fl + 4 * hop + 7]


def _clips(lengths, seed):
    from dsp_final_b200 import synth

    return [synth.host_clip(i, seed=seed, length=int(n)) for i, n in enumerate(lengths)]


@pytest.fixture(scope="module")
def built():
    from dsp_final_b200 import build

    return build.build_native(), build.build_emu()


# ---- layout (host only) ------------------------------------------------------------------------------------
def test_layout_matches_numpy(built):
    from dsp_final_b200.batch import RAGGED_ALIGN, ragged_layout

    rng = np.random.default_rng(3)
    for fl, hop, n_fft in CONFIGS:
        lengths = np.concatenate((_special_lengths(fl, hop), rng.integers(fl, 5 * SR, 40)))
        starts, table, total = ragged_layout(lengths, _cfg(fl, hop, n_fft))
        frames = 1 + (lengths - fl) // hop
        assert total == frames.sum()
        assert np.array_equal(table[:, 0], starts) and np.array_equal(table[:, 1], lengths)
        assert np.array_equal(table[:, 2], frames)
        assert np.array_equal(table[:, 3], np.cumsum(frames) - frames)
        pairs = (frames + 1) // 2
        assert np.array_equal(table[:, 4], np.cumsum(pairs) - pairs)
        assert np.all(starts % RAGGED_ALIGN == 0) and np.all(starts[1:] >= starts[:-1] + lengths[:-1])


def test_layout_rejects_bad_clips(built):
    from dsp_final_b200.batch import ragged_layout

    cfg = _cfg(1024, 512)
    with pytest.raises(ValueError, match=r"clip 2: 1023 samples"):
        ragged_layout([5000, 1024, 1023, 9000], cfg)
    with pytest.raises(ValueError, match=r"clip 1: float32 clips must start at an even sample"):
        ragged_layout([2000, 2000], cfg, starts=[0, 2001])
    ragged_layout([2000, 2000], cfg, np.int16, starts=[0, 2001])          # int16 samples may start anywhere
    starts, table, total = ragged_layout([], cfg)
    assert total == 0 and table.shape == (0, 5) and starts.shape == (0,)


def test_ragged_clip_struct_matches_header(built):
    from dsp_final_b200 import _lib

    assert C.sizeof(_lib.DspxRaggedClip) == 40 and _lib.DspxRaggedClip.first_pair.offset == 32


# ---- CPU replay of the RAGGED mapping (csrc/emu.cu -> the same w8_set_item the kernel runs) ----------------
def _emu_ragged(built, cfg, xs):
    from dsp_final_b200 import _lib
    from dsp_final_b200.batch import ragged_layout
    from dsp_final_b200.plan import config_key, config_struct

    lib = C.CDLL(str(built[1]))
    starts, table, total = ragged_layout([len(x) for x in xs], cfg)
    flat = np.zeros(int(starts[-1] + len(xs[-1])), np.float32)
    for s, x in zip(starts, xs):
        flat[s:s + len(x)] = x
    lm = np.zeros((total, cfg.n_mels), np.float32)
    mf = np.zeros((total, cfg.n_mfcc), np.float32)
    c = config_struct(config_key(cfg), "warp8")
    assert isinstance(c, _lib.DspxConfig)
    rc = lib.emu_features_warp8_ragged(C.byref(c), C.c_void_p(flat.ctypes.data), C.c_void_p(table.ctypes.data),
                                       C.c_int64(len(xs)), C.c_void_p(lm.ctypes.data), C.c_void_p(mf.ctypes.data))
    assert rc == 0
    return table, lm, mf


def test_ragged_replay_matches_oracle(built):
    from oracle import oracle as O

    for fl, hop, n_fft in CONFIGS:
        cfg = _cfg(fl, hop, n_fft)
        xs = _clips(_special_lengths(fl, hop), seed=fl + hop)
        table, lm, mf = _emu_ragged(built, cfg, xs)
        ocfg = O.OracleConfig(SR, fl, hop, n_fft)
        for i, x in enumerate(xs):
            rows = slice(table[i, 3], table[i, 3] + table[i, 2])
            ref = O.features_batch(x[None], ocfg, want=("mfcc", "log_mel"))
            assert rel_err(mf[rows], ref["mfcc"][0]) < 1e-5, (fl, hop, i)
            assert rel_err(lm[rows], ref["log_mel"][0]) < 1e-5, (fl, hop, i)


def test_ragged_replay_is_addresssanitizer_clean(tmp_path):
    """The RAGGED mapping writes only the rows of its own clips: exact-size [total_frames, ...] outputs and an
    exact-size sample buffer under AddressSanitizer."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = tmp_path / "ragged_asan"
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-g", "-std=c++17", "-Xcompiler",
           "-fsanitize=address,-fno-omit-frame-pointer,-ffp-contract=off", "-o", str(exe),
           str(REPO / "tests" / "replay_ragged_asan_main.cu"), str(REPO / "dsp_final_b200" / "csrc" / "emu.cu"), "-lasan"]
    build = subprocess.run(cmd, capture_output=True, text=True)
    out = build.stderr + build.stdout
    if build.returncode != 0 and ("-lasan" in out or "libasan" in out):
        pytest.skip("libasan not available")
    assert build.returncode == 0, build.stderr[-2000:]
    run = subprocess.run([str(exe)], capture_output=True, text=True,
                         env={"ASAN_OPTIONS": "protect_shadow_gap=0:detect_leaks=0", "PATH": "/usr/bin:/bin"})
    assert run.returncode == 0 and "AddressSanitizer" not in run.stderr, run.stderr[-3000:]
    lines = [l for l in run.stdout.splitlines() if l.startswith("ragged ")]
    assert len(lines) == 5 and all(l.endswith("rc 0 finite 1") for l in lines), run.stdout


def test_ragged_headline_variants_keep_their_registers(built):
    """The RAGGED twins of the headline kernel (1024/512: SHARE, 20 warps, with and without pre-emphasis) keep the
    96-register allocation without a stack frame (spills), and every aligned / general / PCM16 variant has one."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    res = subprocess.run([cuobjdump, "-res-usage", str(built[0])], capture_output=True, text=True, check=True).stdout
    kernels = dict((name, (int(reg), int(stack))) for name, reg, stack in
                   re.findall(r"Function (_ZN4dspx17feat_warp8_kernel\S*):\s*\n?\s*REG:(\d+) STACK:(\d+)", res))
    # template arguments <R1, PRE, STFT, SHARE, NW, EMB, U4, PCM, RAGGED>; the RAGGED ones end in "Lb1EEEv..."
    ragged = [k for k in kernels if k.endswith("Lb1EEEvNS_8W8ParamsE")]
    assert len(ragged) >= 40 and len(kernels) - len(ragged) >= 90, (len(kernels), len(ragged))
    for pre in (0, 1):
        name = f"_ZN4dspx17feat_warp8_kernelILi8ELb{pre}ELb0ELb1ELi20ELb0ELb0ELb0ELb1EEEvNS_8W8ParamsE"
        assert kernels[name] == (96, 0), (name, kernels.get(name))
    for tail in ("ELb0ELb0ELb0ELb1E", "ELb1ELb0ELb0ELb1E", "ELb0ELb1ELb0ELb1E", "ELb0ELb1ELb1ELb1E"):   # plain, EMB, U4, PCM
        assert any(k.endswith(tail + "EEvNS_8W8ParamsE") for k in ragged), tail


# ---- GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def _mixed_lengths(fl, hop, n, seed):
    rng = np.random.default_rng(seed)
    special = [fl, fl + 2 * hop, fl + hop - 1, fl + 1, 30 * SR, 4410, 4411]
    return np.concatenate((special, rng.integers(fl, 3 * SR, n - len(special))))


def _alone(torch, x, cfg, want, **kw):
    """features_batch on one clip passed as a [1, L] row with an even stride (8-byte aligned frames when the hop is)."""
    from dsp_final_b200.batch import features_batch

    n = x.shape[0]
    buf = torch.zeros((1, n + (n & 1)), dtype=x.dtype, device=x.device)
    buf[0, :n] = x
    return features_batch(buf[:, :n], cfg, want, **kw)


def _rows(t, offsets, i):
    return t[int(offsets[i]):int(offsets[i + 1])]


@pytest.mark.gpu
def test_ragged_bit_identical_per_clip(torch_cuda):
    torch = torch_cuda
    from dsp_final_b200.batch import embed_stats, features_ragged
    from oracle import oracle as O

    for fl, hop, n_fft in CONFIGS:
        cfg = _cfg(fl, hop, n_fft)
        lengths = _mixed_lengths(fl, hop, 64, seed=fl * 7 + hop)
        host = _clips(lengths, seed=hop)
        xs = [torch.as_tensor(x).cuda() for x in host]
        both = features_ragged(xs, cfg, ("log_mel", "mfcc", "embed"))
        alone_emb = features_ragged(xs, cfg, ("embed",))["embed"]
        off = both["frame_offsets"].cpu().numpy()
        assert off[-1] == both["mfcc"].shape[0] == both["log_mel"].shape[0]
        stats = embed_stats([_rows(both["mfcc"], off, i) for i in range(len(xs))])
        assert torch.equal(stats, both["embed"])
        for i, x in enumerate(xs):
            ref = _alone(torch, x, cfg, ("log_mel", "mfcc", "embed"))
            assert torch.equal(_rows(both["log_mel"], off, i), ref["log_mel"][0]), (fl, hop, i)
            assert torch.equal(_rows(both["mfcc"], off, i), ref["mfcc"][0]), (fl, hop, i)
            assert torch.equal(both["embed"][i], ref["embed"][0]), (fl, hop, i)
            assert torch.equal(alone_emb[i], _alone(torch, x, cfg, ("embed",))["embed"][0]), (fl, hop, i)
            assert torch.equal(stats[i], embed_stats(ref["mfcc"])[0]), (fl, hop, i)
        # PCM16, with and without peak normalisation
        pcm = [torch.as_tensor((x * 20000).astype(np.int16)).cuda() for x in host[:24]]
        for norm in (True, False):
            r = features_ragged(pcm, cfg, ("log_mel", "mfcc", "embed"), normalize=norm)
            e = features_ragged(pcm, cfg, ("embed",), normalize=norm)["embed"]
            o = r["frame_offsets"].cpu().numpy()
            for i, x in enumerate(pcm):
                ref = _alone(torch, x, cfg, ("log_mel", "mfcc", "embed"), normalize=norm)
                assert torch.equal(_rows(r["log_mel"], o, i), ref["log_mel"][0]), (fl, hop, norm, i)
                assert torch.equal(_rows(r["mfcc"], o, i), ref["mfcc"][0]), (fl, hop, norm, i)
                assert torch.equal(r["embed"][i], ref["embed"][0]) and torch.equal(e[i], ref["embed"][0]), (fl, hop, norm, i)
        # oracle parity on a sample, through the NumPy path (pinned staging, one copy each way)
        sample = [host[j] for j in (0, 2, 4, 9)]
        got = features_ragged(sample, cfg, ("mfcc", "log_mel", "embed"))
        o = got["frame_offsets"]
        ocfg = O.OracleConfig(SR, fl, hop, n_fft)
        for i, x in enumerate(sample):
            ref = O.features_batch(x[None], ocfg)
            assert rel_err(_rows(got["mfcc"], o, i), ref["mfcc"][0]) < TOL, (fl, hop, i)
            assert rel_err(_rows(got["log_mel"], o, i), ref["log_mel"][0]) < TOL, (fl, hop, i)
            assert rel_err(got["embed"][i], ref["embed"][0]) < TOL, (fl, hop, i)


@pytest.mark.gpu
def test_ragged_large_mixed_batch(torch_cuda):
    """2000 clips of 0.5-10 s in one call: oracle parity on 32 clips, nothing written past total_frames, and a silent
    clip gives finite embeddings."""
    torch = torch_cuda
    from dsp_final_b200 import _lib
    from dsp_final_b200.batch import features_ragged, ragged_layout
    from dsp_final_b200.plan import get_plan
    from oracle import oracle as O

    cfg = _cfg(1024, 512)
    rng = np.random.default_rng(11)
    lengths = rng.integers(SR // 2, 10 * SR, 2000)
    gen = torch.Generator(device="cuda").manual_seed(5)
    xs = [torch.rand(int(n), generator=gen, device="cuda") - 0.5 for n in lengths]
    xs[7] = torch.zeros(int(lengths[7]), device="cuda")
    res = features_ragged(xs, cfg, ("mfcc", "log_mel"))
    emb = features_ragged(xs, cfg, ("embed",))["embed"]
    off = res["frame_offsets"].cpu().numpy()
    assert torch.isfinite(emb).all() and torch.isfinite(res["mfcc"]).all()
    ocfg = O.OracleConfig(SR, 1024, 512)
    for i in rng.choice(2000, 32, replace=False):
        ref = O.features_batch(xs[i].cpu().numpy()[None], ocfg)
        assert rel_err(_rows(res["mfcc"], off, i).cpu().numpy(), ref["mfcc"][0]) < TOL, i
        assert rel_err(_rows(res["log_mel"], off, i).cpu().numpy(), ref["log_mel"][0]) < TOL, i
        assert rel_err(emb[i].cpu().numpy(), ref["embed"][0]) < TOL, i
    # in-bounds: NaN-filled outputs with 64 spare rows, through the C ABI
    starts, table, total = ragged_layout(lengths, cfg)
    flat = torch.zeros(int(starts[-1] + lengths[-1]), device="cuda")
    for s, x in zip(starts, xs):
        flat[int(s):int(s) + x.numel()] = x
    plan = get_plan(cfg, 0)
    lib = _lib.load()
    tdev = torch.from_numpy(table).cuda()
    lm = torch.full((total + 64, 40), float("nan"), device="cuda")
    mf = torch.full((total + 64, 13), float("nan"), device="cuda")
    em = torch.full((2000 + 4, 26), float("nan"), device="cuda")
    for outs in ((lm, mf, em), (lm, None, em)):
        ws_bytes = int(lib.dspx_features_ragged_workspace(plan.handle, table.ctypes.data, 2000, _lib.DTYPE_F32, 1, 1,
                                                         int(outs[1] is not None), 1))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        _lib.check(lib.dspx_features_ragged(plan.handle, flat.data_ptr(), _lib.DTYPE_F32, 1, tdev.data_ptr(), table.ctypes.data,
                                           2000, total, *[o.data_ptr() if o is not None else None for o in outs],
                                           ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert torch.isnan(lm[total:]).all() and torch.isnan(mf[total:]).all() and torch.isnan(em[2000:]).all()
        assert torch.isfinite(lm[:total]).all() and torch.isfinite(em[:2000]).all()
    assert torch.equal(mf[:total], res["mfcc"]) and torch.equal(lm[:total], res["log_mel"]) and torch.equal(em[:2000], emb)


@pytest.mark.gpu
def test_ragged_fallback_plans(torch_cuda):
    """Plans without a ragged kernel (the generic kernel at n_fft 256, n_fft 4096) loop over the clips: the same
    values as features_batch on each clip alone, float32 and PCM16."""
    torch = torch_cuda
    from dsp_final_b200.batch import features_batch, features_ragged

    for fl, hop in ((256, 128), (4096, 1024)):
        cfg = _cfg(fl, hop)
        host = _clips(_mixed_lengths(fl, hop, 12, seed=fl), seed=3)
        for pcm in (False, True):
            xs = [torch.as_tensor((x * 20000).astype(np.int16) if pcm else x).cuda() for x in host]
            r = features_ragged(xs, cfg, ("log_mel", "mfcc", "embed"))
            e = features_ragged(xs, cfg, ("embed",))["embed"]
            o = r["frame_offsets"].cpu().numpy()
            for i, x in enumerate(xs):
                ref = features_batch(x[None], cfg, ("log_mel", "mfcc", "embed"))
                assert torch.equal(_rows(r["log_mel"], o, i), ref["log_mel"][0]), (fl, pcm, i)
                assert torch.equal(_rows(r["mfcc"], o, i), ref["mfcc"][0]), (fl, pcm, i)
                assert torch.equal(r["embed"][i], ref["embed"][0]) and torch.equal(e[i], ref["embed"][0]), (fl, pcm, i)


def _write_wav16(path, x):
    data = np.ascontiguousarray(x, dtype="<i2").tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 1, 1, SR, SR * 2, 2, 16)
    path.write_bytes(hdr + b"data" + struct.pack("<I", len(data)) + data)


@pytest.fixture()
def wav_items(tmp_path):
    from dsp_final_b200.datasets import Esc50Item

    rng = np.random.default_rng(21)
    lengths = [SR, 2 * SR, SR, 3 * SR + 17] + list(rng.integers(SR // 2, 4 * SR, 28))
    items = []
    for i, n in enumerate(lengths):
        x = (_clips([n], seed=100 + i)[0] * 25000).astype(np.int16)
        path = tmp_path / "audio" / f"clip{i}.wav"
        path.parent.mkdir(exist_ok=True)
        _write_wav16(path, x)
        items.append(Esc50Item(f"clip{i}.wav", 1 + i % 5, i % 7, f"class{i % 7}", path))
    return items


@pytest.mark.gpu
def test_compute_embeddings_mixed_lengths(torch_cuda, wav_items, tmp_path, monkeypatch):
    from dsp_final_b200 import batch as B
    from dsp_final_b200 import retrieval as R
    from dsp_final_b200.audio import load_pcm16
    from dsp_final_b200.cache import BatchFeatureCache

    cfg = _cfg(1024, 512)
    pcm = [load_pcm16(it.path, SR) for it in wav_items]
    groups: dict = {}
    for i, x in enumerate(pcm):
        groups.setdefault(len(x), []).append(i)
    want_emb = np.empty((len(pcm), 26), np.float32)
    want_cached = np.empty((len(pcm), 26), np.float32)
    for rows in groups.values():                          # the per-length grouping compute_embeddings used before
        x = np.stack([pcm[i] for i in rows])
        want_emb[rows] = B.features_batch(x, cfg, ("embed",))["embed"]
        want_cached[rows] = B.embed_stats(B.features_batch(x, cfg, ("mfcc",))["mfcc"])
    calls = []
    real = B.ragged_launch
    monkeypatch.setattr(B, "ragged_launch", lambda *a, **k: calls.append(1) or real(*a, **k))
    monkeypatch.setattr(R, "features_batch", None)       # the mixed-length batch must not go through features_batch
    got = R.compute_embeddings(wav_items, cfg)
    assert len(calls) == 1 and np.array_equal(got, want_emb)
    cache = BatchFeatureCache(tmp_path / "features")
    cached = R.compute_embeddings(wav_items, cfg, feature_cache=cache)
    assert len(calls) == 2 and np.array_equal(cached, want_cached)
    assert np.array_equal(R.compute_embeddings(wav_items, cfg, feature_cache=cache), want_cached)   # hits
    assert len(calls) == 2
    q, db = [i for i, it in enumerate(wav_items) if it.fold == 1], [i for i, it in enumerate(wav_items) if it.fold != 1]
    assert np.array_equal(R.cosine_topk(got[q], got[db], 5), R.cosine_topk(want_emb[q], want_emb[db], 5))
    qi, dbi = [wav_items[i] for i in q], [wav_items[i] for i in db]
    assert R.evaluate_retrieval(dbi, qi, cached[db], cached[q], [1, 5]) == R.evaluate_retrieval(dbi, qi, want_cached[db], want_cached[q], [1, 5])
    # float32 clips: the fused embeddings of the ragged call against the grouped float32 path
    from dsp_final_b200.audio import normalize_audio

    flt = {it.filename: normalize_audio(x.astype(np.float32) / 32768.0).astype(np.float32) for it, x in zip(wav_items, pcm)}
    got_f = R.compute_embeddings(wav_items, cfg, loader=lambda it: flt[it.filename])
    assert len(calls) == 3
    want_f = np.empty_like(got_f)
    for rows in groups.values():
        want_f[rows] = B.features_batch(np.stack([flt[wav_items[i].filename] for i in rows]), cfg, ("embed",))["embed"]
    assert np.max(np.abs(got_f - want_f)) <= 2e-6 * np.max(np.abs(want_f))


@pytest.mark.gpu
def test_precompute_mixed_length_loader(torch_cuda, wav_items, tmp_path):
    import json

    from dsp_final_b200.audio import load_pcm16
    from dsp_final_b200.cache import BatchFeatureCache

    cfg = _cfg(1024, 512)
    cache = BatchFeatureCache(tmp_path / "pre")
    manifests = cache.precompute(wav_items, cfg, loader=lambda it: load_pcm16(it.path, SR), batch=12)
    fresh = BatchFeatureCache(tmp_path / "fresh")
    for ft, path in manifests.items():
        body = json.loads(path.read_text())
        assert body["num_files"] == len(wav_items)
        for it, rec in zip(wav_items, body["files"]):
            arr = np.load(cache.feature_path(it, ft, cfg))
            ref = fresh.get_feature(it, ft, cfg)
            assert np.array_equal(arr, ref), (ft, it.filename)
            assert rec["shape"] == list(ref.shape) == [1 + (len(load_pcm16(it.path, SR)) - 1024) // 512, 40 if ft == "log_mel" else 13]
