"""BASELINE.json configs[2], [3] and [4] at full clip length, and the multi-threaded / multi-GPU paths.

  configs[2]  run_retrieval sweep: frame 512/1024/2048 x hop 256/512/1024, MFCC embeddings, fold-5 queries
              against the folds 1-4 database, Top-10 / Top-20 (reference configs/experiments.yaml:2-3)
  configs[3]  128-mel log-mel in the CNN input layout (scripts/models/train_cnn.py:23,46-47)
  configs[4]  clip-sharded retrieval with the NCCL all-gather of the database embeddings (needs >= 2 GPUs)

Every case feeds 5 s clips (220 500 samples, 429 frames at 1024/512); the oracle runs on a sample per setting.
"""
from __future__ import annotations

import os
import socket
import sys
import threading
from pathlib import Path

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu
REPO = Path(__file__).resolve().parents[1]
TOL = 1e-4          # BASELINE.json north_star: relative tolerance of FP32 features against the NumPy reference


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def clips_5s(torch_cuda):
    from dsp_final_b200 import synth

    return synth.device_clips(250, seed=1234, device=torch_cuda.device("cuda"))


def test_config2_sweep_full_length(torch_cuda, clips_5s):
    """All nine sweep settings on 250 five-second clips: MFCC + embeddings against the oracle on a sample,
    index lists and Top-10 / Top-20 identical to the oracle's ranking of the same embeddings."""
    torch = torch_cuda
    from dsp_final_b200 import retrieval as R
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    n = clips_5s.shape[0]
    folds = np.array([synth.fold_of(i, n) for i in range(n)])
    targets = synth.labels(n)
    sel = [0, 77, 201, 249]
    host_sel = clips_5s[sel].cpu().numpy()
    frames = {(512, 256): 860, (512, 512): 430, (512, 1024): 215, (1024, 256): 858, (1024, 512): 429,
              (1024, 1024): 215, (2048, 256): 854, (2048, 512): 427, (2048, 1024): 214}     # SURVEY.md section 8
    for (fl, hop), t in frames.items():
        cfg = MfccConfig(sample_rate=44100, frame_length=fl, hop_length=hop)
        out = features_batch(clips_5s, cfg, ("mfcc", "embed"))
        assert out["mfcc"].shape == (n, t, 13), (fl, hop)
        ref = O.features_batch(host_sel, O.OracleConfig(44100, fl, hop), want=("mfcc", "embed"))
        mf = out["mfcc"][sel].cpu().numpy()
        for j in range(len(sel)):
            assert rel_err(mf[j], ref["mfcc"][j]) < TOL, (fl, hop, sel[j])
            assert np.allclose(mf[j], ref["mfcc"][j], rtol=TOL, atol=TOL * np.max(np.abs(ref["mfcc"][j]))), (fl, hop)
        emb = out["embed"].cpu().numpy()
        assert rel_err(emb[sel], ref["embed"]) < TOL, (fl, hop)
        db, q = emb[folds <= 4], emb[folds == 5]
        idx = R.cosine_topk(q, db, 20)
        assert np.array_equal(idx, O.cosine_topk(q, db, 20)), (fl, hop)
        items_db = [type("I", (), {"target": int(x)}) for x in targets[folds <= 4]]
        items_q = [type("I", (), {"target": int(x)}) for x in targets[folds == 5]]
        got = R.evaluate_retrieval(items_db, items_q, db, q, (10, 20))
        want = O.evaluate_retrieval(targets[folds <= 4], targets[folds == 5], db, q, (10, 20))
        assert [(r.k, r.precision) for r in got] == [(int(k), float(p)) for k, p in want], (fl, hop)


def test_config2_extended_grid_4096(torch_cuda, clips_5s):
    """The reference's published extended grid has 4096-point frames (logs/precompute_mfcc_fl4096_hl256.log)."""
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    sel = [3, 120]
    host_sel = clips_5s[sel].cpu().numpy()
    for fl, hop in ((4096, 256), (4096, 1024)):
        cfg = MfccConfig(sample_rate=44100, frame_length=fl, hop_length=hop)
        out = features_batch(clips_5s[sel].contiguous(), cfg, ("mfcc", "log_mel"))
        ref = O.features_batch(host_sel, O.OracleConfig(44100, fl, hop), want=("mfcc", "log_mel"))
        assert out["mfcc"].shape[1] == 1 + (220_500 - fl) // hop
        assert rel_err(out["mfcc"].cpu().numpy(), ref["mfcc"]) < TOL
        assert rel_err(out["log_mel"].cpu().numpy(), ref["log_mel"]) < TOL


def test_config3_logmel128_full_length(torch_cuda, clips_5s):
    """128-mel log-mel of 5 s clips, time-major and in the CNN layout [B, 1, 128, 429]."""
    torch = torch_cuda
    from dsp_final_b200.batch import features_batch, log_mel_nchw
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512, n_mels=128)
    x = clips_5s[:128].contiguous()
    lm = features_batch(x, cfg, ("log_mel",))["log_mel"]
    assert lm.shape == (128, 429, 128) and bool(torch.isfinite(lm).all())
    sel = [0, 64, 127]
    ref = O.features_batch(x[sel].cpu().numpy(), O.OracleConfig(44100, 1024, 512, n_mels=128), want=("log_mel",))["log_mel"]
    got = lm[sel].cpu().numpy()
    for j in range(len(sel)):
        assert rel_err(got[j], ref[j]) < TOL
        # Elementwise: FP32 round-off of a 1024-point transform is relative to the frame's strongest bins, so a
        # one-bin filter (128 mels has them below 300 Hz) sitting 60-70 dB under the frame's peak carries a relative
        # energy error near 1e-3.  Cells within 60 dB of their frame's peak must meet the tolerance; the weakest
        # cells are bounded by the round-off model (error x relative amplitude).
        strong = ref[j] >= ref[j].max(axis=1, keepdims=True) - np.log(1e6)
        err = np.abs(got[j] - ref[j])
        assert np.all(err[strong] <= TOL * np.max(np.abs(ref[j]))), float(err[strong].max())
        level = np.exp(0.5 * (ref[j] - ref[j].max(axis=1, keepdims=True)))        # cell amplitude relative to the frame's peak band
        assert float((err * level).max()) < 3e-5, float((err * level).max())     # ~ 2^-24 * sqrt(n_fft) * a small factor
        assert float(err.max()) < 0.1
    # the nine all-zero filters of this table (SURVEY.md a11) sit at the floor, ln 1e-10, in every frame
    floor = np.float32(np.log(1e-10))
    zero_filters = np.where(np.all(ref[0] == ref[0][0, :][None, :], axis=0) & (np.abs(ref[0][0] - floor) < 1e-5))[0]
    assert len(zero_filters) == 9
    assert np.allclose(got[:, :, zero_filters], floor, atol=1e-5)
    nchw = log_mel_nchw(x, cfg)
    assert nchw.shape == (128, 1, 128, 429)
    assert torch.equal(nchw[:, 0], lm.transpose(1, 2))


def test_host_calls_from_two_threads_share_a_plan(torch_cuda):
    """Two threads call the host-buffer entry point on ONE plan with different batch sizes (the staging
    buffers grow under the plan's lock); each must get exactly what a lone call returns."""
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import mfcc_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig

    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    small = synth.host_clips(24, seed=5, length=60_000)
    big = synth.host_clips(400, seed=6, length=60_000)              # > one 48 MiB chunk: several slots in flight
    want_small, want_big = mfcc_batch(small, cfg), mfcc_batch(big, cfg)
    errors: list = []

    def work(x, want, reps):
        try:
            for _ in range(reps):
                got = mfcc_batch(x, cfg)
                if not np.array_equal(got, want):
                    errors.append("result differs")
        except Exception as e:                                        # pragma: no cover
            errors.append(repr(e))

    threads = [threading.Thread(target=work, args=(small, want_small, 12)),
               threading.Thread(target=work, args=(big, want_big, 3)),
               threading.Thread(target=work, args=(small[:5], want_small[:5], 12))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


# ---- configs[4]: the one collective ---------------------------------------------------------------------
def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank: int, world: int, port: int, q):
    sys.path.insert(0, str(REPO))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    try:
        import torch
        import torch.distributed as dist

        from dsp_final_b200 import dist as D
        from dsp_final_b200 import synth
        from dsp_final_b200.batch import features_batch
        from dsp_final_b200.dsp.mfcc import MfccConfig
        from oracle import oracle as O

        r, w, local = D.init_process_group("nccl")
        dev = torch.device("cuda", local)
        n, length = 600, 44_100
        cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
        c0, c1 = D.shard_range(n, rank, world)                       # clips shard by contiguous ranges
        clips = torch.as_tensor(synth.host_clips(c1 - c0, seed=21, length=length, first=c0)).to(dev)
        emb = features_batch(clips, cfg, ("embed",))["embed"]
        tgt = torch.as_tensor(synth.labels(c1 - c0, first=c0)).to(dev)
        split = (c1 - c0) * 4 // 5                                   # 80 / 20 database / query split per shard
        res, idx = D.sharded_retrieval(emb[:split], tgt[:split], emb[split:], tgt[split:], (10, 20))
        # rank 0 redoes the whole job alone through the oracle: same embeddings (gathered), CPU ranking
        all_db = D.all_gather_rows(emb[:split].contiguous())
        all_tdb = D.all_gather_rows(tgt[:split].reshape(-1, 1).contiguous()).reshape(-1)
        all_q = D.all_gather_rows(emb[split:].contiguous())
        all_tq = D.all_gather_rows(tgt[split:].reshape(-1, 1).contiguous()).reshape(-1)
        all_idx = D.all_gather_rows(idx.contiguous())
        if rank == 0:
            want_idx = O.cosine_topk(all_q.cpu().numpy(), all_db.cpu().numpy(), 20)
            assert np.array_equal(all_idx.cpu().numpy(), want_idx), "sharded top-20 differs from the oracle"
            want = [(k, O.hits_at_k(want_idx, k, all_tdb.cpu().numpy(), all_tq.cpu().numpy()), int(all_q.shape[0])) for k in (10, 20)]
            assert res == want, (res, want)
            ref = O.features_batch(synth.host_clips(2, seed=21, length=length), O.OracleConfig(44100, 1024, 512), want=("embed",))
            assert O.relative_error(emb[:2].cpu().numpy(), ref["embed"]) < 1e-4
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok"))
    except Exception as e:                                            # pragma: no cover
        import traceback

        q.put((rank, f"{type(e).__name__}: {e}\n{traceback.format_exc()}"))


def test_sharded_retrieval_nccl(torch_cuda):
    """Two ranks, two GPUs, NCCL: per-rank clip shards -> embeddings -> all-gather of the database ->
    local top-20 -> all-reduce of the hit counts; identical to the oracle on the gathered embeddings."""
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (bench.py --gpus N covers the collective under the driver's scaling run)")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(out) == [(0, "ok"), (1, "ok")], out


def test_cmvn_option_matches_oracle(torch_cuda):
    """north_star's "log/CMVN epilogue": off by default (the reference has none), bit-for-bit float64 statistics."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import cmvn, features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    clips = torch.as_tensor(synth.host_clips(6, seed=3, length=66_150)).cuda()
    out = features_batch(clips, cfg, ("mfcc", "log_mel"))
    for name in ("mfcc", "log_mel"):
        plain = out[name].cpu().numpy()
        normed = cmvn(out[name].clone()).cpu().numpy()
        for b in range(plain.shape[0]):
            want = O.cmvn(plain[b])
            assert np.max(np.abs(normed[b] - want)) <= 1e-6 * max(1.0, np.max(np.abs(want))), (name, b)
            assert np.allclose(normed[b].mean(axis=0), 0.0, atol=1e-5) and np.allclose(normed[b].std(axis=0), 1.0, atol=1e-4)
    host = cmvn(out["mfcc"].cpu().numpy())                           # NumPy in -> new NumPy array out
    assert np.array_equal(host, cmvn(out["mfcc"].clone()).cpu().numpy())
    const = torch.ones((2, 10, 3), device="cuda")
    assert torch.equal(cmvn(const.clone()), torch.zeros_like(const))   # zero variance: (x - mean) / (0 + eps) = 0


def test_logmel_batches_feed_the_epoch_loop(torch_cuda):
    """Row f3: LogMelBatches yields what DataLoader(Esc50FeatureDataset(..., postprocess=to_tensor)) yields
    (train_cnn.py:46-55; per item torch.tensor(log_mel.T, float32).unsqueeze(0), transforms.py:16-18)."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from dsp_final_b200.stream import LogMelBatches
    from oracle import oracle as O

    n, length = 37, 44_100
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512, n_mels=128)
    host = synth.host_clips(n, seed=12, length=length)
    targets = synth.labels(n)
    ref = O.features_batch(host, O.OracleConfig(44100, 1024, 512, n_mels=128), want=("log_mel",))["log_mel"]
    want = torch.tensor(np.transpose(ref, (0, 2, 1)), dtype=torch.float32).unsqueeze(1)       # [N, 1, n_mels, T]

    def collect(loader):
        xs, ys = [], []
        for feats, y in loader:
            assert feats.is_cuda and feats.dtype == torch.float32 and y.dtype == torch.int64 and feats.shape[1:] == (1, 128, 85)
            xs.append(feats.cpu())
            ys.append(y.cpu())
        return torch.cat(xs), torch.cat(ys)

    for clips in (torch.as_tensor(host).cuda(), host):                 # resident in HBM / streamed from the host
        loader = LogMelBatches(clips, targets, cfg, batch_size=8)
        assert len(loader) == 5 and len(loader.dataset) == n
        x, y = collect(loader)
        assert x.shape == (n, 1, 128, 85) and torch.equal(y, torch.as_tensor(targets, dtype=torch.int64))
        assert rel_err(x.numpy(), want.numpy()) < TOL
        assert len(LogMelBatches(clips, targets, cfg, batch_size=8, drop_last=True)) == 4
        sh = LogMelBatches(clips, targets, cfg, batch_size=8, shuffle=True, seed=4)
        x1, y1 = collect(sh)
        x2, y2 = collect(sh)                                           # next epoch: another permutation of the same set
        assert not torch.equal(y1, y2) or n < 3
        for xa, ya in ((x1, y1), (x2, y2)):
            assert sorted(ya.tolist()) == sorted(targets.tolist())
            # every shuffled row is one of the unshuffled rows, with its own target
            key = {xr.numpy().tobytes(): int(t) for xr, t in zip(x, y)}
            assert all(key[xr.numpy().tobytes()] == int(t) for xr, t in zip(xa, ya))
    # PCM16 clips: converted and peak-normalised on the GPU
    pcm = np.round(host * 32767.0).astype(np.int16)
    xp, _ = collect(LogMelBatches(pcm, targets, cfg, batch_size=16))
    f = pcm.astype(np.float32) / np.float32(32768.0)
    f = f / np.max(np.abs(f), axis=1, keepdims=True)
    refp = O.features_batch(f, O.OracleConfig(44100, 1024, 512, n_mels=128), want=("log_mel",))["log_mel"]
    assert rel_err(xp[:, 0].numpy(), np.transpose(refp, (0, 2, 1))) < TOL
    # and it drives the reference's epoch loop shape (classification.py:18-33): a tiny model, one optimizer step per batch
    model = torch.nn.Sequential(torch.nn.Conv2d(1, 4, 3, padding=1), torch.nn.AdaptiveAvgPool2d(1), torch.nn.Flatten(),
                                torch.nn.Linear(4, 50)).cuda()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    loader = LogMelBatches(torch.as_tensor(host).cuda(), targets, cfg, batch_size=8, shuffle=True)
    seen = 0
    for feats, y in loader:
        feats, y = feats.to("cuda"), y.to("cuda")
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(model(feats), y)
        loss.backward()
        opt.step()
        seen += y.size(0)
    assert seen == len(loader.dataset) and bool(torch.isfinite(loss))


def test_fused_embeddings_without_mfcc(torch_cuda, clips_5s):
    """Embeddings alone come from per-clip fixed-point accumulators inside the feature kernel (dspx_embeddings):
    same values as the statistics of the written MFCCs, reproducible bit for bit, oracle parity."""
    torch = torch_cuda
    from dsp_final_b200 import _lib
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from oracle import oracle as O

    for fl, hop, n_fft in ((1024, 512, None), (512, 256, None), (2048, 1024, None), (1024, 300, None), (400, 160, 512)):
        cfg = MfccConfig(sample_rate=44100, frame_length=fl, hop_length=hop, n_fft=n_fft)
        x = clips_5s[:96]
        both = features_batch(x, cfg, ("mfcc", "embed"))                 # embed = statistics of the MFCC tensor
        alone = features_batch(x, cfg, ("embed",))["embed"]              # fused: no MFCC tensor
        again = features_batch(x, cfg, ("embed", "log_mel"))
        assert torch.equal(alone, again["embed"]), (fl, hop)             # order-independent accumulation
        scale = float(both["embed"].abs().max())
        assert float((alone - both["embed"]).abs().max()) <= 2e-6 * scale, (fl, hop)
        assert torch.equal(again["log_mel"], features_batch(x, cfg, ("log_mel",))["log_mel"])
        ref = O.features_batch(x[:3].cpu().numpy(), O.OracleConfig(44100, fl, hop, n_fft), want=("embed",))["embed"]
        assert rel_err(alone[:3].cpu().numpy(), ref) < TOL, (fl, hop)
        host = features_batch(x[:40].cpu().numpy(), cfg, ("embed",))["embed"]      # host pipeline takes the same path
        assert np.array_equal(host, alone[:40].cpu().numpy()), (fl, hop)
    # a silent clip: zero variance must come out as zero, not as the square root of round-off
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    z = torch.zeros((2, 44_100), device="cuda")
    e = features_batch(z, cfg, ("embed",))["embed"]
    assert float(e[:, 13:].abs().max()) < 2e-3 and bool(torch.isfinite(e).all())
    # the generic kernel has no fused path: the call still works (through an MFCC tensor)
    g = features_batch(clips_5s[:4], cfg, ("embed",), kernel="generic")["embed"]
    assert rel_err(g.cpu().numpy(), features_batch(clips_5s[:4], cfg, ("embed",))["embed"].cpu().numpy()) < 1e-5
    ws = _lib.load().dspx_embeddings_workspace(None, 10)
    assert ws == 0


def test_unaligned_frames_stay_on_the_fast_kernel(torch_cuda):
    """Odd hop (441 samples = 10 ms) or an odd row stride: the warp8 kernel's 4-byte-load variant, oracle parity;
    same results as the aligned variant when both apply."""
    torch = torch_cuda
    from dsp_final_b200 import synth
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from dsp_final_b200.plan import get_plan
    from oracle import oracle as O

    host = synth.host_clips(6, seed=23, length=66_151)                        # odd length -> odd stride
    dev = torch.as_tensor(host).cuda()
    for fl, hop in ((1024, 441), (512, 147), (2048, 441), (1024, 512)):
        cfg = MfccConfig(sample_rate=44100, frame_length=fl, hop_length=hop)
        assert get_plan(cfg).kernel == "warp8"
        out = features_batch(dev, cfg, ("mfcc", "log_mel", "embed"))
        ref = O.features_batch(host, O.OracleConfig(44100, fl, hop))
        for name in ("mfcc", "log_mel", "embed"):
            assert rel_err(out[name].cpu().numpy(), ref[name]) < TOL, (fl, hop, name)
    # even hop, even stride: aligned and unaligned variants compute the same frames (offset the base by one sample)
    cfg = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    wide = torch.zeros((4, 66_152), device="cuda")
    wide[:, 1:] = dev[:4, :66_151]
    a = features_batch(dev[:4, :66_150].contiguous(), cfg, ("mfcc",))["mfcc"]
    b = features_batch(wide[:, 1:66_151], cfg, ("mfcc",))["mfcc"]             # base pointer 4 bytes off the grid
    assert rel_err(b.cpu().numpy(), a.cpu().numpy()) < 1e-6
