"""Resampling on the GPU (dspx_resample) against the host path it replaces.

2000 seeded ESC-50-shaped clips: 5 s of int16 at 44.1 kHz (441 MB as int16, 882 MB once read as float32: larger
than the 126 MB L2).  Arms, timed with CUDA events:
  kernel_<rate>   dspx_resample alone, PCM16 -> float32 at 8 / 16 / 22.05 / 32 / 48 kHz, with normalisation (the
                  feature path's call).  Input audio-s/s, plus the bytes moved and the useful FP32 operations (one
                  multiply and one add per filter tap that meets the clip) computed from the shapes.
  features_16k    features_batch(("embed",)) at a 16 kHz config on the resampled clips alone
  embed_16k       compute_embeddings-style PCM16 -> 16 kHz MFCC embeddings: resample + embeddings
  host_16k        load_audio's scipy.signal.resample_poly + normalize_audio on all host cores (a 200-clip subset)
A last line checks sampled clips of every kernel arm against scipy bit for bit.  Every line carries the GPU name and
its power limit, read in the same run.

    python benchmarks/resample_bench.py [--iters 5] [--out profiles/r03_resample_bench.jsonl]
"""
import sys; sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))  # noqa: E401,E702
import argparse
import json
import math
import os
import subprocess
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import torch

from dsp_final_b200.batch import _resample_2d, features_batch
from dsp_final_b200.dsp.mfcc import MfccConfig
from dsp_final_b200.plan import get_resampler

SR, N_CLIPS, SECONDS = 44100, 2000, 5
TARGETS = (8000, 16000, 22050, 32000, 48000)


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, iters: int) -> float:
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def useful_flops(n_in: int, up: int, down: int) -> int:
    """2 x the filter taps that meet the clip, summed over one clip's outputs (scipy's default design)."""
    g = math.gcd(up, down)
    up, down = up // g, down // g
    half = 10 * max(up, down)
    pre = down - half % down
    taps = -(-(2 * half + 1 + pre) // up)
    remove = (half + pre) // down
    n_out = -(-n_in * up // down)
    c = (np.arange(remove, remove + n_out, dtype=np.int64) * down) // up
    lo, hi = np.maximum(c - taps + 1, 0), np.minimum(c, n_in - 1)
    return int(2 * np.clip(hi - lo + 1, 0, None).sum())


def _host_resample(args):
    from scipy.signal import resample_poly

    from dsp_final_b200.audio import normalize_audio

    x, up, down = args
    return normalize_audio(resample_poly(x.astype(np.float32) / np.float32(32768.0), up, down))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "resample_bench needs a CUDA device"
    torch.cuda.set_device(0)
    info = gpu_info()
    rng = np.random.default_rng(2024)
    n_in = SECONDS * SR
    host = (rng.standard_normal((N_CLIPS, n_in)) * 6000).clip(-32768, 32767).astype(np.int16)
    x = torch.as_tensor(host).cuda()
    audio_s = N_CLIPS * SECONDS
    lines = []

    def emit(d):
        d.update(info)
        print(json.dumps(d), flush=True)
        lines.append(d)

    outs = {}
    for target in TARGETS:
        rs = get_resampler(target, SR, 0)
        t = timed(lambda: _resample_2d(x, rs, True), args.iters)
        y = _resample_2d(x, rs, True)
        outs[target] = y
        n_out = y.shape[1]
        flops = N_CLIPS * useful_flops(n_in, target, SR)
        nbytes = N_CLIPS * (2 * n_in + 4 * n_out * 2)                 # int16 in; float32 out written, then read and rewritten
        emit({"arm": f"kernel_{target}", "ms": t * 1e3, "audio_s_per_s": audio_s / t, "gflops_useful": flops / t / 1e9,
              "gbytes_per_s": nbytes / t / 1e9, "taps": useful_flops(n_in, target, SR) // 2 // n_out + 1})

    cfg16 = MfccConfig(sample_rate=16000, frame_length=512, hop_length=256)
    y16 = outs[16000]
    t = timed(lambda: features_batch(y16, cfg16, ("embed",)), args.iters)
    emit({"arm": "features_16k", "ms": t * 1e3, "audio_s_per_s": audio_s / t})
    t = timed(lambda: features_batch(x, cfg16, ("embed",), sample_rate=SR), args.iters)
    emit({"arm": "embed_16k", "ms": t * 1e3, "audio_s_per_s": audio_s / t})

    sub = 200
    workers = os.cpu_count() or 1
    with ProcessPoolExecutor(workers) as pool:
        list(pool.map(_host_resample, [(host[i], 16000, SR) for i in range(workers)]))       # warm the workers
        t0 = time.perf_counter()
        ref = list(pool.map(_host_resample, [(host[i], 16000, SR) for i in range(sub)], chunksize=4))
        t = time.perf_counter() - t0
    emit({"arm": "host_16k", "clips": sub, "cores": workers, "ms_per_2000": t / sub * N_CLIPS * 1e3,
          "audio_s_per_s": sub * SECONDS / t})

    bad, checked = 0, 0
    for target in TARGETS:
        y = outs[target]
        for i in rng.choice(N_CLIPS, 8, replace=False):
            want = ref[i] if (target == 16000 and i < sub) else _host_resample((host[i], target, SR))
            got = y[i].cpu().numpy()
            bad += int(not np.array_equal(got.view(np.uint32), want.astype(np.float32).view(np.uint32)))
            checked += 1
    emit({"arm": "bit_identity_vs_scipy", "clips_checked": checked, "mismatches": bad})
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")
    assert bad == 0, "resampled clips differ from scipy"


if __name__ == "__main__":
    main()
