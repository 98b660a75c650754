"""Ragged batches against the two ways mixed lengths can be batched without them.

2000 seeded clips with lengths uniform in 1-9 s (44.1 kHz, 1.76 GB of float32: larger than the 126 MB L2), 1024/512,
MFCC + log-mel, all on the device.  Arms, timed with CUDA events in the same process, in rotating order:
  a_ragged        one dspx_features_ragged call for the whole batch
  b_per_length    features_batch once per distinct length (what compute_embeddings and the cache did): here one
                  launch per clip, since uniform lengths almost never repeat
  c_equal         features_batch on 2000 x 5 s clips of one length (the ESC-50 shape), the same audio seconds
  a_ragged_pcm16  arm a on int16 samples (conversion and peak normalisation inside the kernel's loads)
Each arm prints one JSON line: audio seconds per second, ms per call, the GPU name and its power limit read in the
same run.  The last line reports whether every clip's rows of arm a equal arm b's bit for bit.

    python benchmarks/ragged_bench.py [--reps 5] [--out results.jsonl]
"""
import sys; sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))  # noqa: E401,E702
import argparse
import json
import subprocess

import numpy as np
import torch

from dsp_final_b200.batch import features_batch, ragged_launch, ragged_layout
from dsp_final_b200.dsp.mfcc import MfccConfig
from dsp_final_b200.plan import get_plan

SR, N_CLIPS = 44100, 2000
WANT = ("log_mel", "mfcc")


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, iters: int) -> float:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "ragged_bench needs a CUDA device"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    cfg = MfccConfig(sample_rate=SR, frame_length=1024, hop_length=512)
    plan = get_plan(cfg, 0)
    rng = np.random.default_rng(2024)
    lengths = rng.integers(1 * SR, 9 * SR + 1, N_CLIPS)
    starts, table, total = ragged_layout(lengths, cfg)
    n_samples = int(starts[-1] + lengths[-1])
    gen = torch.Generator(device=dev).manual_seed(7)
    flat = torch.rand(n_samples, generator=gen, device=dev) - 0.5
    flat_pcm = (flat * 60000.0).clamp(-32768, 32767).to(torch.int16)
    table_dev = torch.from_numpy(table).to(dev)
    audio_s = float(lengths.sum()) / SR
    # arm b inputs: one [n, L] tensor per distinct length, rows with an even stride (the aligned variant, like arm a)
    groups: dict = {}
    for i, n in enumerate(lengths):
        groups.setdefault(int(n), []).append(i)
    batches = []
    for n, rows in groups.items():
        if len(rows) == 1:
            batches.append((rows, flat.as_strided((1, n), (n + (n & 1), 1), int(starts[rows[0]]))))
        else:
            batches.append((rows, torch.stack([flat[int(starts[i]):int(starts[i]) + n] for i in rows])))
    equal = torch.rand((N_CLIPS, 5 * SR), generator=gen, device=dev) - 0.5

    out_a = torch.empty(total * (plan.n_mels + plan.n_mfcc), device=dev)
    out_p = torch.empty_like(out_a)
    arms = {
        "a_ragged": (lambda: ragged_launch(plan, flat, False, table, table_dev, total, WANT, out=out_a), 20, audio_s),
        "b_per_length": (lambda: [features_batch(x, cfg, WANT) for _, x in batches], 2, audio_s),
        "c_equal": (lambda: features_batch(equal, cfg, WANT), 20, N_CLIPS * 5.0),
        "a_ragged_pcm16": (lambda: ragged_launch(plan, flat_pcm, True, table, table_dev, total, WANT, out=out_p), 20, audio_s),
    }
    for fn, _, _ in arms.values():                 # warm every shape the timed windows use
        fn()
    torch.cuda.synchronize()
    names = list(arms)
    times: dict = {k: [] for k in names}
    for rep in range(args.reps):
        for k in names[rep % len(names):] + names[:rep % len(names)]:
            fn, iters, _ = arms[k]
            times[k].append(timed(fn, iters))
    # bit check: every clip's rows of one ragged call against the per-length grouping
    res_a, _ = ragged_launch(plan, flat, False, table, table_dev, total, WANT)
    identical = 0
    for rows, x in batches:
        ref = features_batch(x, cfg, WANT)
        for j, i in enumerate(rows):
            r = slice(int(table[i, 3]), int(table[i, 3] + table[i, 2]))
            identical += int(all(torch.equal(res_a[k][r], ref[k][j]) for k in WANT))
    torch.cuda.synchronize()
    info = gpu_info()
    lines = []
    for k in names:
        t = np.array(times[k])
        lines.append({"arm": k, "audio_s_per_s": round(arms[k][2] / float(np.median(t))), "ms_median": round(float(np.median(t)) * 1e3, 3),
                      "ms_min": round(float(t.min()) * 1e3, 3), "ms_max": round(float(t.max()) * 1e3, 3), "reps": len(t),
                      "clips": N_CLIPS, "audio_s": round(arms[k][2], 1), "cfg": "1024/512 log_mel+mfcc", **info})
    lines.append({"check": "a_ragged rows == b_per_length rows, bit for bit", "clips_identical": identical, "clips": N_CLIPS,
                  "distinct_lengths": len(groups), "total_frames": total, "input_gb": round(n_samples * 4 / 1e9, 3)})
    text = "\n".join(json.dumps(line) for line in lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
