"""WAV decoding on the GPU (dspx_decode_ragged) against the host path it replaces.

Per case, 2000 seeded clips of 5 s at 44.1 kHz, held as the WAV data chunks would store them (stereo PCM16 is 1.76 GB
in, larger than the 126 MB L2):
  stereo_pcm16, stereo_pcm24, surround51_pcm16 (6 channels), mono_f32, mono_pcm8
Arms, timed with CUDA events after a warm-up, input already on the device:
  kernel        dspx_decode_ragged alone, without and with normalisation; bytes moved (computed from the shapes: input
                bytes, float32 outputs, and the second pass each clip takes when normalising) over time, and their
                share of the B200's 7.7 TB/s
  embed_44k     decode with normalisation + MFCC embeddings (one ragged feature launch) at 44.1 kHz
  embed_16k     decode + resample to 16 kHz with normalisation + embeddings at 16 kHz
  host_16k      read_wav + np.mean + scipy resample_poly + normalize_audio (load_audio + normalize_audio) on all
                host cores, from WAV files of a 64-clip subset
A bit check of sampled clips of both GPU arms against load_audio runs in the same job.  Every line carries the GPU
name and its power limit, read in the same run.

    python benchmarks/decode_bench.py [--iters 5] [--out profiles/r04_decode_bench.jsonl]
"""
import sys; sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parents[1]))  # noqa: E401,E702
import argparse
import json
import os
import struct
import subprocess
import tempfile
import time
from concurrent.futures import ProcessPoolExecutor
from pathlib import Path

import numpy as np
import torch

from dsp_final_b200 import _lib
from dsp_final_b200.batch import _decode_layout, decode_device, features_packed, pack_files
from dsp_final_b200.dsp.mfcc import MfccConfig

SR, N_CLIPS, SECONDS = 44100, 2000, 5
HBM = 7.7e12
# case -> (channels, dtype code, WAV format code, bits, bytes per sample)
CASES = {"stereo_pcm16": (2, 2, 1, 16, 2), "stereo_pcm24": (2, 4, 1, 24, 3), "surround51_pcm16": (6, 2, 1, 16, 2),
         "mono_f32": (1, 0, 3, 32, 4), "mono_pcm8": (1, 3, 1, 8, 1)}


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


def clip_bytes(case: str, rng) -> list:
    """read_wav_data tuples of the case's clips, from a seed."""
    c, dtype, _, bits, size = CASES[case]
    n = SECONDS * SR
    if bits == 32:
        data = rng.standard_normal((N_CLIPS, n * c), dtype=np.float32).view(np.uint8)
    else:
        data = np.frombuffer(rng.bytes(N_CLIPS * n * c * size), np.uint8).reshape(N_CLIPS, -1)
    return [(data[i], SR, c, dtype, n) for i in range(N_CLIPS)]


def write_wav(path: Path, case: str, data: np.ndarray) -> Path:
    c, _, code, bits, size = CASES[case]
    fmt = struct.pack("<HHIIHH", code, c, SR, SR * c * size, c * size, bits)
    body = b"WAVE" + b"fmt " + struct.pack("<I", 16) + fmt + b"data" + struct.pack("<I", len(data)) + data.tobytes()
    path.write_bytes(b"RIFF" + struct.pack("<I", len(body)) + body)
    return path


def _host_load(args):
    from dsp_final_b200.audio import load_audio, normalize_audio

    path, target = args
    return normalize_audio(load_audio(path, target)[0])


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "decode_bench needs a CUDA device"
    torch.cuda.set_device(0)
    info = gpu_info()
    lib = _lib.load()
    rng = np.random.default_rng(2025)
    audio_s = N_CLIPS * SECONDS
    cfg44 = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    cfg16 = MfccConfig(sample_rate=16000, frame_length=512, hop_length=256)
    lines = []
    tmp = Path(tempfile.mkdtemp(prefix="decode_bench_"))
    workers = os.cpu_count() or 1
    bad = checked = 0

    def emit(d):
        d.update(info)
        print(json.dumps(d), flush=True)
        lines.append(d)

    for case, (c, dtype, _, _, size) in CASES.items():
        parsed = clip_bytes(case, rng)
        staging, offsets = pack_files(parsed)
        data = staging.cuda()
        table, total = _decode_layout(lib, offsets, parsed, list(range(N_CLIPS)))
        out = torch.zeros(total, dtype=torch.float32, device="cuda")
        table_dev = torch.from_numpy(table.view(np.uint8)).cuda()
        ws_bytes = int(lib.dspx_decode_workspace(N_CLIPS))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream

        def kernel(normalize):
            _lib.check(lib.dspx_decode_ragged(data.data_ptr(), table_dev.data_ptr(), table.ctypes.data, N_CLIPS,
                                              int(normalize), out.data_ptr(), ws.data_ptr(), ws_bytes, stream))

        n_in, n_out = int(sum(len(p[0]) for p in parsed)), N_CLIPS * SECONDS * SR
        fb = c * size
        for normalize in (False, True):
            t = timed(lambda: kernel(normalize), args.iters)
            extra = 0 if not normalize else (n_in if fb < 8 else 8 * n_out)      # decode.cuh: dec_recompute
            nbytes = n_in + 4 * n_out + extra
            emit({"arm": "kernel", "case": case, "normalize": normalize, "ms": t * 1e3, "audio_s_per_s": audio_s / t,
                  "gbytes": nbytes / 1e9, "gbytes_per_s": nbytes / t / 1e9, "hbm_share": nbytes / t / HBM})
        t = timed(lambda: features_packed(decode_device(data, offsets, parsed, 44100, True), cfg44, ("embed",)), args.iters)
        emit({"arm": "embed_44k", "case": case, "ms": t * 1e3, "audio_s_per_s": audio_s / t})
        t = timed(lambda: features_packed(decode_device(data, offsets, parsed, 16000, True), cfg16, ("embed",)), args.iters)
        emit({"arm": "embed_16k", "case": case, "ms": t * 1e3, "audio_s_per_s": audio_s / t})

        sub = 64
        paths = [write_wav(tmp / f"{case}_{i}.wav", case, parsed[i][0]) for i in range(sub)]
        with ProcessPoolExecutor(workers) as pool:
            list(pool.map(_host_load, [(p, 16000) for p in paths[:workers]]))      # warm the workers
            t0 = time.perf_counter()
            ref16 = list(pool.map(_host_load, [(p, 16000) for p in paths], chunksize=2))
            t = time.perf_counter() - t0
        emit({"arm": "host_16k", "case": case, "clips": sub, "cores": workers, "ms_per_2000": t / sub * N_CLIPS * 1e3,
              "audio_s_per_s": sub * SECONDS / t})

        for target, refs in ((16000, ref16), (44100, None)):
            packed = decode_device(data, offsets, parsed, target, True)
            host = packed.samples.cpu().numpy()
            for i in rng.choice(sub, 6, replace=False):
                want = refs[i] if refs is not None else _host_load((paths[i], target))
                got = host[packed.starts[i]:packed.starts[i] + packed.lengths[i]]
                bad += int(not np.array_equal(got.view(np.uint32), want.astype(np.float32).view(np.uint32)))
                checked += 1
        for p in paths:
            p.unlink()
        del data, out, staging
        torch.cuda.empty_cache()
    emit({"arm": "bit_identity_vs_load_audio", "clips_checked": checked, "mismatches": bad})
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")
    assert bad == 0, "decoded clips differ from load_audio"


if __name__ == "__main__":
    main()
