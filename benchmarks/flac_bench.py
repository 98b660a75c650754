"""FLAC decoding on the GPU (dspx_flac_decode) next to the WAV decoder on the same clips.

Per case, 2000 clips of 5 s at 44.1 kHz, written as FLAC files with LPC order 8 (Rice partition order 4, coefficients
of 15 bits) by tests/flac_ref.py's writer, and as WAV files of the same integers: 32 distinct synthetic clips
(synth.host_clips at 0.8 of full scale), each file read 62-63 times, so the batch is as large as 2000 distinct clips
(the L2 holds none of it) and the writer's time stays small; the files are in the page cache.  Cases: mono_pcm16,
stereo_pcm16, stereo_pcm24.  Arms (CUDA events after a warm-up; host arms by the wall clock):
  ratio            FLAC file bytes over the WAV data bytes of the same integers
  read             read_flac_data / read_wav_data of the 2000 paths on one host core: file read plus, for FLAC, the
                   one pass that finds the frames
  kernel           dspx_flac_decode alone, input on the device, without and with normalisation
  embed_44k        decode with normalisation + MFCC embeddings (one ragged feature launch) at 44.1 kHz, from the
                   parsed tuples with the files' bytes on the device
  embed_16k        decode + resample to 16 kHz with normalisation + embeddings at 16 kHz, the same way
  files_to_embed   paths -> embeddings at 44.1 kHz as compute_embeddings runs it: read_*_data of every path, then
                   decode_packed (pinned staging, one host-to-device copy, decode) and one feature launch, for the
                   FLAC files and for the WAV files of the same clips
A bit check runs in the same job: the FLAC path's outputs equal the WAV path's for every clip, and sampled clips equal
the writer's integers scaled and averaged as load_audio does.  Every line carries the GPU name and power limit.

    python benchmarks/flac_bench.py [--iters 5] [--out profiles/r05_flac_bench.jsonl]
"""
import sys; sys.path[:0] = [str(__import__('pathlib').Path(__file__).resolve().parents[1]), str(__import__('pathlib').Path(__file__).resolve().parents[1] / "tests")]  # noqa: E401,E702,E501
import argparse
import json
import os
import struct
import tempfile
import time
from pathlib import Path
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import torch

import flac_ref as F
from decode_bench import gpu_info, timed
from dsp_final_b200 import _lib, synth
from dsp_final_b200.audio import read_flac_data, read_wav_data
from dsp_final_b200.batch import _flac_decode, _flac_layout, decode_device, decode_packed, features_packed, pack_files
from dsp_final_b200.dsp.mfcc import MfccConfig

SR, N_CLIPS, SECONDS, DISTINCT = 44100, 2000, 5, 32
CASES = {"mono_pcm16": (1, 16), "stereo_pcm16": (2, 16), "stereo_pcm24": (2, 24)}


def _clip(args):
    """(FLAC bytes, WAV data bytes, integers) of distinct clip j of a case."""
    j, c, bps = args
    n = SECONDS * SR
    top = (1 << (bps - 1)) - 1
    x = np.stack([np.round(synth.host_clips(1, seed=100 + ch, length=n, first=j)[0].astype(np.float64) * 0.8 * top)
                  for ch in range(c)], 1).astype(np.int64).clip(-top - 1, top)
    data = F.encode(x, SR, bps, blocks=4096, opts={"assignment": "mid_side" if c == 2 else "independent",
                                                    "subframes": {"kind": "lpc", "order": 8, "precision": 15, "porder": 4}})
    if bps == 16:
        raw = x.astype("<i2").tobytes()
    else:
        raw = x.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3].tobytes()
    return bytes(data), raw, x


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "flac_bench needs a CUDA device"
    torch.cuda.set_device(0)
    info = gpu_info()
    lib = _lib.load()
    audio_s = N_CLIPS * SECONDS
    cfg44 = MfccConfig(sample_rate=44100, frame_length=1024, hop_length=512)
    cfg16 = MfccConfig(sample_rate=16000, frame_length=512, hop_length=256)
    lines = []
    bad = checked = 0
    tmp = Path(tempfile.mkdtemp(prefix="flac_bench_"))

    def emit(d):
        d.update(info)
        print(json.dumps(d), flush=True)
        lines.append(d)

    for case, (c, bps) in CASES.items():
        t0 = time.perf_counter()
        with ProcessPoolExecutor(os.cpu_count() or 1) as pool:
            distinct = list(pool.map(_clip, [(j, c, bps) for j in range(DISTINCT)]))
        write_s = time.perf_counter() - t0
        fpaths, wpaths = [], []
        for k, (fl, raw, _) in enumerate(distinct):
            fpaths.append(tmp / f"{case}_{k}.flac")
            fpaths[-1].write_bytes(fl)
            fmt = struct.pack("<HHIIHH", 1, c, SR, SR * c * bps // 8, c * bps // 8, bps)
            body = b"WAVE" + b"fmt " + struct.pack("<I", 16) + fmt + b"data" + struct.pack("<I", len(raw)) + raw
            wpaths.append(tmp / f"{case}_{k}.wav")
            wpaths[-1].write_bytes(b"RIFF" + struct.pack("<I", len(body)) + body)
        fpaths = [fpaths[i % DISTINCT] for i in range(N_CLIPS)]
        wpaths = [wpaths[i % DISTINCT] for i in range(N_CLIPS)]
        for reader, paths, name in ((read_flac_data, fpaths, "flac"), (read_wav_data, wpaths, "wav")):
            [reader(p) for p in paths[:DISTINCT]]                                 # the page cache
            t0 = time.perf_counter()
            parsed = [reader(p) for p in paths]
            t = time.perf_counter() - t0
            emit({"arm": "read", "case": case, "input": name, "ms": t * 1e3,
                  "file_gbytes_per_s": sum(p.stat().st_size for p in paths) / t / 1e9})
        flac = [read_flac_data(p) for p in fpaths]
        wav = [read_wav_data(p) for p in wpaths]
        n_flac, n_wav = sum(len(p[0]) for p in flac), sum(len(p[0]) for p in wav)
        emit({"arm": "ratio", "case": case, "flac_bytes": n_flac, "wav_data_bytes": n_wav, "ratio": n_flac / n_wav,
              "writer_s": write_s})

        staging, offsets = pack_files(flac)
        data = staging.cuda()
        files, frames, total = _flac_layout(lib, offsets, flac, list(range(N_CLIPS)))
        out = torch.zeros(total, dtype=torch.float32, device="cuda")
        tabs = (files, frames, 0, list(range(N_CLIPS)))
        for normalize in (False, True):
            t = timed(lambda: _flac_decode(lib, data, tabs, normalize, out, out.device), args.iters)
            emit({"arm": "kernel", "case": case, "normalize": normalize, "frames": len(frames), "ms": t * 1e3,
                  "audio_s_per_s": audio_s / t, "in_gbytes_per_s": n_flac / t / 1e9})
        t = timed(lambda: features_packed(decode_device(data, offsets, flac, 44100, True), cfg44, ("embed",)), args.iters)
        emit({"arm": "embed_44k", "case": case, "ms": t * 1e3, "audio_s_per_s": audio_s / t})
        t = timed(lambda: features_packed(decode_device(data, offsets, flac, 16000, True), cfg16, ("embed",)), args.iters)
        emit({"arm": "embed_16k", "case": case, "ms": t * 1e3, "audio_s_per_s": audio_s / t})
        del data, out, staging
        torch.cuda.empty_cache()

        for name, reader, paths in (("flac", read_flac_data, fpaths), ("wav", read_wav_data, wpaths)):
            t = timed(lambda: features_packed(decode_packed([reader(p) for p in paths], 44100, True, names=paths), cfg44,
                                              ("embed",)), args.iters)
            emit({"arm": "files_to_embed", "case": case, "input": name, "ms": t * 1e3, "audio_s_per_s": audio_s / t})

        for target in (44100, 16000):
            a = decode_packed(flac, target, True)
            b = decode_packed(wav, target, True)
            same = np.array_equal(a.samples.cpu().numpy().view(np.uint32), b.samples.cpu().numpy().view(np.uint32))
            bad += int(not same)
            checked += 1
        a = decode_packed(flac, None, False)
        host = a.samples.cpu().numpy()
        for k in range(4):
            y = (distinct[k][2].astype(np.float64) / float(1 << (bps - 1))).astype(np.float32)
            y = y[:, 0] if c == 1 else np.mean(y, axis=1).astype(np.float32)
            got = host[a.starts[k]:a.starts[k] + a.lengths[k]]
            bad += int(not np.array_equal(got.view(np.uint32), y.view(np.uint32)))
            checked += 1
        del a, b
        torch.cuda.empty_cache()
        for p in set(fpaths) | set(wpaths):
            p.unlink()
    emit({"arm": "bit_identity", "checks": checked, "mismatches": bad})
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")
    assert bad == 0, "FLAC outputs differ from the WAV path or from the written integers"


if __name__ == "__main__":
    main()
