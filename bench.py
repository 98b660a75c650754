#!/usr/bin/env python
"""Headline benchmark: MFCC + log-mel extraction throughput in audio-seconds per second.

Workload (BASELINE.json configs[1]): an ESC-50-shaped synthetic set, 2000 clips x 5 s mono at
44.1 kHz per GPU, frame 1024 / hop 512, 40 mels, 13 MFCCs; one "step" = one pass of the fused
feature kernel over the whole set, producing MFCC [2000,429,13] and log-mel [2000,429,40].

    python bench.py [--gpus N --steps K --warmup W]            our arm (CUDA kernels via the C ABI)
    python bench.py --impl reference [...]                     the CPU arm (oracle port, all host threads)

Under torchrun (N > 1) every rank owns its own 2000-clip shard (clips are independent: weak
scaling, no data-path collective); the time is the max over ranks and `value` the aggregate.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

SR, CLIP_LEN, FL, HOP, N_MELS, N_MFCC = 44_100, 220_500, 1024, 512, 40, 13
CLIP_SECONDS = CLIP_LEN / SR
DUMP_CLIPS = 512                            # --dump-outputs: 512 x 429 x (13 + 40) float32 = 46.6 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=("ours", "reference"), default="ours")
    ap.add_argument("--clips", type=int, default=2000, help="clips per GPU (ESC-50 has 2000)")
    ap.add_argument("--outputs", default="mfcc+log_mel", choices=("mfcc", "log_mel", "mfcc+log_mel"))
    ap.add_argument("--kernel", default="auto", choices=("auto", "generic", "warp8"))
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--stft-steps", type=int, default=10, help="secondary stft() measurement (0 = skip)")
    ap.add_argument("--retrieval-steps", type=int, default=3, help="secondary cosine top-20 measurement (0 = skip)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, default=None,
                    help=f"after the timed steps, write the last step's features of a fixed, seeded sample of "
                         f"{DUMP_CLIPS} of rank 0's clips as float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def dump_outputs(out_dir: Path, outputs: dict, n_clips: int) -> None:
    """Write rows of each [clips, frames, coeffs] output for a sample of clips that depends only on n_clips."""
    import torch

    sel = np.sort(np.random.default_rng(0).choice(n_clips, min(n_clips, DUMP_CLIPS), replace=False))
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, t in outputs.items():
        np.save(out_dir / f"{name}.npy", t[torch.as_tensor(sel, device=t.device)].cpu().numpy())


def algorithmic_bytes_per_clip(outputs: str, n_frames: int) -> int:
    """SURVEY.md 8d: every sample read once + features written once."""
    b = 4 * CLIP_LEN
    if "mfcc" in outputs:
        b += 4 * n_frames * N_MFCC
    if "log_mel" in outputs:
        b += 4 * n_frames * N_MELS
    return b


def measured_peaks() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def measured_tensor_peak() -> tuple[float, str]:
    """Dense bf16 TFLOP/s (MEASURED_PEAKS.json, burst figure; nominal 2250 otherwise)."""
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["bf16_tflops"]), "measured"
        except Exception:
            pass
    return 2250.0, "fallback"


def workload_config(outputs: str, clips: int, world: int) -> dict:
    """`config` of the JSON line: the workload, identical for our arm and for the CPU (reference) arm."""
    return {"workload": f"ESC-50-shaped synthetic set: {clips} clips x 5 s @44.1 kHz per GPU, frame {FL} hop {HOP}, "
                        f"{N_MELS} mels, {N_MFCC} MFCC (BASELINE.json configs[1])",
            "outputs": outputs, "clips_per_gpu": clips,
            "l2_policy": "inputs_larger_than_l2 (1.76 GB per pass vs 126 MB L2)", "parallelism": f"clip-sharded x{world}"}


def gpu_topology(index: int) -> dict:
    """PCI bus id, NUMA node and local CPU list of GPU `index` (sysfs; -1 / None when the kernel does not say)."""
    info = {"gpu": index, "pci": None, "numa_node": -1, "local_cpus": None}
    try:
        import pynvml

        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        info["pci"] = bus
        dev = Path("/sys/bus/pci/devices") / bus.lower()[-12:]
        if (dev / "numa_node").exists():
            info["numa_node"] = int((dev / "numa_node").read_text().strip())
        if (dev / "local_cpulist").exists():
            info["local_cpus"] = (dev / "local_cpulist").read_text().strip()
    except Exception:
        pass
    return info


def parse_cpulist(text: str) -> set:
    cpus = set()
    for part in (text or "").split(","):
        part = part.strip()
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_gpu_numa(index: int) -> dict:
    """Pin this rank's threads to the CPUs local to its GPU *before* pinned buffers are allocated, so that
    first-touch places the staging memory on the GPU's NUMA node.  No-op when the platform reports one node."""
    topo = gpu_topology(index)
    try:
        allowed = os.sched_getaffinity(0)
        local = parse_cpulist(topo["local_cpus"]) & allowed
        if topo["numa_node"] >= 0 and local and local != allowed:
            os.sched_setaffinity(0, local)
            topo["bound"] = True
        else:
            topo["bound"] = False
        topo["affinity_cpus"] = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        topo["bound"] = False
    return topo


def host_cores() -> int:
    """Host threads this process may use (torchrun exports OMP_NUM_THREADS=1, so ask the OS instead)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:                                    # pragma: no cover
        return max(1, os.cpu_count() or 1)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                break
            time.sleep(self.period)

    def stop(self) -> dict:
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_arm(args, n_frames: int):
    """The CPU implementation of the path (oracle port of src/dsp, all host threads)."""
    from dsp_final_b200 import synth
    from oracle import oracle as O

    cfg = O.OracleConfig(SR, FL, HOP, n_mels=N_MELS, n_mfcc=N_MFCC)
    cores = host_cores()
    want = tuple(n for n in ("mfcc", "log_mel") if n in args.outputs)
    per_step = max(4 * cores, 64)                          # bounded sample of the 2000-clip set: >= 4 clips per core
    clips = synth.host_clips(min(per_step, 64), seed=1234)
    if clips.shape[0] < per_step:
        clips = np.concatenate([clips] * ((per_step + clips.shape[0] - 1) // clips.shape[0]))[:per_step]
    return O, cfg, cores, want, clips


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    n_frames = 1 + (CLIP_LEN - FL) // HOP
    O, cfg, cores, want, clips = cpu_arm(args, n_frames)
    per_step = clips.shape[0]
    O.features_batch(clips, cfg, want=want, n_threads=cores)                       # first step (counts as warm-up)
    steps, warm = args.steps, max(0, args.warmup - 1)
    for _ in range(warm):
        O.features_batch(clips, cfg, want=want, n_threads=cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.features_batch(clips, cfg, want=want, n_threads=cores)
    dt = time.perf_counter() - t0
    value = per_step * CLIP_SECONDS * steps / dt
    sample = (f"{per_step} of the {args.clips} synthetic 5 s clips per step x {steps} steps, C port of src/dsp "
              f"(complex128 radix-2), OpenMP over clips on {cores} host threads")
    line = {
        "impl": "reference", "metric": "mfcc_logmel_audio_seconds_per_second", "value": value,
        "unit": "audio-s/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.outputs, args.clips, args.gpus),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist

    from dsp_final_b200 import _lib, synth
    from dsp_final_b200.batch import features_batch
    from dsp_final_b200.dist import init_process_group
    from dsp_final_b200.dsp.mfcc import MfccConfig
    from dsp_final_b200.plan import get_plan

    _lib.load()
    _lib.require_device()
    rank, world, local = init_process_group()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    topo = bind_to_gpu_numa(local)          # before any pinned allocation (first touch decides the NUMA node)
    cfg = MfccConfig(sample_rate=SR, frame_length=FL, hop_length=HOP, n_mels=N_MELS, n_mfcc=N_MFCC)
    plan = get_plan(cfg, local, args.kernel)
    n_frames = plan.num_frames(CLIP_LEN)
    want = tuple(n for n in ("mfcc", "log_mel") if n in args.outputs)
    b = args.clips
    lib = _lib.load()

    # inputs resident in HBM before the timed region (1.76 GB per GPU: larger than the 126 MB L2)
    clips = synth.device_clips(b, seed=1234, device=dev, first=rank * b)
    mf = torch.empty((b, n_frames, N_MFCC), dtype=torch.float32, device=dev) if "mfcc" in want else None
    lm = torch.empty((b, n_frames, N_MELS), dtype=torch.float32, device=dev) if "log_mel" in want else None
    stream = torch.cuda.current_stream(dev)

    def step():
        _lib.check(lib.dspx_features(plan.handle, clips.data_ptr(), b, CLIP_LEN, clips.stride(0),
                                     lm.data_ptr() if lm is not None else None,
                                     mf.data_ptr() if mf is not None else None, None, stream.cuda_stream),
                   "dspx_features")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    evs[0].record(stream)
    for i in range(args.steps):
        step()
        evs[i + 1].record(stream)
    barrier()
    clocks = sampler.stop()
    total_ms = evs[0].elapsed_time(evs[-1])
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * b * CLIP_SECONDS * args.steps / (total_ms * 1e-3)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, {name: out for name, out in (("mfcc", mf), ("log_mel", lm)) if out is not None}, b)

    # roofline of the dominant (only) kernel of the step
    bytes_per_launch = b * algorithmic_bytes_per_clip(args.outputs, n_frames)
    avg_launch_s = float(np.mean(per_launch_ms)) * 1e-3
    peak, peak_src = measured_peaks()
    achieved = bytes_per_launch / avg_launch_s / 1e9
    traffic = None
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get(plan.kernel, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "kernel": f"feat_{plan.kernel}",
                "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": avg_launch_s * 1e3,
                "note": "co-bound by FP32 issue + shared-memory bandwidth (DESIGN.md): 2.67 MFLOP per audio-second"}

    # secondary: the stft() entry point on the same clips (complex64 [B, 429, 513] out: write-heavy, HBM-bound)
    stft_info = None
    if args.stft_steps > 0:
        from dsp_final_b200.batch import stft_batch

        s_out = stft_batch(clips, FL, HOP)
        for _ in range(2):
            stft_batch(clips, FL, HOP)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(args.stft_steps):
            s_out = stft_batch(clips, FL, HOP)
        s1.record(stream)
        barrier()
        st_ms = s0.elapsed_time(s1) / args.stft_steps
        tt = torch.tensor([st_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        st_ms = float(tt.item())
        st_bytes = b * (4 * CLIP_LEN + 8 * n_frames * (FL // 2 + 1))
        stft_info = {"value": world * b * CLIP_SECONDS / (st_ms * 1e-3), "unit": "audio-s/s", "ms_per_step": st_ms,
                     "roofline": {"bound": "hbm", "achieved": st_bytes / (st_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": st_bytes / (st_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": st_bytes},
                     "kernel": "feat_warp8 (STFT mode)", "steps": args.stft_steps}
        stft_sel = s_out[[0, b - 1]][:, [0, 1, n_frames - 1]].cpu().numpy()
        del s_out

    # secondary: MFCC-embedding retrieval (src/retrieval/retrieval.py): top-20 of 20 000 queries against 1 000 000
    # database embeddings of dimension 26 per GPU (synthetic unit-variance embeddings), through dspx_cosine_topk
    retrieval_info = None
    if args.retrieval_steps > 0:
        from dsp_final_b200 import retrieval as R

        RQ, RDB, RDIM, RK = 20_000, 1_000_000, 26, 20
        gen = torch.Generator(device=dev)
        gen.manual_seed(77 + rank)
        r_q = torch.randn((RQ, RDIM), generator=gen, device=dev)
        r_db = torch.randn((RDB, RDIM), generator=gen, device=dev)
        r_idx = R.cosine_topk(r_q, r_db, RK)
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record(stream)
        for _ in range(args.retrieval_steps):
            r_idx = R.cosine_topk(r_q, r_db, RK)
        r1.record(stream)
        barrier()
        r_ms = r0.elapsed_time(r1) / args.retrieval_steps
        tt = torch.tensor([r_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        r_ms = float(tt.item())
        f16_peak, tpeak_src = measured_tensor_peak()               # kind::f16 MMAs run at the dense bf16 rate
        useful = 2.0 * RDIM * RQ * RDB / (r_ms * 1e-3) / 1e12
        retrieval_info = {"value": world * RQ / (r_ms * 1e-3), "unit": "queries/s", "ms_per_step": r_ms,
                          "pair_scores_per_s": world * RQ * RDB / (r_ms * 1e-3), "n_queries": RQ, "n_db": RDB, "dim": RDIM, "k": RK,
                          "roofline": {"bound": "tensor", "achieved": useful, "peak": f16_peak, "unit": "TFLOP/s",
                                       "frac": useful / f16_peak, "peak_source": tpeak_src + " bf16 (= fp16 rate)",
                                       "executed_tflops": useful * 192.0 / 52.0, "tensor_cycles_per_tile": 768,
                                       "note": "achieved = 2*dim flop per pair (what the path needs); the kernel executes the three terms of "
                                               "the hi/lo split (lo*hi + hi*lo + hi*hi, K = 32 each: 192 flop per pair) as 12 kind::f16 MMAs = "
                                               "768 tensor cycles per 256 x 128 tile (round 1: 24 TF32 MMAs = 1536 cycles), plus float64 "
                                               "re-scoring of the rows that pass"},
                          "kernel": "cosine_topk_tc (tcgen05 split-fp16 filter, TMA bulk-copy operands, exact float64 re-score)",
                          "steps": args.retrieval_steps}
        r_sel_q = r_q[:8].cpu().numpy()
        r_sel_idx = r_idx[:8].cpu().numpy()
        r_db_host = r_db.cpu().numpy() if rank == 0 else None
        del r_q, r_db, r_idx

    # end to end through the host-buffer C ABI: pinned host clips in, host features out
    e2e = e2e_pcm16 = None
    if args.e2e_steps > 0:
        h_clips = torch.empty((b, CLIP_LEN), dtype=torch.float32, pin_memory=True)
        h_clips.copy_(clips)
        h_mf = torch.empty((b, n_frames, N_MFCC), dtype=torch.float32, pin_memory=True) if mf is not None else None
        h_lm = torch.empty((b, n_frames, N_MELS), dtype=torch.float32, pin_memory=True) if lm is not None else None
        torch.cuda.synchronize(dev)
        d2h = (h_mf.numel() * 4 if h_mf is not None else 0) + (h_lm.numel() * 4 if h_lm is not None else 0)

        def timed_all_ranks(fn, reps):
            """Wall time of `reps` calls of a synchronous host-API call, all ranks at once, max over ranks."""
            fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        # the ceiling of this box for the same bytes: plain pinned->device and device->pinned copies on two
        # streams (full duplex), every rank at once -- no kernel, no library.  e2e is reported against it.
        d_in = torch.empty((b, CLIP_LEN), dtype=torch.float32, device=dev)
        d_out = torch.empty(d2h // 4, dtype=torch.float32, device=dev)
        h_out = torch.empty(d2h // 4, dtype=torch.float32, pin_memory=True)
        s_up, s_dn = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

        def copy_step():
            with torch.cuda.stream(s_up):
                d_in.copy_(h_clips, non_blocking=True)
            with torch.cuda.stream(s_dn):
                h_out.copy_(d_out, non_blocking=True)
            s_up.synchronize()
            s_dn.synchronize()

        dt_copy = timed_all_ranks(copy_step, args.e2e_steps)
        ceiling = world * b * CLIP_SECONDS * args.e2e_steps / dt_copy
        copy_gbs = (b * CLIP_LEN * 4 + d2h) * args.e2e_steps / dt_copy / 1e9
        del d_in, d_out, h_out

        def e2e_step():
            _lib.check(lib.dspx_features_host(plan.handle, h_clips.data_ptr(), b, CLIP_LEN, CLIP_LEN,
                                              h_lm.data_ptr() if h_lm is not None else None,
                                              h_mf.data_ptr() if h_mf is not None else None, None),
                       "dspx_features_host")

        dt = timed_all_ranks(e2e_step, args.e2e_steps)
        e2e = {"value": world * b * CLIP_SECONDS * args.e2e_steps / dt, "unit": "audio-s/s",
               "h2d_bytes_per_step": b * CLIP_LEN * 4, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
               "api": "dspx_features_host (pinned host buffers in and out)",
               "copy_ceiling": {"value": ceiling, "unit": "audio-s/s", "gb_per_s_per_gpu": copy_gbs,
                                "what": "same bytes as plain cudaMemcpyAsync pinned<->device, both directions overlapped, all ranks at once"},
               "frac_of_copy_ceiling": (world * b * CLIP_SECONDS * args.e2e_steps / dt) / ceiling}
        # the host path and the device path run the same kernel: results must be identical
        if h_mf is not None:
            assert torch.equal(h_mf[:8], mf[:8].cpu()), "host-pipeline result differs from device-path result"
        # the same call fed with PCM16 clips (what ESC-50 files hold; SURVEY 8f row f2): int16 -> float32 and peak
        # normalisation happen in the feature kernel's sample loads, host->device bytes halve
        h_pcm = torch.empty((b, CLIP_LEN), dtype=torch.int16, pin_memory=True)
        h_pcm.copy_((clips * 32767.0).round().to(torch.int16))
        torch.cuda.synchronize(dev)

        def pcm_step():
            _lib.check(lib.dspx_features_host_pcm16(plan.handle, h_pcm.data_ptr(), b, CLIP_LEN, CLIP_LEN, 1,
                                                    h_lm.data_ptr() if h_lm is not None else None,
                                                    h_mf.data_ptr() if h_mf is not None else None, None),
                       "dspx_features_host_pcm16")

        dtp = timed_all_ranks(pcm_step, args.e2e_steps)
        e2e_pcm16 = {"value": world * b * CLIP_SECONDS * args.e2e_steps / dtp, "unit": "audio-s/s",
                     "h2d_bytes_per_step": b * CLIP_LEN * 2, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
                     "api": "dspx_features_host_pcm16 (int16 PCM in, peak normalisation on the GPU)"}
        pcm_mf_sel = h_mf[:2].clone() if h_mf is not None else None
        pcm_src_sel = h_pcm[:2].clone()
        del h_clips, h_pcm

    # configs[4] in miniature, N > 1 only: every rank holds 125 000 clip embeddings (100 000 database + 25 000
    # queries, the 80/20 split); ONE NCCL all-gather of the database shards, local top-20, one all-reduce of the
    # hit counters (dsp_final_b200.dist.sharded_retrieval = src/tasks/retrieval.py:11-21 at scale)
    sharded_info = None
    sharded_check = None
    if world > 1 and args.retrieval_steps > 0:
        from dsp_final_b200 import dist as D
        from dsp_final_b200.batch import features_batch as fb

        S_DB, S_Q = 100_000, 25_000
        real = fb(clips, cfg, ("embed",))["embed"]                      # 2000 real MFCC embeddings of this rank's clips
        real_t = torch.arange(rank * b, rank * b + b, device=dev, dtype=torch.int32) % 50
        gen = torch.Generator(device=dev)
        gen.manual_seed(4000 + rank)
        src = torch.randint(0, b, (S_DB + S_Q,), generator=gen, device=dev)
        emb = real[src] * (1.0 + 0.05 * torch.randn((S_DB + S_Q, real.shape[1]), generator=gen, device=dev))
        tgt = real_t[src].contiguous()
        db_e, db_t, q_e, q_t = emb[:S_DB].contiguous(), tgt[:S_DB].contiguous(), emb[S_DB:].contiguous(), tgt[S_DB:].contiguous()
        D.sharded_retrieval(db_e, db_t, q_e, q_t, (10, 20))             # warm-up (NCCL channels, workspaces)
        barrier()
        phases = []
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(args.retrieval_steps):
            prof = {}
            s_res, s_idx = D.sharded_retrieval(db_e, db_t, q_e, q_t, (10, 20), profile=prof)
            phases.append(prof)
        s1.record(stream)
        barrier()
        s_ms = s0.elapsed_time(s1) / args.retrieval_steps
        tt = torch.tensor([s_ms] + [float(np.mean([p[k] for p in phases])) for k in ("gather_ms", "topk_ms", "reduce_ms")],
                          dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        s_ms, g_ms, t_ms, r_ms2 = [float(v) for v in tt.tolist()]
        gbytes = phases[-1]["gather_bytes"]
        sharded_info = {"value": world * S_Q / (s_ms * 1e-3), "unit": "queries/s", "ms_per_step": s_ms,
                        "n_queries": world * S_Q, "n_db": world * S_DB, "dim": int(emb.shape[1]), "k": 20,
                        "pair_scores_per_s": world * S_Q * world * S_DB / (s_ms * 1e-3),
                        "all_gather_ms": g_ms, "all_gather_bytes_received_per_rank": gbytes,
                        "all_gather_gb_per_s_per_rank": gbytes / (g_ms * 1e-3) / 1e9 if g_ms > 0 else None,
                        "topk_ms": t_ms, "hits_all_reduce_ms": r_ms2, "steps": args.retrieval_steps,
                        "top10_top20": [[k, h / n] for k, h, n in s_res],
                        "what": "per-rank shards of clustered MFCC embeddings (real embeddings of this rank's clips, jittered 5 %); "
                                "NCCL all-gather of database rows + targets, dspx_cosine_topk on the local queries, all-reduce of hit counts"}
        if rank == 0:
            full_db = D.all_gather_rows(db_e).cpu().numpy()
            sharded_check = (q_e[:64].cpu().numpy(), full_db, s_idx[:64].cpu().numpy())
        else:
            D.all_gather_rows(db_e)
        del emb, db_e, q_e

    topos = [topo]
    if world > 1:
        topos = [None] * world
        dist.all_gather_object(topos, topo)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # parity spot check + CPU baseline (rank 0, N = 1 only for the baseline)
    from oracle import oracle as O

    ocfg = O.OracleConfig(SR, FL, HOP, n_mels=N_MELS, n_mfcc=N_MFCC)
    sel = [0, b // 2, b - 1]
    host_sel = clips[sel].cpu().numpy()
    ref = O.features_batch(host_sel, ocfg, want=want)
    parity = {}
    if mf is not None:
        parity["mfcc_rel_err"] = O.relative_error(mf[sel].cpu().numpy(), ref["mfcc"])
    if lm is not None:
        parity["log_mel_rel_err"] = O.relative_error(lm[sel].cpu().numpy(), ref["log_mel"])
    parity["clips_checked"] = len(sel)
    if stft_info is not None:
        ref_st = np.stack([O.stft(clips[i].cpu().numpy(), FL, HOP)[[0, 1, n_frames - 1]] for i in (0, b - 1)])
        parity["stft_rel_err"] = O.relative_error(stft_sel, ref_st)
    if retrieval_info is not None:
        parity["retrieval_top20_identical"] = bool(np.array_equal(r_sel_idx, O.cosine_topk(r_sel_q, r_db_host, 20)))
        parity["retrieval_queries_checked"] = 8
    if sharded_check is not None:
        sq, sdb, sidx = sharded_check
        parity["sharded_top20_identical"] = bool(np.array_equal(sidx, O.cosine_topk(sq, sdb, 20)))
        parity["sharded_queries_checked"] = int(sq.shape[0])
    if e2e_pcm16 is not None and pcm_mf_sel is not None:
        x = pcm_src_sel.numpy().astype(np.float32) / np.float32(32768.0)
        x = x / np.max(np.abs(x), axis=1, keepdims=True)
        parity["pcm16_mfcc_rel_err"] = O.relative_error(pcm_mf_sel.numpy(), O.features_batch(x, ocfg, want=("mfcc",))["mfcc"])
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        host = synth.host_clips(min(max(cores, 8), 64), seed=1234)
        t0 = time.perf_counter()
        O.features_batch(host[: max(1, min(cores, host.shape[0]))], ocfg, want=want, n_threads=cores)
        one = time.perf_counter() - t0
        reps = max(1, int(args.cpu_seconds / max(one, 1e-3)))
        n_cal = max(1, min(cores, host.shape[0]))
        t0 = time.perf_counter()
        for _ in range(reps):
            O.features_batch(host[:n_cal], ocfg, want=want, n_threads=cores)
        dtc = time.perf_counter() - t0
        cpu_baseline = {"value": n_cal * reps * CLIP_SECONDS / dtc, "unit": "audio-s/s", "cores": cores, "kind": "port",
                        "sample": f"{n_cal * reps} synthetic 5 s clips ({dtc:.1f} s), C port of src/dsp (complex128 radix-2), OpenMP over clips"}

    line = {
        "metric": "mfcc_logmel_audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.outputs, b, world),
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "e2e_pcm16": e2e_pcm16, "gpu_launches": args.steps,
        "stft": stft_info, "retrieval": retrieval_info, "retrieval_sharded": sharded_info,
        "clocks": clocks, "parity": parity, "topology": topos,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
