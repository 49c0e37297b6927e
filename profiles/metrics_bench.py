"""Throughput of the device speech-quality metrics (deepfilternet_b200.metrics.evaluate -> dfb_metrics) in audio-seconds
scored per second, beside the reference's CPU implementations.

  python profiles/metrics_bench.py --out OUT.json [--batch 512 --seconds 10 --reps 5]
      GPU: every metric together and each alone, 48 kHz and 16 kHz inputs, CUDA-event timing of whole evaluate() calls
      on device-resident inputs (the inputs, 2 x 512 x 10 s x 48 kHz float32 = 1.97 GB, are far larger than L2);
      a second pass under torch.profiler for the per-kernel device times.  Records the card name and power
      limit of the same run.  Adds the CPU figures of --reference-json when that file exists.
  DFB_REFERENCE_ROOT=<reference tree> python profiles/metrics_bench.py --reference --out REF.json
      CPU: the reference's df.stoi.stoi, df.sepm.SNRseg + llr + wss and si_sdr_speechmetrics on one core (torch with one
      thread), 3 s utterances at 16 kHz, as its evaluation code calls them per file.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import platform
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def speech_like(B: int, T: int, sr: int, seed: int, device) -> tuple:
    """Seeded harmonic source with a 4 Hz envelope over a noise floor, and a degraded copy (+ noise at 5 dB SNR)."""
    g = torch.Generator(device=device).manual_seed(seed)
    t = torch.arange(T, device=device, dtype=torch.float32) / sr
    f0 = 100 + 120 * torch.rand(B, 1, generator=g, device=device)
    x = torch.zeros(B, T, device=device)
    for h in range(1, 16):
        x += torch.sin(2 * math.pi * f0 * h * t + 6.283 * torch.rand(B, 1, generator=g, device=device)) / h
    x *= (0.05 + torch.sin(2 * math.pi * 4.0 * t + 6.283 * torch.rand(B, 1, generator=g, device=device)).clamp_min(0) ** 2)
    x = 0.1 * x / x.pow(2).mean(1, keepdim=True).sqrt() + 0.005 * torch.randn(B, T, generator=g, device=device)
    y = 0.9 * x + 0.056 * torch.randn(B, T, generator=g, device=device) * x.pow(2).mean(1, keepdim=True).sqrt() / 0.1
    return x.contiguous(), y.contiguous()


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def bench_gpu(args) -> dict:
    from deepfilternet_b200 import metrics
    assert torch.cuda.is_available(), "the device benchmark needs a GPU"
    dev = torch.device("cuda", 0)
    res = {"card": card(), "batch": args.batch, "seconds": args.seconds, "reps": args.reps, "runs": []}
    for sr in (48000, 16000):
        T = int(args.seconds * sr)
        x, y = speech_like(args.batch, T, sr, 7, dev)
        audio_s = args.batch * args.seconds
        for sel in (metrics.METRICS, ("stoi",), ("sisdr",), ("ssnr",), ("llr",), ("wss",), ("ssnr", "llr", "wss")):
            metrics.evaluate(x, y, sr, metrics=sel)   # warm-up: module load, allocator pools
            torch.cuda.synchronize()
            times = []
            for _ in range(args.reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                metrics.evaluate(x, y, sr, metrics=sel)
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1) / 1e3)
            med = float(np.median(times))
            run = {"sr": sr, "metrics": list(sel), "median_s": med, "min_s": float(min(times)),
                   "audio_s_per_s": audio_s / med}
            res["runs"].append(run)
            print(json.dumps(run), flush=True)
        # per-kernel device times of one all-metrics call (torch.profiler, a pass of its own)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            metrics.evaluate(x, y, sr)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA":
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                kern[ev.key[:80]] = {"count": int(ev.count), "ms": float(t) / 1e3}
        res[f"kernels_{sr}"] = kern
        print(sr, json.dumps(kern), flush=True)
        del x, y
        torch.cuda.empty_cache()
    if os.path.exists(args.reference_json):
        res["reference_cpu"] = json.load(open(args.reference_json))
    return res


def bench_reference(args) -> dict:
    import types
    import gen_golden_metrics as ggm
    import ref_harness as rh
    stub = types.ModuleType("pesq")
    stub.pesq = None
    sys.modules["pesq"] = stub
    rh.import_reference()
    import df.sepm as sepm
    import df.stoi as dstoi
    sisdr = ggm.si_sdr_speechmetrics()
    torch.set_num_threads(1)
    sr, secs, n = 16000, 3.0, 4
    x, y = speech_like(n, int(secs * sr), sr, 7, "cpu")
    x, y = x.numpy(), y.numpy()
    dstoi.stoi(torch.from_numpy(x[:1]), torch.from_numpy(y[:1]), sr)   # first-call overhead (resampler kernel, imports)
    out = {"host_cpu": platform.processor() or platform.machine(), "cores": os.cpu_count(), "threads_used": 1,
           "utterance_s": secs, "sr": sr, "utterances": n, "note": "reference Python/numpy on one CPU core of the build host"}
    for name, fn in (("stoi", lambda a, b: dstoi.stoi(torch.from_numpy(a)[None], torch.from_numpy(b)[None], sr)),
                     ("sisdr", lambda a, b: sisdr(a, b)),
                     ("ssnr+llr+wss", lambda a, b: (sepm.SNRseg(a, b, sr), sepm.llr(a, b, sr), sepm.wss(a, b, sr)))):
        t0 = time.perf_counter()
        for i in range(n):
            fn(x[i], y[i])
        dt = time.perf_counter() - t0
        out[name] = {"s_per_utterance": dt / n, "audio_s_per_s_one_core": n * secs / dt}
        print(name, out[name], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", action="store_true", help="time the reference's CPU functions instead")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--reference-json", default=os.path.join(ROOT, "profiles", "metrics_bench_reference_cpu.json"))
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    res = bench_reference(args) if args.reference else bench_gpu(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
