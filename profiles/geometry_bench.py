"""Throughput of DeepFilterNet3 (seeded random weights) at several STFT geometries, device resident, in one process:
48000/960/480 (the specialised kernels, the in-run baseline) against the runtime mixed-radix kernels at 16000/320/160,
44100/882/441 and 48000/480/240.

    python profiles/geometry_bench.py OUT_DIR [--streams 128] [--seconds 10] [--steps 10] [--warmup 3]

Per geometry: step time (median of `steps` CUDA-event timed enhance_device calls after `warmup`), audio-s/s, and the
per-kernel times of the analysis and apply + synthesis kernels (dfb_profile_enable, a separate profiled pass) with
their HBM fraction from the algorithmic bytes per frame
    analysis  4 H read + 8 F + 4 E written;   apply  8 F + 4 E + 8 O nb_df read + 4 H written
against the HBM peak bench.py's peaks() reads (MEASURED_PEAKS.json, else labelled "fallback").  The GPU name and power
limit are read in the same run.  Writes OUT_DIR/geometry_bench.json.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GEOMETRIES = [(48000, 960, 480), (16000, 320, 160), (44100, 882, 441), (48000, 480, 240)]
KERNELS = {True: ("k_analysis", "k_apply_synthesis"), False: ("k_analysis_any", "k_apply_synthesis_any")}


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [s.strip() for s in r.stdout.strip().split(",")]
        info.update(smi_name=name, power_limit=power, sm_max_clock=clk)
    except Exception as e:  # the name from the runtime is still reported
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def run_geometry(geo, streams, seconds, steps, warmup, hbm_gbs):
    import torch
    from deepfilternet_b200 import DfNet, _lib, enhance_device, libdf
    from deepfilternet_b200.config import ModelConfig
    from deepfilternet_b200.weights import random_state_dict
    from tests_common import synth_audio
    sr, fft, hop = geo
    L = _lib.lib()
    cfg = ModelConfig(model="deepfilternet3", conv_ch=64, conv_lookahead=2, df_lookahead=2, emb_num_layers=3, df_num_layers=2,
                      lin_groups=16, enc_lin_groups=32, df_gru_skip="groupedlinear", df_pathway_kernel_size_t=5,
                      sr=sr, fft_size=fft, hop_size=hop)
    st = libdf.DF(sr, fft, hop, cfg.nb_erb, cfg.min_nb_erb_freqs)
    model = DfNet(cfg, random_state_dict(cfg, seed=1), st)
    audio = synth_audio(streams, sr * seconds, seed=1234, device="cuda", sr=sr)
    out = torch.empty_like(audio)
    for _ in range(warmup):
        enhance_device(model, st, audio, out=out)
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        enhance_device(model, st, audio, out=out)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = statistics.median(times)
    # profiled pass
    buf = ctypes.create_string_buffer(1 << 16)
    L.dfb_profile_report(buf, len(buf))
    L.dfb_profile_enable(1, None)
    psteps = 3
    for _ in range(psteps):
        enhance_device(model, st, audio, out=out)
    torch.cuda.synchronize()
    L.dfb_profile_report(buf, len(buf))
    L.dfb_profile_enable(0, None)
    prof = {}
    for ln in buf.value.decode().splitlines():
        name, cnt, tot = ln.rsplit(" ", 2)
        prof[name] = (int(cnt) / psteps, float(tot) / psteps)
    F, E, O, Fd = fft // 2 + 1, cfg.nb_erb, cfg.df_order, cfg.nb_df
    frames = streams * ((sr * seconds + fft) // hop)
    bytes_per_frame = {"analysis": 4 * hop + 8 * F + 4 * E, "apply": 8 * F + 4 * E + 8 * O * Fd + 4 * hop}
    kernels = {}
    for role, kname in zip(("analysis", "apply"), KERNELS[(fft, hop) == (960, 480)]):
        launches, kms = prof.get(kname, (0, 0.0))
        gbs = bytes_per_frame[role] * frames / (kms * 1e-3) / 1e9 if kms > 0 else None
        kernels[role] = dict(kernel=kname, launches_per_step=launches, ms_per_step=round(kms, 4),
                             bytes_per_frame=bytes_per_frame[role], achieved_gbs=gbs and round(gbs, 1),
                             hbm_fraction=gbs and round(gbs / hbm_gbs, 4))
    del model, st, audio, out
    torch.cuda.empty_cache()
    return dict(sr=sr, fft_size=fft, hop_size=hop, F=F, frames_per_step=frames, step_ms_median=round(ms, 3),
                step_ms_all=[round(t, 3) for t in times], audio_s_per_s=round(streams * seconds / (ms * 1e-3), 1),
                dnn_frames_per_audio_s=sr / hop, kernels=kernels, dsp_ms_total=round(sum(k["ms_per_step"] for k in kernels.values()), 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--streams", type=int, default=128)
    ap.add_argument("--seconds", type=int, default=10)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("geometry_bench needs a CUDA device")
    import bench
    hbm_gbs, _, _, peak_src = bench.peaks()
    res = dict(gpu=gpu_info(), hbm_peak_gbs=hbm_gbs, hbm_peak_source=peak_src, streams=a.streams, seconds=a.seconds,
               steps=a.steps, warmup=a.warmup, model="DeepFilterNet3, seeded random weights", geometries=[])
    for geo in GEOMETRIES:
        r = run_geometry(geo, a.streams, a.seconds, a.steps, a.warmup, hbm_gbs)
        res["geometries"].append(r)
        print(json.dumps({k: r[k] for k in ("sr", "fft_size", "hop_size", "step_ms_median", "audio_s_per_s", "dsp_ms_total")}), flush=True)
    base = res["geometries"][0]["audio_s_per_s"]
    for r in res["geometries"]:
        r["vs_960_480"] = round(r["audio_s_per_s"] / base, 3)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "geometry_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "vs_960_480": {f"{r['sr']}/{r['fft_size']}/{r['hop_size']}": r["vs_960_480"]
                                                        for r in res["geometries"]}}))


if __name__ == "__main__":
    main()
