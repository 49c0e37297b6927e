#!/usr/bin/env python
"""bench.py -- 48 kHz audio-seconds enhanced per wall-second (batched enhance()), BASELINE.json's
metric, on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2..5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the whole enhancement path (pad -> STFT -> features -> DNN -> mask + deep
filter -> ISTFT -> crop) over one batch of synthetic noisy streams.

Headline workload at every N (the JSON line's value / e2e / roofline): BASELINE.json configs[1] per GPU --
DeepFilterNet3, 128 streams x 10 s @ 48 kHz -- i.e. weak scaling, streams sharded across ranks with no
data-path collective (SURVEY.md 8e).  The other BASELINE configs (numbered as in SURVEY.md 8: cfg3 =
DeepFilterNet2 512 x 10 s, cfg4 = DeepFilterNet3_ll 256 streams per GPU, cfg5 = DeepFilterNet3 512 x 30 s per GPU)
are measured with a few steps each and attached under `extra.configs`, each with its own value / e2e / roofline /
parity; `--config N` makes one of them the headline instead.

  value   : whole-job audio-s/s with the noisy batch already resident in HBM (device-pointer C ABI), timed WITHOUT
            the per-kernel event profiler
  e2e     : the same through the reference-facing call enhance(model, df_state, cpu_tensor) with pinned HOST
            buffers, H2D / D2H copies inside the timed region
  roofline: dominant kernel, CUDA-event timed on its launching stream in a separate, profiled pass of the same
            steps; `traffic` from the ncu capture committed under profiles/ (same batch)
  parity  : RMS of 4 streams of the timed batch's output against the CPU oracle (outside the timed region)
  cpu_baseline: the CPU oracle port (C DSP + torch-CPU DNN) on this box's host cores, bounded sample

--dump-outputs DIR writes the headline's enhanced audio of the last timed step to DIR/enhanced.npy (float32
[streams, samples]): a fixed, seeded sample of the batch's streams (all of them when they fit DUMP_BYTES), so that two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the tree may be read-only; nothing is written into it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SR = 48000
# SURVEY.md 8 numbering: (model, streams per GPU, seconds, GPUs the config is quoted on)
CONFIGS = {
    2: ("DeepFilterNet3", 128, 10, 1),
    3: ("DeepFilterNet2", 512, 10, 1),
    4: ("DeepFilterNet3_ll", 256, 10, 4),
    5: ("DeepFilterNet3", 512, 30, 8),
    6: ("DeepFilterNet", 128, 10, 1),     # SURVEY.md 8f-2 ("next" row): DeepFilterNet v1 at configs[1]'s shape -- not a BASELINE config
}
BASELINE_NAME = {2: "BASELINE.json configs[1]", 3: "BASELINE.json configs[2]", 4: "BASELINE.json configs[3] (per-GPU shard)",
                 5: "BASELINE.json configs[4] (per-GPU shard)", 6: "SURVEY.md 8f-2, DeepFilterNet v1; not a BASELINE config"}
# Algorithmic DNN flops per frame per stream (SURVEY.md 8d / BASELINE.md 2)
FLOP_PER_FRAME = {"DeepFilterNet3": 6_614_784, "DeepFilterNet2": 6_956_800, "DeepFilterNet3_ll": 21_846_784}
DTYPE = "f32 (bf16x3 tensor-core contractions, fp32 accumulate; DSP and gates IEEE fp32)"
PARITY_TOL = 1e-4  # BASELINE.json north_star: RMS vs the reference path
DUMP_BYTES = 48 << 20  # --dump-outputs budget


def kernel_model(cfg, g: dict) -> dict:
    """Algorithmic bytes / flops per frame per stream of every kernel (DESIGN.md section 4), from the model's
    hyper-parameters.  name -> (bound, amount, "bytes" | "flops")."""
    E, Fd, O2 = cfg.nb_erb, cfg.nb_df, 2 * cfg.df_order
    H, Hd = cfg.emb_hidden_dim, cfg.df_hidden_dim
    ED = E // 4 * 64
    emb_in = 2 * ED if cfg.enc_concat else ED
    emb = H if cfg.model == "deepfilternet2" else ED
    enc_l, erb_l, df_l = g["enc_gru_layers"], g["erb_gru_layers"], g["df_gru_layers"]
    rec = 2 * 3 * (H * H * (enc_l + erb_l) + Hd * Hd * df_l)        # W_hh h, all layers
    if cfg.model == "deepfilternet":                                 # GroupedGRU: block-diagonal, 1 / G of the dense product
        rec //= cfg.gru_groups
    proj = rec                                                       # W_ih x: same shapes (inputs are H wide)
    gl = gl_bytes = 0
    for (i, o, grp) in ((Fd // 2 * 64, ED, g["g_df_fc_emb"]), (emb_in, H, g["g_enc_in"]), (H, ED, g["g_enc_out"]),
                        (emb, H, g["g_erb_in"]), (H, ED, g["g_erb_out"]), (emb, Hd, g["g_df_in"]),
                        (emb, Hd, g["g_df_skip"]), (Hd, Fd * O2, g["g_df_out"])):
        if grp:
            gl += 2 * i * o // grp
            gl_bytes += 4 * (i + o)                                  # fp32 row in, fp32 row out
    rows = (Fd + Fd // 2) + (E + E // 2) + (E // 2 + E // 4) + (E // 4 + E // 4) + 3 * (E // 4) + (E // 4 + E // 4 + E // 2) \
        + (E // 2 + E // 2 + E)
    return {
        "k_analysis": ("hbm", 1920 + 8 * cfg.freq_bins + 4 * E, "bytes"),
        "k_feat_norm": ("hbm", 2 * (4 * E + 8 * Fd), "bytes"),
        "k_apply_synthesis": ("hbm", 8 * cfg.freq_bins + 4 * E + 4 * Fd * O2 + 1920, "bytes"),
        "k_gru_tc": ("tensor", rec, "flops"), "k_gru": ("tensor", rec, "flops"), "k_gru_tc512": ("tensor", rec, "flops"),
        "k_gemm_bf16x3[gru_proj]": ("tensor", proj, "flops"), "k_grouped_linear[gru_proj]": ("tensor", proj, "flops"),
        "k_grouped_linear": ("tensor", gl, "flops"),
        # grouped linears on tcgen05: 2 * I * O / G flops per row are ~20 flop/B, far under the ridge -> HBM bound
        "k_gl_bx": ("hbm", gl_bytes, "bytes"),
        "k_dwpw": ("tensor", 2 * 64 * 64 * (Fd // 2 + E // 2 + E // 4 + E // 4 + E // 4 + E // 2 + E), "flops"),
        # fused depthwise -> tcgen05 1x1: rows read (input + pathway) + rows written, 256 B each, over the 7 separable blocks
        "k_dwpw_bx": ("hbm", 256 * rows, "bytes"),
        "k_conv_in[df_conv0]": ("hbm", Fd * 8 + Fd * 256, "bytes"),
        "k_conv_in[erb_conv0]": ("hbm", 4 * E + E * 256, "bytes"),
        "k_df_convp": ("hbm", Fd * 256 + Fd * 4 * O2, "bytes"),
        "k_df_convp_tc": ("hbm", Fd * 256 + Fd * 4 * O2, "bytes"),
        "k_mask_out": ("hbm", 2 * E * 256 + 4 * E, "bytes"),
        # DeepFilterNet v1 only: re-ordering passes (read + write one 2 KB row each, 3 KB for the c1 gather) and the 1x1 pathway conv
        "k_gather_sum": ("hbm", 2 * 4 * (Fd // 2 * 64) + 4 * 3 * 4 * H + 6 * 4 * H, "bytes"),
        "k_convp_v1": ("hbm", Fd * 256 + 2 * Fd * 4 * O2, "bytes"),
    }


def per_gpu_report(rows, knames, streams: int, seconds: int):
    """rows[r] = [device ms/step, end-to-end ms/step, roofline fraction, avg launch ms, index into knames (or -1), share of
    the step] of rank r -> the `per_gpu` list of the JSON line.  Never raises (the line must not depend on it)."""
    try:
        num = lambda x: None if x != x else x   # NaN -> null
        return [{"rank": r, "ms_per_step": row[0], "value": streams * seconds / (row[0] / 1e3),
                 "e2e_ms_per_step": row[1], "e2e_value": streams * seconds / (row[1] / 1e3),
                 "roofline_kernel": knames[int(row[4])] if row[4] >= 0 else None, "roofline_frac": num(row[2]),
                 "avg_launch_ms": num(row[3]), "share_of_step": num(row[5])} for r, row in enumerate(rows)]
    except Exception as e:
        return [{"error": f"{type(e).__name__}: {e}"}]


def ncu_traffic(model_name: str, streams: int, seconds: int):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) per kernel from the committed
    `ncu --set full` capture of exactly this workload (profiles/r02_ncu_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.isfile(p):
        return None, None
    d = json.load(open(p))
    key = f"{model_name}:{streams}x{seconds}"
    return d.get(key), d.get("_source")


def model_config(name: str):
    from deepfilternet_b200.config import ModelConfig, load_config
    p = os.path.join(ROOT, "models", "_ref", name, "config.ini")
    if os.path.isfile(p):
        return load_config(p, env={})
    base = dict(conv_ch=64, df_pathway_kernel_size_t=5)
    if name == "DeepFilterNet3":
        return ModelConfig(model="deepfilternet3", conv_lookahead=2, df_lookahead=2, emb_num_layers=3, df_num_layers=2,
                           lin_groups=16, enc_lin_groups=32, df_gru_skip="groupedlinear", **base)
    if name == "DeepFilterNet2":
        return ModelConfig(model="deepfilternet2", conv_lookahead=2, df_lookahead=2, emb_num_layers=3, df_num_layers=2,
                           lin_groups=8, enc_lin_groups=8, enc_concat=True, **base)
    if name == "DeepFilterNet3_ll":
        return ModelConfig(model="deepfilternet3", conv_lookahead=0, df_lookahead=0, conv_kernel=(2, 3), emb_hidden_dim=512,
                           df_hidden_dim=512, emb_num_layers=3, df_num_layers=3, lin_groups=16, enc_lin_groups=16,
                           df_gru_skip="groupedlinear", **base)
    if name == "DeepFilterNet":
        return ModelConfig(model="deepfilternet", conv_lookahead=2, df_lookahead=1, conv_ch=64, conv_kernel=(2, 3), convt_kernel=(2, 3),
                           conv_kernel_inp=(2, 3), conv_k_enc=2, conv_k_dec=2, emb_hidden_dim=512, df_hidden_dim=512, emb_num_layers=3,
                           df_num_layers=2, gru_groups=8, lin_groups=8, enc_lin_groups=8, group_shuffle=True, dfop_method="real_unfold")
    raise SystemExit(f"no config for {name}")


def load_weights(name: str, cfg):
    """Pretrained weights when models/_ref travelled with the snapshot, else random-init weights of
    the same architecture (there is no network for checkpoints)."""
    from deepfilternet_b200.model import find_checkpoint, load_state_dict_file
    from deepfilternet_b200.weights import random_state_dict
    d = os.path.join(ROOT, "models", "_ref", name)
    if os.path.isdir(os.path.join(d, "checkpoints")):
        p, _ = find_checkpoint(os.path.join(d, "checkpoints"))
        if p:
            return load_state_dict_file(p), "pretrained"
    if os.path.isfile(os.path.join(d, "enc.onnx")):
        from deepfilternet_b200.onnx_import import state_dict_from_onnx_dir
        sd = state_dict_from_onnx_dir(d, cfg)
        if sd is not None:
            return sd, "pretrained (ONNX transplant)"
    return random_state_dict(cfg, seed=0), "random-init"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms.  The sampler is started before the warm-up (the tool
    needs ~100 ms to come up and the timed region of 10 steps is only ~140 ms long); `window()` brackets the timed
    regions with wall-clock stamps and only samples inside the window are reported."""

    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.t0, self.t1 = index, None, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def window_begin(self):
        self.t0 = time.time()

    def window_end(self):
        self.t1 = time.time()

    @staticmethod
    def parse(lines, t0=None, t1=None) -> dict:
        def collect(filtered):
            sm, mx, reasons = [], None, set()
            for ts, ln in lines:
                if filtered and t0 is not None and t1 is not None and not (t0 <= ts <= t1 + 0.06):
                    continue
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 10:
                    continue
                try:
                    sm.append(float(f[2])); mx = float(f[3])
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons
        sm, mx, reasons = collect(True)
        scope = "timed regions"
        if not sm:  # nothing landed inside the window: fall back to everything sampled under load (warm-up included)
            sm, mx, reasons = collect(False)
            scope = "warm-up + timed regions"
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "scope": scope}

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        return self.parse(self.lines, self.t0, self.t1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def host_threads() -> int:
    """Host cores this process may actually use (affinity mask and cgroup CPU quota respected)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return max(1, n)


def bind_to_gpu_numa_node(dev_index: int):
    """Pin this rank's host threads (and, by first touch, its pinned staging buffers) to the NUMA node of its GPU:
    at N = 8 the eight ranks' H2D / D2H traffic otherwise crosses the inter-socket link (SCALE_r01: e2e efficiency
    0.925 while the device-timed efficiency was 1.00).  Returns a description for the JSON line, or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev_index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"gpu": dev_index, "pci": bdf, "numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None


def cpu_reference_run(cfg, sd, seconds: int, steps: int, warmup: int, threads: int, budget_s: float):
    """The reference's CPU path restated (oracle/): C DSP + torch-CPU DNN with `threads` host
    threads.  The per-step sample (whole streams of the same synthetic workload) is sized from
    a 1-stream probe so that the run stays near `budget_s` seconds."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dfnet_oracle
    import libdf_oracle
    from tests_common import synth_audio
    libdf_oracle.build()
    torch.set_num_threads(threads)
    cfgd = cfg.as_dict()
    probe = synth_audio(1, SR * seconds, seed=1234)
    dfnet_oracle.enhance(sd, cfgd, probe[:, : SR * 2])
    t0 = time.perf_counter()
    dfnet_oracle.enhance(sd, cfgd, probe)
    t_probe = time.perf_counter() - t0
    streams = int(max(1, min(32, budget_s / max(steps + warmup, 1) / max(t_probe, 1e-3))))
    audio = synth_audio(streams, SR * seconds, seed=1234)
    for _ in range(warmup):
        dfnet_oracle.enhance(sd, cfgd, audio)
    t0 = time.perf_counter()
    for _ in range(steps):
        dfnet_oracle.enhance(sd, cfgd, audio)
    dt = time.perf_counter() - t0
    return streams * seconds * steps / dt, dt / steps, streams


def dump_sample(out):
    """A fixed, seeded sample of the streams of `out` [streams, T] (and a prefix of each when one stream alone exceeds
    DUMP_BYTES), copied to the host as float32."""
    import torch
    streams, T = out.shape
    cols = min(T, DUMP_BYTES // 4)
    k = max(1, min(streams, DUMP_BYTES // (4 * cols)))
    rows = torch.randperm(streams, generator=torch.Generator().manual_seed(0))[:k].sort().values
    return out[rows.to(out.device), :cols].float().cpu()


def ctypes_buf():
    import ctypes
    return ctypes.create_string_buffer(1 << 16)


class Ctx:
    """Per-process context shared by all measured configs."""

    def __init__(self, a):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.n_gpus = a.gpus
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
        self.dev = self.local_rank % torch.cuda.device_count()
        torch.cuda.set_device(self.dev)
        self.numa = bind_to_gpu_numa_node(self.dev)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.dev))

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def gather_rows(self, vals):
        """[world][len(vals)]: every rank's figures on every rank (per-GPU report; one all_gather, outside the timed regions)."""
        from deepfilternet_b200.sharding import gather_rank_rows
        return gather_rank_rows(vals, device=f"cuda:{self.dev}")

    def max_over_ranks(self, vals):
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=f"cuda:{self.dev}")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


def measure(ctx: Ctx, cfg_id: int, model_name: str, streams: int, seconds: int, steps: int, warmup: int,
            roofline_kernel=None, parity_streams: int = 4, clocks=None, dump: bool = False):
    """One workload on this process' GPU (all ranks run it in lock step): returns the JSON fields."""
    import torch
    from deepfilternet_b200 import DfNet, _lib, enhance, enhance_device, libdf
    from tests_common import synth_audio
    L = _lib.lib()
    dev = ctx.dev
    cfg = model_config(model_name)
    sd, weights_kind = load_weights(model_name, cfg)
    st = libdf.DF(cfg.sr, cfg.fft_size, cfg.hop_size, cfg.nb_erb, cfg.min_nb_erb_freqs, device=dev)
    model = DfNet(cfg, sd, st, device=dev)
    frames = (SR * seconds + cfg.fft_size) // cfg.hop_size
    T = SR * seconds
    # this rank's shard of the global batch: streams [rank * streams, (rank + 1) * streams)
    audio = synth_audio(streams, T, seed=1234 + ctx.rank * streams, device=f"cuda:{dev}")
    out = torch.empty_like(audio)
    host_in = torch.empty(audio.shape, dtype=torch.float32, pin_memory=True)   # first touch on the GPU's NUMA node
    host_in.copy_(audio)
    host_out = torch.empty(audio.shape, dtype=torch.float32, pin_memory=True)
    # ---------------- device-resident timing (un-instrumented)
    for _ in range(warmup):
        enhance_device(model, st, audio, out=out)
    ctx.sync_all()
    if clocks:
        clocks.window_begin()
    launches0 = L.dfb_kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.sync_all()
    ev0.record()
    for _ in range(steps):
        enhance_device(model, st, audio, out=out)
    ev1.record()
    ctx.sync_all()
    ms = ev0.elapsed_time(ev1)
    launches = int(L.dfb_kernel_launches() - launches0)
    dumped = dump_sample(out) if dump else None   # the last timed step's output, before later passes reuse `out`
    # ---------------- end to end through the public API with host buffers
    for _ in range(2):
        enhance(model, st, host_in, out=host_out)
    ctx.sync_all()
    t0 = time.perf_counter()
    for _ in range(steps):
        enhance(model, st, host_in, out=host_out)   # synchronous: returns with the result on the host
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if clocks:
        clocks.window_end()
    # ---------------- profiled pass (per-kernel CUDA events on the launching streams) for the roofline
    L.dfb_profile_report(ctypes_buf(), 1 << 16)  # drain
    L.dfb_profile_enable(1, None)
    psteps = min(steps, 5)
    for _ in range(psteps):
        enhance_device(model, st, audio, out=out)
    torch.cuda.synchronize()
    buf = ctypes_buf()
    L.dfb_profile_report(buf, 1 << 16)
    L.dfb_profile_enable(0, None)
    prof = {}
    for ln in buf.value.decode().splitlines():
        name, cnt, tot = ln.rsplit(" ", 2)
        prof[name] = (int(cnt), float(tot))
    t_dev, t_e2e = ctx.max_over_ranks([ms / 1e3, e2e_s])
    # ---------------- parity gate: a few streams of the timed batch against the CPU oracle
    parity = None
    if ctx.rank == 0 and parity_streams > 0:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import dfnet1_oracle
        import dfnet_oracle
        rows = sorted({0, 1, streams // 2, streams - 1})[:parity_streams]
        got_dev = out[rows].cpu()
        got_e2e = host_out[rows]
        if cfg.model == "deepfilternet":
            ref = dfnet1_oracle.enhance(sd, dict(dfnet1_oracle.DEFAULTS_DFN1), audio[rows].cpu())
        else:
            ref = dfnet_oracle.enhance(sd, cfg.as_dict(), audio[rows].cpu())
        rms_dev = float((got_dev - ref).double().pow(2).mean().sqrt())
        rms_e2e = float((got_e2e - ref).double().pow(2).mean().sqrt())
        parity = {"streams": rows, "rms_vs_oracle_device": rms_dev, "rms_vs_oracle_e2e": rms_e2e, "tol": PARITY_TOL,
                  "ok": bool(rms_dev <= PARITY_TOL and rms_e2e <= PARITY_TOL and torch.isfinite(out).all().item())}
    n_gpus = ctx.n_gpus
    total_audio_s = streams * n_gpus * seconds * steps
    value, e2e = total_audio_s / t_dev, total_audio_s / t_e2e
    hbm, tf_burst, tf_sust, peak_src = peaks()
    km = kernel_model(cfg, model._derived)
    total_prof_ms = sum(v[1] for v in prof.values()) or 1.0
    kname = roofline_kernel or max(prof, key=lambda k: prof[k][1])
    cnt, tot_ms = prof.get(kname, (0, 0.0))
    bound, per_frame, kind = km.get(kname.split("[")[0] if kname not in km else kname, ("hbm", 0, "bytes"))
    frames_per_step = streams * frames
    launches_per_step = cnt / psteps if psteps else 0
    avg_launch_s = (tot_ms / 1e3) / cnt if cnt else float("nan")
    per_launch = per_frame * frames_per_step / launches_per_step if launches_per_step else 0.0
    if kind == "bytes":
        achieved, peak, unit = per_launch / avg_launch_s / 1e9, hbm, "GB/s"
    else:
        achieved, peak, unit = per_launch / avg_launch_s / 1e12, tf_sust, "TFLOP/s"
    traffic_tbl, traffic_src = ncu_traffic(model_name, streams, seconds)

    def frac_of(k):
        c, t = prof[k]
        b, pf, kd = km.get(k, km.get(k.split("[")[0], ("hbm", 0, "bytes")))
        if not c or not pf:
            return None
        rate = pf * frames_per_step * psteps / (t / 1e3)
        return round(rate / 1e9 / hbm, 4) if kd == "bytes" else round(rate / 1e12 / tf_sust, 4)

    roofline = {"kernel": kname, "bound": bound, "achieved": achieved, "peak": peak, "unit": unit,
                "frac": achieved / peak if peak else None,
                "traffic": (traffic_tbl or {}).get(kname), "traffic_source": traffic_src, "peak_source": peak_src,
                "launches_per_step": launches_per_step, "avg_launch_ms": avg_launch_s * 1e3,
                "share_of_step": tot_ms / total_prof_ms,
                "kernel_ms_per_step": {k: round(v[1] / psteps, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])},
                "kernel_frac_of_peak": {k: frac_of(k) for k in sorted(prof, key=lambda k: -prof[k][1])},
                "end_to_end_tensor_frac": (value * 100 * FLOP_PER_FRAME.get(model_name, 0) / n_gpus) / (tf_sust * 1e12),
                "end_to_end_hbm_frac_21264B": (value * 100 * 21264 / n_gpus) / (hbm * 1e9)}
    # per-GPU report (SURVEY.md 8e): each rank's own device / end-to-end step time and the roofline fraction of ITS dominant
    # kernel, gathered on every rank; `value` above is the aggregate over ranks at the slowest rank's time
    knames = sorted(km)
    own = [ms / steps, e2e_s * 1e3 / steps, (achieved / peak) if peak else float("nan"), avg_launch_s * 1e3,
           float(knames.index(kname.split("[")[0] if kname not in km else kname)) if (kname in km or kname.split("[")[0] in km) else -1.0,
           tot_ms / total_prof_ms]
    per_gpu = per_gpu_report(ctx.gather_rows(own), knames, streams, seconds)
    workload = (f"{model_name}, batch={streams} x {seconds} s 48 kHz synthetic noisy streams per GPU "
                f"({BASELINE_NAME.get(cfg_id, 'custom')}), pad=True, {frames} frames/stream")
    res = {"cfg": cfg_id, "workload": workload, "model": model_name, "streams_per_gpu": streams, "seconds": seconds,
           "frames_per_stream": frames, "global_streams": streams * n_gpus, "weights": weights_kind,
           "value": value, "unit": "audio-s/s", "ms_per_step": t_dev * 1e3 / steps, "steps": steps, "warmup": warmup,
           "gpu_launches": launches,
           "e2e": {"value": e2e, "unit": "audio-s/s", "h2d_bytes_per_step": int(host_in.numel() * 4),
                   "d2h_bytes_per_step": int(host_out.numel() * 4), "ms_per_step": t_e2e * 1e3 / steps},
           "roofline": roofline, "per_gpu": per_gpu, "parity": parity, "workspace_bytes": model.workspace_bytes()}
    if dumped is not None:
        res["dumped"] = dumped
    # RTF at batch = 1 (BASELINE.json metric, second half): one stream, device resident and end to end
    a1 = audio[:1].contiguous()
    o1 = torch.empty_like(a1)
    h1, ho1 = host_in[:1].contiguous().pin_memory(), torch.empty((1, T), dtype=torch.float32, pin_memory=True)
    for _ in range(3):
        enhance_device(model, st, a1, out=o1)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(5):
        enhance_device(model, st, a1, out=o1)
    ev1.record()
    torch.cuda.synchronize()
    res["rtf_batch1"] = (ev0.elapsed_time(ev1) / 5 / 1e3) / seconds
    enhance(model, st, h1, out=ho1)
    t0 = time.perf_counter()
    for _ in range(5):
        enhance(model, st, h1, out=ho1)
    res["rtf_batch1_e2e"] = ((time.perf_counter() - t0) / 5) / seconds
    res["rtf_note"] = "rtf_batch1: device resident (CUDA events); rtf_batch1_e2e: host tensor in, host tensor out"
    del model, st, audio, out, host_in, host_out
    torch.cuda.empty_cache()
    return res, cfg, sd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="headline workload (SURVEY.md 8 numbering)")
    ap.add_argument("--model", default=None)
    ap.add_argument("--streams", type=int, default=None, help="streams per GPU")
    ap.add_argument("--seconds", type=int, default=None)
    ap.add_argument("--extra", default=None, help="comma list of extra configs (default: 3,4,5,6 at N=1; 4 at N=4; 5 at N=8; 'none')")
    ap.add_argument("--roofline-kernel", default=None, help="kernel to report (default: the one with most time)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the headline's output of the last timed step (a fixed, seeded sample of streams) as DIR/enhanced.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    n_gpus = a.gpus
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    model_name, streams, seconds, _ = CONFIGS[a.config]
    model_name = a.model or model_name
    streams = a.streams or streams
    seconds = a.seconds or seconds
    cfg_id = a.config if (a.model is None and a.streams is None and a.seconds is None) else 0
    threads = host_threads()

    if a.impl == "reference":
        if rank != 0:
            return
        cfg = model_config(model_name)
        sd, weights_kind = load_weights(model_name, cfg)
        frames = (SR * seconds + cfg.fft_size) // cfg.hop_size
        v, s_per_step, sample_streams = cpu_reference_run(cfg, sd, seconds, a.steps, min(a.warmup, 1), threads, budget_s=90.0)
        sample = (f"{sample_streams} of the {streams} streams x {seconds} s per step (CPU oracle port: "
                  f"C libDF restatement + torch-CPU DfNet, {threads} host threads)")
        line = {"impl": "reference", "metric": "48kHz audio-sec/sec (batched enhance)", "value": v,
                "unit": "audio-s/s", "n_gpus": n_gpus, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"{model_name}, batch={streams} x {seconds} s 48 kHz synthetic noisy streams per GPU "
                                       f"({BASELINE_NAME.get(cfg_id, 'custom')}), pad=True, {frames} frames/stream",
                           "streams_per_gpu": streams, "seconds": seconds, "frames_per_stream": frames,
                           "reference_sample": sample, "weights": weights_kind,
                           "note": "a rate: the CPU arm times a bounded sample of the batch, one process at every N"},
                "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": threads, "kind": "port", "sample": sample},
                "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    ctx = Ctx(a)
    clocks = ClockSampler(ctx.dev)
    clocks.start()
    head, cfg, sd = measure(ctx, cfg_id, model_name, streams, seconds, a.steps, a.warmup, a.roofline_kernel, clocks=clocks,
                            dump=bool(a.dump_outputs) and ctx.rank == 0)
    clk = clocks.stop()
    if "dumped" in head:
        import numpy as np
        os.makedirs(a.dump_outputs, exist_ok=True)
        np.save(os.path.join(a.dump_outputs, "enhanced.npy"), head.pop("dumped").numpy())
    if a.extra is None:
        extra_ids = {1: [3, 4, 5, 6], 4: [4], 8: [5]}.get(n_gpus, [])
        extra_ids = [i for i in extra_ids if i != cfg_id] if cfg_id == 2 else []
    else:
        extra_ids = [] if a.extra in ("", "none") else [int(x) for x in a.extra.split(",")]
    extras = []
    for cid in extra_ids:
        mn, s_, sec_, quoted = CONFIGS[cid]
        try:
            r, _, _ = measure(ctx, cid, mn, s_, sec_, steps=3, warmup=3, parity_streams=2)
            r["quoted_on_gpus"] = quoted
            extras.append(r)
        except Exception as e:  # an extra config must never take the headline line down with it
            extras.append({"cfg": cid, "error": f"{type(e).__name__}: {e}"})
    if ctx.rank != 0:
        if ctx.world > 1:
            ctx.dist.destroy_process_group()
        return
    config = {"workload": head["workload"], "streams_per_gpu": streams, "seconds": seconds,
              "frames_per_stream": head["frames_per_stream"], "global_streams": streams * n_gpus,
              "parallelism": f"stream-sharded x{n_gpus}, no collective", "weights": head["weights"],
              "l2": f"inputs larger than L2 (batch audio {streams * seconds * SR * 4 / 1e6:.0f} MB + "
                    f"{head['workspace_bytes'] / 1e9:.1f} GB of workspace per step)",
              "numa_binding": ctx.numa}
    line = {"metric": "48kHz audio-sec/sec (batched enhance)", "value": head["value"], "unit": "audio-s/s",
            "n_gpus": n_gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": config, "clocks": clk, "gpu_launches": head["gpu_launches"], "e2e": head["e2e"],
            "rtf_batch1": head["rtf_batch1"], "rtf_batch1_e2e": head["rtf_batch1_e2e"], "rtf_note": head["rtf_note"],
            "roofline": head["roofline"], "per_gpu": head["per_gpu"], "parity": head["parity"], "extra": {"configs": extras}}
    if n_gpus == 1 and not a.no_cpu_baseline:
        v, s_step, ns = cpu_reference_run(cfg, sd, seconds, 2, 0, threads, budget_s=25.0)
        line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": threads, "kind": "port",
                                "sample": f"2 steps of {ns} of the {streams} streams x {seconds} s (CPU oracle port: C libDF "
                                          f"restatement + torch-CPU DfNet, {threads} threads), {s_step:.2f} s/step"}
    print(json.dumps(line))
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
