"""Speech-quality metrics on the device: STOI, SI-SDR, segmental SNR, LLR and WSS for batches of (clean, degraded)
pairs, with the reference's semantics and names:

    stoi(x, y, fs_source)                 df.stoi.stoi                                 (df/stoi.py:163-231)
    si_sdr(reference, estimate)           df.evaluation_utils.si_sdr_speechmetrics     (df/evaluation_utils.py:599-619)
    ssnr / llr / wss(clean, degraded, fs) df.sepm.SNRseg / llr / wss                   (df/sepm.py:28-51, 200-487)
    evaluate(clean, degraded, sr, ...)    all of them for a batch, one dict of [B] tensors

Every value is computed by the CUDA library (``dfb_metrics`` -> k_stoi_* / k_sisdr / k_sepm_*); there is no CPU
compute path.  Pair b of a padded batch is scored on its first ``lengths[b]`` samples, exactly as if it were scored
alone.  STOI works at 10 kHz and the sepm measures at 16 kHz (inputs are resampled on the device with df.io.resample's
taps), SI-SDR at the input rate.  INTEGRATION.md lists where the results differ from the reference's (NaN where the
reference leaves garbage, returns None or raises).
"""
from __future__ import annotations

from typing import Dict, Iterable, Optional, Sequence, Union

import numpy as np
import torch
from torch import Tensor

from . import _lib
from ._lib import check

METRICS = ("stoi", "sisdr", "ssnr", "llr", "wss")
_BIT = {name: 1 << i for i, name in enumerate(METRICS)}   # DFB_METRIC_* of include/dfb200.h
SAMPLE_RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)

ArrayLike = Union[Tensor, np.ndarray]


def _as_tensor(x) -> Tensor:
    return x if isinstance(x, Tensor) else torch.as_tensor(np.asarray(x))


def _batch(x, name: str):
    """[B, T] float32 tensor (device kept) and the per-row lengths of a tensor / array ([T] or [B, T]) or a list of 1-D
    signals (zero padded to the longest)."""
    if isinstance(x, (list, tuple)):
        rows = [_as_tensor(r) for r in x]
        if not rows or any(r.dim() != 1 for r in rows):
            raise ValueError(f"{name}: a list of 1-D signals is expected")
        T = max(int(r.shape[0]) for r in rows)
        out = torch.zeros((len(rows), T), dtype=torch.float32, device=rows[0].device)
        for i, r in enumerate(rows):
            out[i, :r.shape[0]] = r.to(out.device, torch.float32)
        return out, [int(r.shape[0]) for r in rows]
    t = _as_tensor(x)
    if t.dim() == 1:
        t = t.unsqueeze(0)
    if t.dim() != 2:
        raise ValueError(f"{name}: expected [T] or [B, T], got shape {tuple(t.shape)}")
    return t.to(torch.float32), None


def evaluate(clean, degraded, sr: int, lengths: Optional[Sequence[int]] = None,
             metrics: Iterable[str] = METRICS) -> Dict[str, Tensor]:
    """Scores every pair of a batch: clean / degraded are [B, T] or [T] tensors or arrays (CPU or CUDA) or lists of 1-D
    signals; ``lengths`` (optional, [B]) the valid samples of each row.  Returns {metric: float32 [B]} on the inputs'
    device (CUDA inputs) or on the CPU.  Metrics: "stoi", "sisdr", "ssnr", "llr", "wss"."""
    names = list(metrics)
    bad = [m for m in names if m not in _BIT]
    if bad or not names:
        raise ValueError(f"unknown metrics {bad}; choose from {METRICS}")
    if int(sr) not in SAMPLE_RATES:
        raise ValueError(f"unsupported sample rate {sr}; supported: {SAMPLE_RATES}")
    x, lx = _batch(clean, "clean")
    y, ly = _batch(degraded, "degraded")
    if x.shape != y.shape:
        raise ValueError(f"clean and degraded shapes differ: {tuple(x.shape)} vs {tuple(y.shape)}")
    if lx != ly:
        raise ValueError("clean and degraded lists hold signals of different lengths")
    B, T = x.shape
    if T == 0:
        raise ValueError("empty signals")
    if lengths is None:
        lengths = lx
    lens = None
    if lengths is not None:
        lens = torch.as_tensor(lengths, dtype=torch.int64).cpu().reshape(-1).contiguous()
        if lens.numel() != B:
            raise ValueError(f"lengths has {lens.numel()} entries for a batch of {B}")
        if bool((lens <= 0).any()) or bool((lens > T).any()):
            raise ValueError(f"lengths must lie in [1, {T}]")
    which = 0
    for m in names:
        which |= _BIT[m]
    out_dev = x.device if x.device.type == "cuda" else None
    dev = out_dev if out_dev is not None else torch.device("cuda", torch.cuda.current_device())
    xd = x.to(dev).contiguous()
    yd = y.to(dev).contiguous()
    order = [m for m in METRICS if which & _BIT[m]]
    out = torch.empty((B, len(order)), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(_lib.lib().dfb_metrics(dev.index, xd.data_ptr(), yd.data_ptr(), None if lens is None else lens.data_ptr(),
                                     B, T, int(sr), which, out.data_ptr(), stream))
    if out_dev is None:
        out = out.cpu()
    return {m: out[:, order.index(m)] for m in names}


def stoi(x: Tensor, y: Tensor, fs_source: int) -> Tensor:
    """df.stoi.stoi: x (target) and y (degraded) [batch, samples] -> STOI [batch] in x's dtype and device.  NaN for an
    utterance with fewer than 512 samples at 10 kHz after the silent-frame removal (the reference leaves the entry
    uninitialised)."""
    assert x.shape == y.shape, "Inputs must have the same shape"
    assert x.dim() == 2, f"Expected input shape of [batch_size, samples], but got {x.shape}"
    return evaluate(x, y, fs_source, metrics=("stoi",))["stoi"].to(x.device, x.dtype)


def si_sdr(reference: ArrayLike, estimate: ArrayLike) -> float:
    """df.evaluation_utils.si_sdr_speechmetrics for one pair (float32 semantics, eps = float32 eps), in dB."""
    r, e = _as_tensor(reference).reshape(-1), _as_tensor(estimate).reshape(-1)
    if r.shape != e.shape:
        raise ValueError(f"shapes differ: {tuple(r.shape)} vs {tuple(e.shape)}")
    # any supported rate: SI-SDR is computed at the input rate without resampling
    return float(evaluate(r, e, 16000, metrics=("sisdr",))["sisdr"][0])


def _sepm(metric: str, clean: ArrayLike, degraded: ArrayLike, fs: int) -> float:
    if int(fs) != 16000:
        raise ValueError(f"{metric}: the sepm measures are computed at 16 kHz (fs = {fs}); resample first, or use "
                         "evaluate(), which resamples like CompositeMetric")
    c, d = _as_tensor(clean).reshape(-1), _as_tensor(degraded).reshape(-1)
    if c.shape != d.shape:
        raise ValueError("The two signals do not match!")
    return float(evaluate(c, d, 16000, metrics=(metric,))[metric][0])


def ssnr(clean: ArrayLike, degraded: ArrayLike, fs: int) -> float:
    """df.sepm.SNRseg (30 ms hann frames, 75 % overlap, clamped to [-10, 35] dB, last frame dropped) at 16 kHz."""
    return _sepm("ssnr", clean, degraded, fs)


def llr(clean: ArrayLike, degraded: ArrayLike, fs: int) -> float:
    """df.sepm.llr (LPC order 16, mean of the 95 % smallest frame distances) at 16 kHz; NaN where the reference returns
    None (no frame)."""
    return _sepm("llr", clean, degraded, fs)


def wss(clean: ArrayLike, degraded: ArrayLike, fs: int) -> float:
    """df.sepm.wss (25 critical bands, 1024-point FFT, mean of the 95 % smallest frame distances) at 16 kHz."""
    return _sepm("wss", clean, degraded, fs)
