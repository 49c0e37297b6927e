"""Generate tests/golden/metrics.npz: speech-quality metrics computed by the REFERENCE's own Python code (imported from
$DFB_REFERENCE_ROOT, see ref_harness.py).  Run:  DFB_REFERENCE_ROOT=<reference tree> python oracle/gen_golden_metrics.py

Reference functions (each pair is scored alone, batch size 1, float32 inputs as the reference's callers pass them):
  stoi    df.stoi.stoi(x[None], y[None], fs)                  (df/stoi.py:163-231)
  sisdr   df.evaluation_utils.si_sdr_speechmetrics(x, y)      (df/evaluation_utils.py:599-619, at the input rate)
  ssnr    df.sepm.SNRseg(x16, y16, 16000)                     (df/sepm.py:28-51)
  llr     df.sepm.llr(x16, y16, 16000)                        (df/sepm.py:200-277)
  wss     df.sepm.wss(x16, y16, 16000)                        (df/sepm.py:280-487)
x16 / y16 are the inputs resampled to 16 kHz with df.io.resample, as df.evaluation_utils.CompositeMetric does; at
16 kHz they are the inputs.  `df.sepm` imports `pesq` and `df.evaluation_utils` imports pystoi, librosa and onnx
helpers at module level; none of the functions above uses them, so `pesq` is a stub module and si_sdr_speechmetrics
is taken from the source file by itself.  A result the reference cannot produce (STOI "not enough frames left" leaves
torch.empty garbage; llr returns None) is stored as NaN.

Pairs (key prefix `p<i>_`; `names` lists them):
  asset48      noisy_snr0.wav against clean_freesound_33711.wav, 48 kHz (full files from tests/golden/assets)
  asset16      the same pair resampled to 16 kHz with df.io.resample
  dfn3         the enhance() output of tests/golden/dfnet_DeepFilterNet3.npz (seeded random weights) against its input,
               both channels, 48 kHz
  synthetic pairs at 16 kHz, stored as int16 codes (value = code / 32768) with their seed:
    identical, scaled (0.5 x), silence (0.4 s of zeros before and after 0.8 s of signal), short (800 samples: too short
    for STOI), zero_clean (all-zero clean signal), ragged0..3 (four lengths)
Stored per pair: `<key>_clean`, `<key>_deg` (int16 codes, synthetic pairs only), and the five values in `values`
[n_pairs, 5] (columns stoi, sisdr, ssnr, llr, wss) with the rate in `rates`.
"""
from __future__ import annotations

import ast
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import ref_harness as rh  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
METRICS = ("stoi", "sisdr", "ssnr", "llr", "wss")


def si_sdr_speechmetrics():
    """The reference's function, compiled from df/evaluation_utils.py alone (the module's imports are not available)."""
    path = os.path.join(rh.REF_ROOT, "DeepFilterNet", "df", "evaluation_utils.py")
    tree = ast.parse(open(path).read())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "si_sdr_speechmetrics")
    ns = {"np": np}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), path, "exec"), ns)
    return ns["si_sdr_speechmetrics"]


def synth_pair(seed: int, n: int, snr_db: float = 5.0):
    """Speech-like clean signal (harmonic source with a syllable-rate envelope and formant-like ripple over a noise floor
    26 dB down) and a degraded copy (white + low-passed noise at `snr_db`, slight gain change), quantised to int16 codes."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 16000.0
    f0 = 100.0 + 120.0 * rng.random()
    s = np.zeros(n)
    for h in range(1, 30):
        if f0 * h < 7600:
            s += np.sin(2 * np.pi * f0 * h * t + 2 * np.pi * rng.random()) / h * (1 + np.cos(2 * np.pi * h * f0 / 3000))
    env = 0.05 + np.maximum(0.0, np.sin(2 * np.pi * (3.0 + 2 * rng.random()) * t + 2 * np.pi * rng.random())) ** 2
    s *= env
    s *= 0.1 / max(np.sqrt(np.mean(s ** 2)), 1e-9)
    s += 0.005 * rng.standard_normal(n)  # recording noise floor: keeps the LPC normal equations well conditioned
    noise = rng.standard_normal(n)
    noise = noise + 0.8 * np.concatenate([[0.0], noise[:-1]])
    noise *= np.sqrt(np.mean(s ** 2) / np.mean(noise ** 2)) * 10 ** (-snr_db / 20)
    d = 0.9 * s + noise
    q = lambda v: np.clip(np.round(v * 32768), -32768, 32767).astype(np.int16)  # noqa: E731
    return q(s), q(d)


def main():
    for m in ("pesq",):
        stub = types.ModuleType(m)
        stub.pesq = None
        sys.modules[m] = stub
    rh.import_reference()
    import df.sepm as sepm
    import df.stoi as dstoi
    from df.io import resample
    sisdr = si_sdr_speechmetrics()

    def score(x: np.ndarray, y: np.ndarray, fs: int):
        x = np.ascontiguousarray(x, dtype=np.float32)
        y = np.ascontiguousarray(y, dtype=np.float32)
        xt, yt = torch.from_numpy(x)[None], torch.from_numpy(y)[None]
        # too short for STOI: the reference leaves torch.empty garbage and logs a warning
        x10 = resample(xt, fs, 10000)
        xs, _ = dstoi.remove_silent_frames(x10, resample(yt, fs, 10000), 40, 256, 128)
        st = float(dstoi.stoi(xt, yt, fs)[0]) if xs[0].numel() >= 512 else float("nan")
        sd = float(sisdr(x, y))
        if fs != 16000:
            x16, y16 = resample(xt, fs, 16000)[0].numpy(), resample(yt, fs, 16000)[0].numpy()
        else:
            x16, y16 = x, y
        with np.errstate(all="ignore"):
            ss = float(sepm.SNRseg(x16, y16, 16000))
            ll = sepm.llr(x16, y16, 16000)
            ll = float("nan") if ll is None else float(ll)
            ws = float(sepm.wss(x16, y16, 16000))
        return [st, sd, ss, ll, ws]

    names, rates, values, arrays = [], [], [], {}

    clean = rh.read_wav(os.path.join(GOLD, "assets", "clean_freesound_33711.wav"))[0]
    noisy = rh.read_wav(os.path.join(GOLD, "assets", "noisy_snr0.wav"))[0]
    names.append("asset48"); rates.append(48000); values.append(score(clean, noisy, 48000))
    c16 = resample(torch.from_numpy(clean)[None], 48000, 16000)[0].numpy()
    n16 = resample(torch.from_numpy(noisy)[None], 48000, 16000)[0].numpy()
    names.append("asset16"); rates.append(16000); values.append(score(c16, n16, 16000))

    d3 = np.load(os.path.join(GOLD, "dfnet_DeepFilterNet3.npz"))
    for ch in range(d3["audio"].shape[0]):
        names.append(f"dfn3_{ch}"); rates.append(48000); values.append(score(d3["audio"][ch], d3["enhanced"][ch], 48000))

    c, d = synth_pair(11, 16000)
    synth = {"identical": (c, c.copy()), "scaled": (2 * c, c)}  # |c| < 2^14: 2 c is exact
    c, d = synth_pair(12, 12800)
    z = np.zeros(6400, np.int16)
    synth["silence"] = (np.concatenate([z, c, z]), np.concatenate([z, d, z]))
    c, d = synth_pair(13, 8000)
    synth["short"] = (c[3000:3800], d[3000:3800])
    synth["zero_clean"] = (np.zeros(8000, np.int16), synth_pair(14, 8000)[1])
    for i, n in enumerate((8000, 12000, 16800, 19200)):
        synth[f"ragged{i}"] = synth_pair(20 + i, n, snr_db=float(2 * i))
    for k, (c, d) in synth.items():
        p = len(names)
        arrays[f"p{p}_clean"], arrays[f"p{p}_deg"] = c, d
        names.append(k); rates.append(16000)
        values.append(score(c.astype(np.float32) / 32768, d.astype(np.float32) / 32768, 16000))

    values = np.asarray(values, dtype=np.float64)
    for n, v in zip(names, values):
        print(f"{n:12s} " + " ".join(f"{m}={x:.6f}" for m, x in zip(METRICS, v)))
    out = os.path.join(GOLD, "metrics.npz")
    np.savez_compressed(out, names=np.array(names), rates=np.array(rates, np.int64), values=values,
                        metrics=np.array(METRICS), **arrays)
    print(out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
