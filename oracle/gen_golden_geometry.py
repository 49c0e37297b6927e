"""Generate the golden fixtures of two STFT geometries other than 960 / 480 by running the REFERENCE's own Python
modules (imported from $DFB_REFERENCE_ROOT, see ref_harness.py) with the seeded random DeepFilterNet3 weights of
oracle/random_models.py.  Run:  DFB_REFERENCE_ROOT=<reference tree> python oracle/gen_golden_geometry.py

The two models are the shipped DeepFilterNet3 config.ini with only sr / fft_size / hop_size changed:
  DeepFilterNet3_16k   16000 / 320 / 160   (F = 161)
  DeepFilterNet3_5ms   48000 / 480 / 240   (F = 241)
The DNN weights depend on nb_erb / nb_df only, so both models carry the DeepFilterNet3 weights.

Outputs (small; committed):
  tests/golden/models/<name>/config.ini   the derived configs
  tests/golden/dfnet_<name>.npz           reference DfNet.forward / enhance() outputs on a 0.2 s two-channel excerpt of
                                          noisy_snr0.wav (resampled to 16 kHz with df.io.resample for the 16 kHz model);
                                          same keys as tests/golden/dfnet_DeepFilterNet3.npz
"""
from __future__ import annotations

import os
import re
import shutil
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import random_models  # noqa: E402
import ref_harness as rh  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
GEOMETRIES = {"DeepFilterNet3_16k": (16000, 320, 160), "DeepFilterNet3_5ms": (48000, 480, 240)}


def derive_config(src_ini: str, sr: int, fft_size: int, hop_size: int) -> str:
    """The text of `src_ini` with the [df] section's sr / fft_size / hop_size replaced."""
    text = open(src_ini).read()
    for key, val in (("sr", sr), ("fft_size", fft_size), ("hop_size", hop_size)):
        text, n = re.subn(rf"(?m)^{key} = .*$", f"{key} = {val}", text, count=1)
        assert n == 1, key
    return text


def excerpt(noisy: torch.Tensor) -> torch.Tensor:
    """0.2 s at 48 kHz, two channels (second = time-shifted, attenuated), as oracle/gen_golden.py."""
    return torch.stack([noisy[0, 96000:105600], 0.5 * noisy[0, 130000:139600]])


def main():
    rh.import_reference()
    from df.enhance import df_features, enhance, init_df
    from df.io import resample
    import torch.nn.functional as F

    noisy = torch.from_numpy(rh.read_wav(os.path.join(GOLD, "assets", "noisy_snr0.wav")))
    sd = random_models.state_dict("DeepFilterNet3")
    tmp = tempfile.mkdtemp()
    for name, (sr, fft, hop) in GEOMETRIES.items():
        cfg_dir = os.path.join(GOLD, "models", name)
        os.makedirs(cfg_dir, exist_ok=True)
        with open(os.path.join(cfg_dir, "config.ini"), "w") as f:
            f.write(derive_config(os.path.join(random_models.CONFIGS, "DeepFilterNet3", "config.ini"), sr, fft, hop))
        d = os.path.join(tmp, name)
        os.makedirs(os.path.join(d, "checkpoints"))
        shutil.copyfile(os.path.join(cfg_dir, "config.ini"), os.path.join(d, "config.ini"))
        torch.save(sd, os.path.join(d, "checkpoints", random_models.CHECKPOINTS["DeepFilterNet3"]))
        model, st, _, _ = init_df(d, log_file=None, log_level="ERROR", epoch="none")
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected and set(missing) <= {"erb_fb", "mask.erb_inv_fb"}, (missing, unexpected)
        model.eval()
        assert (st.sr(), st.fft_size(), st.hop_size()) == (sr, fft, hop)
        x = excerpt(noisy)
        if sr != 48000:
            x = resample(x, 48000, sr).contiguous()
        y = enhance(model, st, x, pad=True)
        xa = F.pad(x, (0, st.fft_size()))
        spec, ef, sf = df_features(xa, st, 96)
        with torch.no_grad():
            spec_e, m, lsnr, c = model(spec.clone(), ef, sf)
        arrays = dict(audio=x.numpy(), enhanced=y.numpy(), spec=spec.numpy(), feat_erb=ef.numpy(), feat_spec=sf.numpy(),
                      spec_e=spec_e.numpy(), m=m.numpy(), lsnr=lsnr.numpy(),
                      enhanced_nopad=enhance(model, st, x, pad=False).numpy(),
                      enhanced_atten12=enhance(model, st, x, pad=True, atten_lim_db=12.0).numpy(),
                      coefs=(c if c.dim() == 5 else torch.zeros(0)).numpy())
        path = os.path.join(GOLD, f"dfnet_{name}.npz")
        np.savez_compressed(path, **arrays)
        print(name, {k: v.shape for k, v in arrays.items()}, os.path.getsize(path), "bytes")
    shutil.rmtree(tmp)


if __name__ == "__main__":
    main()
