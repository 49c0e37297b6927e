"""Generate the committed golden fixtures under tests/golden/ by running the REFERENCE's own
Python modules (imported from $DFB_REFERENCE_ROOT) on top of the CPU oracle for the Rust DSP.
The models carry the seeded random weights of oracle/random_models.py (the shipped checkpoints are
too large to keep in the repository).  Run:  DFB_REFERENCE_ROOT=<reference tree> python oracle/gen_golden.py

Outputs (small; committed):
  tests/golden/erb_widths.json       ERB band widths recovered from the `erb_fb` buffers stored in
                                     the shipped checkpoints (pins libDF/src/lib.rs:68-100 bit-exact)
  tests/golden/kat.json              SI-SDR of the reference modules + oracle on the whole recording
  tests/golden/dfnet_<model>.npz     reference DfNet.forward / enhance() outputs on a 0.2 s excerpt
  tests/golden/assets/*.wav          the two 48 kHz test recordings used by the reference's KAT
"""
from __future__ import annotations

import json
import os
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


def excerpt(noisy: torch.Tensor) -> torch.Tensor:
    """0.2 s, two channels (second = time-shifted, attenuated) to exercise batching."""
    return torch.stack([noisy[0, 96000:105600], 0.5 * noisy[0, 130000:139600]])


def main():
    os.makedirs(os.path.join(GOLD, "assets"), exist_ok=True)
    for w in ("noisy_snr0.wav", "clean_freesound_33711.wav"):
        shutil.copyfile(os.path.join(rh.REF_ROOT, "assets", w), os.path.join(GOLD, "assets", w))
    d = rh.unpack_models()
    rh.import_reference()
    from df.enhance import df_features, enhance, init_df
    import torch.nn.functional as F

    widths = {}
    for name in ("DeepFilterNet3", "DeepFilterNet2"):
        fb = init_df(os.path.join(d, name), log_file=None, log_level="ERROR")[0].state_dict()["erb_fb"].numpy()
        # [F, E], non-zero pattern = band membership
        widths[name] = [int((fb[:, b] != 0).sum()) for b in range(fb.shape[1])]
        # bands must be contiguous and ordered
        starts = [int(np.argmax(fb[:, b] != 0)) for b in range(fb.shape[1])]
        assert starts == list(np.cumsum([0] + widths[name][:-1]))

    noisy = torch.from_numpy(rh.read_wav(os.path.join(GOLD, "assets", "noisy_snr0.wav")))
    clean = rh.read_wav(os.path.join(GOLD, "assets", "clean_freesound_33711.wav"))
    kat = {}
    tmp = tempfile.mkdtemp()
    for name in ("DeepFilterNet3", "DeepFilterNet2", "DeepFilterNet", "DeepFilterNet3_ll"):
        model, st, _ = rh.init_random_df(tmp, name)
        out = enhance(model, st, noisy, pad=True)
        kat[name] = dict(target=rh.si_sdr(clean, out.numpy()), epoch=random_models.epoch(name), n_samples=int(noisy.shape[1]))
        print(name, kat[name])
        if name == "DeepFilterNet":
            continue  # oracle/gen_golden_v1.py
        x = excerpt(noisy)
        y = enhance(model, st, x, pad=True)
        xa = F.pad(x, (0, st.fft_size()))
        spec, ef, sf = df_features(xa, st, 96)
        with torch.no_grad():
            spec_e, m, lsnr, c = model(spec.clone(), ef, sf)
        arrays = dict(audio=x.numpy(), enhanced=y.numpy(), spec=spec.numpy(), feat_erb=ef.numpy(), feat_spec=sf.numpy(),
                      spec_e=spec_e.numpy(), m=m.numpy(), lsnr=lsnr.numpy())
        if name != "DeepFilterNet3_ll":
            arrays.update(enhanced_nopad=enhance(model, st, x, pad=False).numpy(),
                          enhanced_atten12=enhance(model, st, x, pad=True, atten_lim_db=12.0).numpy(),
                          coefs=(c if c.dim() == 5 else torch.zeros(0)).numpy())
        np.savez_compressed(os.path.join(GOLD, f"dfnet_{name}.npz"), **arrays)
    shutil.rmtree(tmp)
    with open(os.path.join(GOLD, "erb_widths.json"), "w") as f:
        json.dump(dict(params=dict(sr=48000, fft_size=960, nb_bands=32, min_nb_freqs=2),
                       from_checkpoint_erb_fb=widths), f, indent=1)
    with open(os.path.join(GOLD, "kat.json"), "w") as f:
        json.dump(kat, f, indent=1)


if __name__ == "__main__":
    main()
