"""Golden fixtures of the DeepFilterNet (v1) row: outputs of the REFERENCE's own modules (df/deepfilternet.py imported
from $DFB_REFERENCE_ROOT) with the random weights of oracle/random_models.py, on top of the CPU oracle for the Rust DSP.
Run: DFB_REFERENCE_ROOT=<reference tree> python oracle/gen_golden_v1.py

Output (small; committed):
  tests/golden/dfnet_DeepFilterNet.npz   DfNet.forward / enhance() on the same 0.2 s two-channel excerpt as the other models
                                         (gen_golden.py), plus a 0.75 s single-channel excerpt for the longer recurrences
"""
from __future__ import annotations

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
from gen_golden import GOLD, excerpt  # noqa: E402


def main():
    rh.import_reference()
    from df.enhance import df_features, enhance
    import torch.nn.functional as F

    noisy = torch.from_numpy(rh.read_wav(os.path.join(GOLD, "assets", "noisy_snr0.wav")))
    tmp = tempfile.mkdtemp()
    model, st, _ = rh.init_random_df(tmp, "DeepFilterNet")
    shutil.rmtree(tmp)
    x = excerpt(noisy)
    y = enhance(model, st, x, pad=True)
    y_nopad = enhance(model, st, x, pad=False)
    y_att = enhance(model, st, x, pad=True, atten_lim_db=12.0)
    xa = F.pad(x, (0, st.fft_size()))
    spec, ef, sf = df_features(xa, st, 96)
    with torch.no_grad():
        spec_e, m, lsnr, alpha = model(spec.clone(), ef, sf)
    x2 = noisy[:, 200000:236000]
    y2 = enhance(model, st, x2, pad=True)
    np.savez_compressed(
        os.path.join(GOLD, "dfnet_DeepFilterNet.npz"), audio=x.numpy(), enhanced=y.numpy(), enhanced_nopad=y_nopad.numpy(),
        enhanced_atten12=y_att.numpy(), spec=spec.numpy(), feat_erb=ef.numpy(), feat_spec=sf.numpy(), spec_e=spec_e.numpy(),
        m=m.numpy(), lsnr=lsnr.numpy(), alpha=alpha.numpy(), audio2=x2.numpy(), enhanced2=y2.numpy(),
        epoch=random_models.epoch("DeepFilterNet"))
    print("wrote dfnet_DeepFilterNet.npz", spec_e.shape, alpha.shape)


if __name__ == "__main__":
    main()
