"""Golden vectors for the optional stages of the enhancement path -- the post filter (`init_df(post_filter=True)`,
deepfilternet3.py:448-454 / modules.py:234-245) and `mask_only` (enhance.py:172-175, checkpoint.py:32) -- produced by the
REFERENCE's own modules (imported from $DFB_REFERENCE_ROOT) with the random weights of oracle/random_models.py on the
excerpt of gen_golden.py.
Run:  DFB_REFERENCE_ROOT=<reference tree> python oracle/gen_golden_pf.py   ->  tests/golden/dfnet_pf.npz
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
import ref_harness as rh  # noqa: E402
from gen_golden import GOLD, excerpt  # noqa: E402


def main():
    rh.import_reference()
    from df.enhance import enhance
    noisy = torch.from_numpy(rh.read_wav(os.path.join(GOLD, "assets", "noisy_snr0.wav")))
    x = excerpt(noisy)
    out = {"audio": x.numpy()}
    tmp = tempfile.mkdtemp()
    for name in ("DeepFilterNet3", "DeepFilterNet2"):
        model, st, suffix = rh.init_random_df(tmp, name, post_filter=True)
        assert suffix.endswith("_pf")
        out[f"{name}_pf"] = enhance(model, st, x, pad=True).numpy()
        out[f"{name}_pf_atten12"] = enhance(model, st, x, pad=True, atten_lim_db=12.0).numpy()
        model, st, _ = rh.init_random_df(tmp, name, mask_only=True)
        out[f"{name}_mask_only"] = enhance(model, st, x, pad=True).numpy()
    shutil.rmtree(tmp)
    np.savez_compressed(os.path.join(GOLD, "dfnet_pf.npz"), **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
