"""Import the reference's *Python* package (``$DFB_REFERENCE_ROOT/DeepFilterNet/df``) with the
CPU oracle bound as module ``libdf``.

TEST INFRASTRUCTURE ONLY.  Used by oracle/gen_golden*.py (fixture generation) and, for
``read_wav`` / ``si_sdr``, by the tests.  The reference tree is found at $DFB_REFERENCE_ROOT.
Recipe from SURVEY.md Appendix C:
  * the reference's Rust ``libdf`` cannot be built here, so ``sys.modules['libdf']`` is the
    oracle binding (oracle/libdf_oracle.py);
  * torchaudio 2.11 dropped ``AudioMetaData`` which ``df/io.py:10-19`` needs at import time;
  * model archives are unpacked to a scratch directory so ``maybe_download_model`` (network) is
    never reached (enhance.py:92-98).
"""
from __future__ import annotations

import collections
import glob
import os
import sys
import tarfile
import tempfile
import types
import wave
import zipfile

import numpy as np

REF_ROOT = os.environ.get("DFB_REFERENCE_ROOT", "")
SCRATCH = os.environ.get("DFB_REF_SCRATCH", os.path.join(tempfile.gettempdir(), "dfb_ref_models"))


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "DeepFilterNet", "df"))


def unpack_models() -> str:
    os.makedirs(SCRATCH, exist_ok=True)
    for z in glob.glob(os.path.join(REF_ROOT, "models", "*.zip")):
        name = os.path.basename(z)[:-4]
        if not os.path.isdir(os.path.join(SCRATCH, name)):
            zipfile.ZipFile(z).extractall(SCRATCH)
    for t in glob.glob(os.path.join(REF_ROOT, "models", "*_onnx*.tar.gz")):
        name = os.path.basename(t)[:-7]
        dst = os.path.join(SCRATCH, name)
        if not os.path.isdir(dst):
            os.makedirs(dst)
            with tarfile.open(t) as tf:
                for m in tf.getmembers():
                    if m.isfile():
                        m.name = os.path.basename(m.name)
                        tf.extract(m, dst)
    return SCRATCH


def import_reference():
    """Returns the reference's ``df`` package with the oracle as ``libdf``."""
    if not available():
        raise RuntimeError("reference tree not present")
    here = os.path.dirname(os.path.abspath(__file__))
    if here not in sys.path:
        sys.path.insert(0, here)
    import libdf_oracle

    mod = types.ModuleType("libdf")
    for k in ("DF", "erb", "erb_inv", "erb_norm", "unit_norm", "unit_norm_init"):
        setattr(mod, k, getattr(libdf_oracle, k))
    sys.modules["libdf"] = mod
    import torchaudio

    if not hasattr(torchaudio, "AudioMetaData"):
        torchaudio.AudioMetaData = collections.namedtuple(
            "AudioMetaData", "sample_rate num_frames num_channels bits_per_sample encoding")
    p = os.path.join(REF_ROOT, "DeepFilterNet")
    if p not in sys.path:
        sys.path.insert(0, p)
    for k in list(os.environ):
        # df/config.py:119-122: env vars named like options override the ini file
        if k in ("MODEL", "DEVICE", "SR", "FFT_SIZE", "HOP_SIZE", "NB_ERB", "NB_DF", "DF_ORDER",
                 "CONV_CH", "DF_LOOKAHEAD", "CONV_LOOKAHEAD"):
            del os.environ[k]
    import df  # noqa: F401
    import df.enhance  # noqa: F401

    return df


def init_random_df(root: str, name: str, **kw):
    """The reference's ``init_df`` on the random-weight model directory of ``random_models`` (written under `root`):
    the reference builds the model from the shipped config, then loads the seeded weights; the only tensors it keeps
    from its own init are the ERB filterbanks, which it computes from the DF state."""
    import random_models
    d = random_models.write_model_dir(root, name)
    from df.enhance import init_df
    model, st, suffix, _ = init_df(d, log_file=None, log_level="ERROR", epoch="none", **kw)
    missing, unexpected = model.load_state_dict(random_models.state_dict(name), strict=False)
    assert not unexpected and set(missing) <= {"erb_fb", "mask.erb_inv_fb"}, (missing, unexpected)
    model.eval()
    return model, st, suffix


def read_wav(path: str) -> np.ndarray:
    """int16 PCM -> float32 [C, T] (as torchaudio.load(normalize=True): /32768)."""
    with wave.open(path, "rb") as w:
        assert w.getsampwidth() == 2
        n, ch = w.getnframes(), w.getnchannels()
        x = np.frombuffer(w.readframes(n), dtype="<i2").reshape(n, ch).T
    return (x.astype(np.float32) / 32768.0).copy()


def si_sdr(reference: np.ndarray, estimate: np.ndarray) -> float:
    """Restatement of DeepFilterNet/df/evaluation_utils.py:599-619 (that module needs pystoi at
    import time)."""
    reference = reference.reshape(-1, 1)
    estimate = estimate.reshape(-1, 1)
    eps = np.finfo(reference.dtype).eps
    Rss = np.dot(reference.T, reference)
    a = (eps + np.dot(reference.T, estimate)) / (Rss + eps)
    e_true = a * reference
    e_res = estimate - e_true
    Sss = (e_true ** 2).sum()
    Snn = (e_res ** 2).sum()
    return float(10 * np.log10((eps + Sss) / (eps + Snn)))
