"""Model directories laid out like the shipped pretrained models (``config.ini`` + ``checkpoints/``), with the shipped
configs (tests/golden/models/<name>/config.ini) and seeded random weights in place of the trained checkpoints, which are
too large to keep in the repository.  The golden fixtures (oracle/gen_golden*.py) and the tests build the same weights
from the same seed, so the tests compare against the reference modules' outputs without any file from outside the tree.

TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
CONFIGS = os.path.join(ROOT, "tests", "golden", "models")
SEED = 1
# checkpoint file names of the shipped models (the epoch is part of the name; DeepFilterNet3_ll ships only as ONNX)
CHECKPOINTS = {"DeepFilterNet3": "model_120.ckpt.best", "DeepFilterNet2": "model_96.ckpt.best",
               "DeepFilterNet": "model_30.ckpt", "DeepFilterNet3_ll": "model_0.ckpt.best"}


def epoch(name: str) -> int:
    return int(CHECKPOINTS[name].split(".")[0].split("_")[1])


def config(name: str):
    from deepfilternet_b200.config import load_config
    return load_config(os.path.join(CONFIGS, name, "config.ini"), env={})


def state_dict(name: str):
    """The seeded random weights of model `name`, with the shipped checkpoint's tensor names."""
    from deepfilternet_b200.weights import random_state_dict
    return random_state_dict(config(name), seed=SEED)


def write_model_dir(root: str, name: str) -> str:
    """<root>/<name>/{config.ini, checkpoints/<checkpoint>} -> the model directory."""
    import shutil

    import torch
    d = os.path.join(root, name)
    os.makedirs(os.path.join(d, "checkpoints"), exist_ok=True)
    shutil.copyfile(os.path.join(CONFIGS, name, "config.ini"), os.path.join(d, "config.ini"))
    torch.save(state_dict(name), os.path.join(d, "checkpoints", CHECKPOINTS[name]))
    return d
