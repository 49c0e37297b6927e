import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def model_dir(tmp_path_factory):
    """Model directories laid out like the shipped ones (config.ini + checkpoints/): the shipped configs with seeded
    random weights (oracle/random_models.py), the weights the golden fixtures were made with."""
    import random_models
    root = str(tmp_path_factory.mktemp("models"))
    for name in random_models.CHECKPOINTS:
        random_models.write_model_dir(root, name)
    return root
