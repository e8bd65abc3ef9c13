import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    path = os.path.join(ROOT, "tests", "golden", "golden_v1.pt")
    return torch.load(path, weights_only=False)


@pytest.fixture(scope="session")
def golden_seghead():
    path = os.path.join(ROOT, "tests", "golden", "golden_seghead_v1.pt")
    return torch.load(path, weights_only=False)


@pytest.fixture(scope="session")
def ref_vq():
    """The live reference vq_img module, or None without a reference checkout (VQSEG_REF, oracle/ref_loader.py)."""
    from oracle.ref_loader import load_reference_vq_img
    return load_reference_vq_img()
