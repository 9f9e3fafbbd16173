import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "sc-sfmlearner-release_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden")
for p in (ROOT, PKG, GOLDEN):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden_warp():
    """warp_loss_{in,zeros,border,misc}.npz (make_golden.py stores the vectors in parts of under 1 MB) as one mapping."""
    out = {}
    for part in ("in", "zeros", "border", "misc"):
        out.update(np.load(os.path.join(GOLDEN, "warp_loss_%s.npz" % part)))
    return out


@pytest.fixture(scope="session")
def golden_nets():
    return np.load(os.path.join(GOLDEN, "nets.npz"))
