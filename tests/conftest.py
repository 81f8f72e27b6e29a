import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    """Every case of tests/golden/latent_ref_<case>.npz (one file per case keeps each under 1 MB), keys '<case>/...'."""
    out = {}
    for path in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "latent_ref_*.npz"))):
        with np.load(path) as g:
            out.update({k: g[k] for k in g.files})
    return out


@pytest.fixture(scope="session")
def lib():
    """The C-ABI library, built if stale (nvcc cross-compiles without a GPU)."""
    from shacira_b200 import build, _lib
    build.build()
    return _lib
