import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


def pytest_collection_modifyitems(config, items):
    """`pytest tests` on a machine without a CUDA device skips the gpu-marked tests instead of failing them."""
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device (run with `-m gpu` on the B200 box)")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    cases = {}
    for name in ("raster_golden.npz", "clip_golden.npz"):  # (two files: each stays under 1 MB)
        data = np.load(os.path.join(ROOT, "tests", "golden", name))
        for key in data.files:
            case, field = key.rsplit("/", 1)
            cases.setdefault(case, {})[field] = data[key]
    return cases


@pytest.fixture(scope="session")
def built_lib():
    """The C-ABI library, built in-tree (nvcc cross-compiles without a GPU)."""
    from pytorch3d_b200 import build
    return build.build()
