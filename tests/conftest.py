import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 CUDA devices on one box (skipped otherwise)")


def pytest_collection_modifyitems(config, items):
    import torch
    n_dev = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n_dev < 2:
        skip_multi = pytest.mark.skip(reason=f"needs >= 2 CUDA devices ({n_dev} present)")
        for item in items:
            if "multigpu" in item.keywords:
                item.add_marker(skip_multi)
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
