import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu)")
    config.addinivalue_line("markers", "multigpu: needs at least two B200s on the machine (skipped otherwise)")


def _have_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _gpu_count() -> int:
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def pytest_collection_modifyitems(config, items):
    if _have_gpu():
        if _gpu_count() < 2:
            skip_multi = pytest.mark.skip(reason="needs at least two GPUs; this machine has one")
            for item in items:
                if "multigpu" in item.keywords:
                    item.add_marker(skip_multi)
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
