import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    have_gpu = None
    for item in items:
        if "gpu" in item.keywords:
            if have_gpu is None:
                have_gpu = _has_gpu()
            if not have_gpu:
                item.add_marker(pytest.mark.skip(reason="no CUDA device"))
