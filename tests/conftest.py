import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = False


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    import _golden
    return _golden.load(os.path.join(ROOT, "tests", "golden", "sr3_golden.pt"))


@pytest.fixture(scope="session")
def golden_schedules():
    import torch
    p = os.path.join(ROOT, "tests", "golden", "schedules.pt")
    return torch.load(p, map_location="cpu", weights_only=False)
