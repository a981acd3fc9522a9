import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (runs on the B200 box)")


def _has_gpu():
    try:
        from tracs_b200 import _lib
        return _lib.lib().tracs_device_count() > 0
    except Exception:
        return False


HAS_GPU = None


def pytest_collection_modifyitems(config, items):
    global HAS_GPU
    if HAS_GPU is None:
        HAS_GPU = _has_gpu()
    if HAS_GPU:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle_mod():
    from oracle import oracle
    oracle.lib()
    return oracle
