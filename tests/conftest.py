import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def _have_gpu() -> bool:
    try:
        from structure_from_motion_b200 import _native

        return _native.load_library().sfm_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    gpu = _have_gpu()
    for item in items:
        if "gpu" in item.keywords and not gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def engine():
    from structure_from_motion_b200 import _native

    return _native.get_engine(0)
