import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (sm_100a)")


def _has_gpu():
    try:
        from pylinac_b200 import _native

        return _native.device_count() > 0
    except Exception:
        return False
