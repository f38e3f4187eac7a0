import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    import oracle as o
    return o


@pytest.fixture(scope="session")
def ref():
    """The reference's own kernels, answered from tests/golden/ref_calls.npz (tests/ref_golden.py)."""
    import ref_golden
    return ref_golden.session_ref()
