import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200 box)")


@pytest.fixture(scope="session")
def port():
    """Our CPU restatement (oracle/libnavoracle.so); built on demand with g++."""
    from oracle import pyoracle
    return pyoracle.load("port")


@pytest.fixture(scope="session")
def ref():
    """The reference's own compiled sources (oracle/_ref/libnavref.so); only where it was built."""
    from oracle import pyoracle
    if not pyoracle.available("reference"):
        if pyoracle.reference_dir():
            pyoracle.build("reference")
        else:
            pytest.skip("oracle/_ref/libnavref.so not present (needs NAVIGATION_REFERENCE to build)")
    return pyoracle.load("reference")


@pytest.fixture(scope="session")
def cuda():
    """The product: navigation_b200/libnavgpu.so through its C ABI.  No fallback: a missing library or device fails."""
    import navigation_b200
    from navigation_b200 import build
    build.build()
    api = navigation_b200.load()
    assert api.device_count() > 0, "GPU tests need a CUDA device; libnavgpu has no CPU path"
    return api
