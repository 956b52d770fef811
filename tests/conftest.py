import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def port():
    from oracle import bindings
    if not os.path.exists(bindings.PORT_LIB):
        bindings.build("port")
    return bindings.PortOracle()


@pytest.fixture(scope="session")
def ref():
    """The compiled reference itself, as recorded in tests/golden/reference.npz (tests/recorded_reference.py)."""
    from tests import recorded_reference
    return recorded_reference.oracle()


def pytest_sessionfinish(session):
    from tests import recorded_reference
    recorded_reference.save()


@pytest.fixture(scope="session")
def gpu():
    """The product library on a real device.  Fails loudly if the CUDA extension is missing."""
    from madronalib_b200 import api
    api.lib()  # raises FileNotFoundError when libmlb200.so is absent: no silent fallback
    assert api.device_count() > 0, "no CUDA device visible on a -m gpu run"
    api.init(0)
    return api
