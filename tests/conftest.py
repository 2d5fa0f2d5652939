"""pytest configuration: the `gpu` marker and shared library fixtures."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def port():
    from tests import oracle_lib
    return oracle_lib.load_port()


@pytest.fixture
def reference(request):
    """What the reference build computes for the values this test compares: the library in oracle/_ref when it is
    built, else the recorded CRC-32s of tests/golden/reference_pins.npz (tests/golden/pins.py)."""
    from tests.golden import pins
    r = pins.Reference(request.node.module.__name__ + "::" + request.node.name)
    yield r
    r.finish()
