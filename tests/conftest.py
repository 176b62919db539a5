import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import pyoracle
    pyoracle.build()
    return pyoracle


@pytest.fixture
def ref(request, oracle):
    """Outputs of the original SceneLib2 sources for this test (tests/refgolden.py)."""
    from refgolden import Recording
    r = Recording(request.node.name[len("test_"):], oracle)
    yield r
    r.close()


@pytest.fixture(scope="session")
def refmodels(oracle):
    r = oracle.ref_models()
    if r is None:
        pytest.skip("oracle/_ref/libsl2refmodels.so not built (reference tree absent)")
    return r
