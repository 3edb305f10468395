import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def pytest_collection_modifyitems(config, items):
    # `-m gpu` on a box without a device must fail loudly, not skip: there is no CPU fallback.
    pass


@pytest.fixture(scope="session")
def oracle():
    import oracle_lib

    return oracle_lib.port()


@pytest.fixture
def ref(request):
    """For a test that compares with the reference: its calls into oracle/_ref answer from tests/golden/reference/."""
    import oracle_lib

    with oracle_lib.reference_tape(request.module.__name__, request.node.name):
        yield
