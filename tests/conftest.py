import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def lib():
    """the product library; building it is part of the fixture so `pytest` alone works from a clean tree"""
    from matrixone_b200 import build, capi
    build.build()
    return capi.load_library()


@pytest.fixture(scope="module")
def _ref_tape_store(request):
    import ref_tape
    name = request.module.__name__.rpartition(".")[2]
    store = ref_tape.module_store(name)
    yield store
    ref_tape.write_store(name, store)


@pytest.fixture
def ref_tape(request, _ref_tape_store):
    """the original's results for this test, replayed from tests/golden/ (see ref_tape.py)"""
    import ref_tape
    tape = ref_tape.Tape(_ref_tape_store, request.node.name)
    yield tape
    tape.close()


@pytest.fixture(scope="session")
def gpu(lib):
    from matrixone_b200 import capi
    rc = lib.MoB200_Init(-1)
    if rc != 0:
        pytest.fail("libmo_b200 could not initialise a CUDA device: " + capi.last_error(lib))
    return lib
