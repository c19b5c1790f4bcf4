import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


@pytest.fixture(scope="session")
def emu():
    """Binds the host-only test double of the device backend (tests/emu) for CPU tests."""
    import common
    common.use_emu()
    yield
    

@pytest.fixture(scope="session")
def cuda():
    import common
    common.use_cuda()
    yield


@pytest.fixture(autouse=True)
def _bind_requested_library(request):
    """emu and cuda are set up once per session, but one session may run CPU and GPU tests in turn: every test
    that asks for one of them gets its library bound again, not the one the test before it left bound."""
    import common
    if "cuda" in request.fixturenames:
        common.use_cuda()
    elif "emu" in request.fixturenames:
        common.D._ffi.use_library(common.EMU_LIB)
    yield
