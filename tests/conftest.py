import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


# HSB200_EMU=1: run the tests marked `gpu` on a CPU against the SIMT-emulated build of the
# library (tests/emu: the kernels' own sources compiled as C++; test infrastructure, kernel
# LOGIC only).  Tests that need the real device (torch CUDA tensors, peer memory, the linked C
# example, timing) skip themselves through `real_gpu`.
EMU = os.environ.get("HSB200_EMU") == "1"


@pytest.fixture(scope="session")
def hs():
    """The product C-ABI library through its ctypes binding (built on demand)."""
    from hyperscan_b200 import build, capi
    if EMU:
        sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
        import build_emu
        assert capi._lib is None
        capi.LIB_PATH = build_emu.build()
        capi.lib()
        return capi
    build.build_product()
    capi.lib()
    return capi


@pytest.fixture
def real_gpu():
    if EMU:
        pytest.skip("needs the real device (not modelled by the SIMT emulator)")


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference runtime (oracle/_ref), or where it is not built
    the answers it gave, recorded under tests/golden/ref_results."""
    import oracle.ref as r
    if not r.available():
        pytest.skip("oracle/_ref not built and no recorded reference answers")
    return r


@pytest.fixture(autouse=True)
def _reset_build_options():
    yield
    try:
        from hyperscan_b200 import capi
        if capi._lib is not None:
            capi.set_build_option("reset", 0)
    except Exception:
        pass


@pytest.fixture
def emu_only():
    if not EMU:
        pytest.skip("single-process stand-in for a multi-GPU path: runs on the SIMT emulator only")
