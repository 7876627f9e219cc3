import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def vectors():
    import util
    return util.golden_vectors()


@pytest.fixture(scope="session")
def oracle():
    """our CPU restatement (oracle/liboracle.so)"""
    import util
    return util.oracle_lib()


@pytest.fixture(scope="session")
def ref():
    """the unmodified reference built by `make -C oracle ref REF=<its source tree>` (oracle/_ref); skipped when not built"""
    import util
    lib = util.ref_lib()
    if lib is None:
        pytest.skip("oracle/_ref not built")
    return lib


@pytest.fixture(scope="session")
def chk():
    """the checker used for parity: the real reference when present, else the restatement"""
    import util
    return util.checker_lib()


@pytest.fixture(scope="session")
def sim():
    """device math compiled for the host (tests/hostsim) -- CPU-tier check of the CUDA sources"""
    import util
    return util.hostsim_lib()


@pytest.fixture(scope="session")
def gpu():
    """the product: libgoldilocks_b200.so on a real GPU.  No fallback: a missing library is an error."""
    import libgoldilocks_b200 as g
    lib = g.load()
    import ctypes as C
    lib.lib.goldilocks_b200_init.restype = C.c_int32
    assert lib.lib.goldilocks_b200_init() == -1, "goldilocks_b200_init failed (no B200?)"
    return lib
