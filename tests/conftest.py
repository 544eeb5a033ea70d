import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box: pytest -m gpu)")


@pytest.fixture(scope="session")
def port():
    from oracles import port_lib
    return port_lib()


@pytest.fixture(scope="session")
def ref():
    from oracles import ref_lib
    lib = ref_lib()
    if lib is None:
        pytest.skip("oracle/_ref not built (PTB_REFERENCE_DIR names no checkout of the reference); the golden fixtures carry its outputs")
    return lib


@pytest.fixture(scope="session")
def devsim():
    from oracles import devsim_lib
    return devsim_lib()


@pytest.fixture(scope="session")
def gpu():
    import pathtracer_b200
    return pathtracer_b200.load()
