import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


@pytest.fixture(scope="session")
def golden():
    from tests.golden import load
    return load("golden")


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as o
    o.build()
    return o


@pytest.fixture(scope="session")
def ref_lib():
    """oracle/_ref (the reference's own shims); optional -- skip when not built."""
    from lilliput_b200 import abi
    if not os.path.exists(abi.REF_LIB):
        pytest.skip("oracle/_ref/libref_oracle.so not built (needs /root/reference)")
    return abi.load_reference()


@pytest.fixture(scope="session")
def cuda_lib():
    """The product library.  No fallback: a missing .so or device is a hard failure."""
    from lilliput_b200 import abi
    lib = abi.load_cuda()
    assert lib.backend == "cuda-sm100a"
    return lib
