import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Before any test loads an OpenBLAS: the oracle's convolutions must run the sgemm kernel the reference's outputs in
# tests/golden/ref_host.npz were recorded with (test_oracle.py::test_conv_vs_reference_code_same_blas).
from oracle import refcases  # noqa: E402

refcases.pin_blas_core()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


def pytest_sessionstart(session):
    """The shared objects are git-ignored build artefacts: build them once if a fresh checkout lacks them
    (nvcc cross-compiles for sm_100a without a GPU)."""
    need = [os.path.join(ROOT, "caffe_rtpose_b200", "libposeengine.so"), os.path.join(ROOT, "caffe_rtpose_b200", "rtpose.bin"),
            os.path.join(ROOT, "oracle", "liboracle.so")]
    if not all(os.path.exists(p) for p in need):
        import __graft_entry__
        __graft_entry__.build()


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")
