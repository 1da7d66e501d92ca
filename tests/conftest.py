import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "thesis-pai-reconstruction_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# a checkout of the original thesis-pai-reconstruction project, for the tests that import its modules directly
REFERENCE = os.environ.get("PAI_REFERENCE_DIR", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs a checkout of the original project in $PAI_REFERENCE_DIR")


def pytest_collection_modifyitems(config, items):
    import torch

    has_gpu = torch.cuda.is_available()
    has_ref = bool(REFERENCE) and os.path.isdir(REFERENCE)
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason="PAI_REFERENCE_DIR does not name a checkout of the original project"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def reference_dir():
    return REFERENCE


@pytest.fixture(scope="session")
def ssim_ref_lib():
    """ctypes handle on the independent fp64 C oracle (oracle/ssim_ref.c)."""
    import ctypes
    import subprocess

    so = os.path.join(ROOT, "oracle", "_build", "libssim_ref.so")
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")])
    lib = ctypes.CDLL(so)
    lib.ssim_ref_f64.restype = ctypes.c_int
    lib.ssim_psnr_grad_ref_f64.restype = ctypes.c_int
    return lib
