import os
import sys

import pytest

# The oracle tests compare CPU fp32 results with stored fixtures to within op-ordering noise, and the fake
# quantisers turn a last-bit difference into a rounding flip.  The fixtures were computed on MKL's AVX-512 code
# path; pinning MKL to that branch (conditional numerical reproducibility) makes other x86 hosts compute the same
# bits.  MKL reads the setting at its first call, so it is set here, before any test runs.
os.environ.setdefault("MKL_CBWR", "AVX512")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "myrtle-vision_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
