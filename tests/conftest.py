import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
if GOLDEN not in sys.path:
    sys.path.insert(0, GOLDEN)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden():
    from compact import expand_nrms
    return expand_nrms(np.load(os.path.join(GOLDEN, "nrms_golden.npz")))


@pytest.fixture(scope="session")
def golden_sd(golden):
    return {k[3:]: v for k, v in golden.items() if k.startswith("sd/")}


def rel_l2_rows(a, b):
    """max over rows of ||a-b|| / ||b|| (the north_star's relative tolerance measure)."""
    a = np.asarray(a, dtype=np.float64).reshape(-1, a.shape[-1])
    b = np.asarray(b, dtype=np.float64).reshape(-1, b.shape[-1])
    num = np.linalg.norm(a - b, axis=1)
    den = np.maximum(np.linalg.norm(b, axis=1), 1e-12)
    return float((num / den).max())
