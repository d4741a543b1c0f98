import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def sampler256_golden():
    """case -> the arrays of tests/golden/sampler256_<case>.npz with ``adjs_ls`` [10, 2, C_e, N, N] rebuilt from what
    the file stores (tests/golden/make_golden_full.py: save_sampler256): snapshot 9 is ``adjs[:2]``; snapshot 0, the
    initial noise, is not stored and reads as NaN so that no comparison can pass against it."""
    def load(case):
        g = dict(np.load(os.path.join(GOLDEN, f"sampler256_{case}.npz")))
        mid = g.pop("adjs_ls_mid")
        g["adjs_ls"] = np.concatenate([np.full_like(mid[:1], np.nan), mid, g["adjs"][None, :2]])
        return g
    return load
