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
def twin():
    from oracle import twin as tw
    tw.build()
    return tw


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


@pytest.fixture(scope="session")
def golden():
    return load_golden
