import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def seeded_theta(g):
    """Parameter vector of a fixture that stores how to draw it rather than its values (large parameter
    vectors would push a fixture past 1 MB): segment i is ``theta_sizes[i]`` draws from
    U(theta_lo[i], theta_hi[i]) of ``np.random.RandomState(theta_seed)``, rounded to fp16."""
    rng = np.random.RandomState(int(g["theta_seed"]))
    parts = [rng.uniform(lo, hi, int(n)) for n, lo, hi in zip(g["theta_sizes"], g["theta_lo"], g["theta_hi"])]
    return np.concatenate(parts).astype(np.float16).astype(np.float32)


@pytest.fixture
def golden():
    return load_golden


def rel_err(a, b):
    """max|a-b| / max|b| -- the tolerance definition of SURVEY App. A.5."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))
