import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle_mod():
    import oracle
    oracle.build()
    return oracle


@pytest.fixture(scope="session")
def synth_sd():
    from read_b200 import synth
    return synth.synth_state_dict(synth.SEED)


def load_golden(name):
    import numpy as np
    return np.load(os.path.join(GOLDEN, name + ".npz"))
