import os
import sys

import pytest

REPO_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO_ROOT not in sys.path:
    sys.path.insert(0, REPO_ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA GPU (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    from tests import oracle_lib
    return oracle_lib.load_oracle()


@pytest.fixture(scope="session")
def recorded():
    """The reference's answers to the seeded cases of tests/golden/make_golden.py
    (tests/golden/ref_recorded.json)."""
    import json
    with open(os.path.join(REPO_ROOT, "tests", "golden", "ref_recorded.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def native():
    from elbencho_b200 import _native
    return _native.load()


@pytest.fixture(scope="session")
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch.device("cuda:0")
