import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLDEN)
from golden_io import load_golden  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


@pytest.fixture(scope="session")
def small_cfg():
    import json
    with open(os.path.join(GOLDEN, "small_cfg.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def golden_fwd():
    return load_golden(os.path.join(GOLDEN, "small_fwd"))


@pytest.fixture(scope="session")
def golden_step():
    return load_golden(os.path.join(GOLDEN, "small_step"))


@pytest.fixture(scope="session")
def golden_modules():
    return load_golden(os.path.join(GOLDEN, "modules"))
