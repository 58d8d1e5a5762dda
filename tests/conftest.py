import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden2():
    """Round-2 fixtures: BASELINE configs and the chunked / outpaint branches (tests/golden/make_golden_r2.py)."""
    from tests.golden.sampled import Golden
    return Golden(os.path.join(ROOT, "tests", "golden", "reference_outputs_r2.npz"))


@pytest.fixture(scope="session")
def golden():
    from tests.golden.sampled import Golden
    return Golden(os.path.join(ROOT, "tests", "golden", "reference_outputs.npz"))
