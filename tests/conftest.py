import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle_lib import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def ref():
    from oracle_lib import RefAnswers
    return RefAnswers()
