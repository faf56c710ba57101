import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.oracle_py import Oracle
    return Oracle()
