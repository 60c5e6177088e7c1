import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    import _util
    return _util.load_oracle()


@pytest.fixture(scope="session")
def emul():
    import _util
    return _util.load_emul()


@pytest.fixture(scope="session")
def hmref():
    """the reference's compiled functions (oracle/_ref/libhmref.so), or None where they were not built"""
    import _util
    return _util.load_hmref()


@pytest.fixture(scope="session")
def cucd():
    import _util
    return _util.load_package()
