import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    import _libs
    return _libs.load_oracle()


@pytest.fixture(scope="session")
def gemm():
    import _libs
    return _libs.load_pkg()
