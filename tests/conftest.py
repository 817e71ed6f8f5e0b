import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def port():
    from oracle.oracle import Oracle
    return Oracle("port")


@pytest.fixture(scope="session")
def built_libs():
    """The product libraries must exist (built in-tree by __graft_entry__.build())."""
    from ntg_b200 import build
    if not os.path.exists(build.CORE_SO):
        build.build_all()
    return build.LIB
