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
    from oracle import pyoracle as po
    po.build(ref=False)    # the checker only; tests that need the reference use oracle/_ref when the tree has it
    return po.Oracle()


@pytest.fixture(scope="session")
def fi():
    """The product C-ABI library through ctypes. GPU tests fail loudly if it is missing."""
    from freeimpala_b200 import build
    build.build()          # no-op when the in-tree .so is up to date
    import freeimpala_b200 as m
    m.load_library()
    return m
