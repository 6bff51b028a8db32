import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def pkg():
    return importlib.import_module("lc-crf-slam_b200")


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def ref():
    from util import Reference
    return Reference()


@pytest.fixture(scope="session")
def ctx(pkg):
    c = pkg.Context(0)
    yield c
    c.close()
