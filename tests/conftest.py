import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def product():
    """the product package (directory name has a hyphen, so importlib by string)"""
    return importlib.import_module("swift-png_b200")


@pytest.fixture(scope="session")
def pngb200():
    return product()


@pytest.fixture(scope="session")
def ctx(pngb200):
    c = pngb200.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="session")
def orc():
    from oracle import oracle
    oracle.build()
    return oracle
