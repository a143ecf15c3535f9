import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def lib():
    from splatt_b200 import _abi
    return _abi.load()


@pytest.fixture(scope="session")
def refmod():
    """The reference's answers: the compiled, unmodified reference (oracle/_ref) where it was
    built, otherwise its stored answers to the same calls (tests/refgold.py)."""
    from tests import refgold
    return refgold
