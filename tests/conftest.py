"""pytest configuration: the `gpu` marker and shared helpers.

`-m "not gpu"` : oracle vs golden vectors, host logic, ABI/symbol checks (CPU only).
`-m gpu`       : parity of the CUDA path against the oracle, through the C ABI.
"""
import sys
from pathlib import Path

import pytest

import os

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
os.environ.setdefault("ABPOA_GPU_CHECK_ORDER", "1")     # the whole suite runs with the spliced-order invariants asserted (poa_graph.c)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def product_lib():
    from abpoa_b200 import capi
    return capi.product()


@pytest.fixture(scope="session")
def reference_lib():
    """The unmodified reference's answers, stored under tests/golden/ (tests/golden_reference.py); with
    ABPOA_REFERENCE_RECORD=<file> they come from the live reference and are written to <file>."""
    from golden_reference import GoldenReference
    ref = GoldenReference(os.environ.get("ABPOA_REFERENCE_RECORD") or None)
    yield ref
    ref.save()
