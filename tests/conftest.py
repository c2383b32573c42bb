"""pytest configuration: registers the `gpu` marker and puts the repo root on sys.path.

`-m "not gpu"` = oracle vs golden vectors / compiled reference, host logic, C-ABI symbol
checks (runs in the CPU-only authoring container).  `-m gpu` = the parity tests proper,
calling the CUDA path through the C-ABI on a real B200.
"""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import pyoracle

    pyoracle.build(ref=True)
    return pyoracle


@pytest.fixture(scope="session")
def reference(oracle):
    """The reference's outputs: live from oracle/_ref where it is built, else as stored digests."""
    from reference_outputs import Reference

    r = Reference(oracle)
    yield r
    r.save()


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")
