"""pytest configuration: registers the `gpu` marker and builds the CPU oracle once.

`-m "not gpu"`: oracle vs golden fixtures (made by the reference itself), host-side logic, C-ABI
symbol check.  `-m gpu`: the parity tests proper — CUDA path (through the C-ABI) vs oracle/golden.
"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session", autouse=True)
def _build_oracle():
    # test infrastructure only; the product library is built by __graft_entry__.build()
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"], check=True,
                   stdout=subprocess.DEVNULL)
    # the live comparisons with the reference: oracle/Makefile builds it where its sources are (REF, or the checkout
    # $HANABIZERO_REFERENCE names) and does nothing without them
    ref = os.environ.get("HANABIZERO_REFERENCE")
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "ref"] + (["REF=" + os.path.abspath(ref)] if ref else []),
                   check=True, stdout=subprocess.DEVNULL)


def golden(name):
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", name), allow_pickle=False)
