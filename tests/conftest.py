"""Test tiers:
  -m "not gpu": oracle vs golden vectors, host logic (tokenizer, lowering, grid, slabs), C-ABI symbol check — CPU only.
  -m gpu      : parity of the CUDA path (through the C ABI) against the oracle / golden vectors — needs a B200.
"""
import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_report_header(config):
    from oracle import refbind
    return "reference for the `refbind` tests: " + ("the unmodified reference (oracle/_ref)" if refbind.available() else
                                                    "its plain-C restatement (oracle/restated_ref.py); oracle/_ref is not built")


@pytest.fixture(scope="session")
def mcb():
    if os.environ.get("MCB_TEST_EMU") == "1":
        # developer switch: run the `-m gpu` tests' small cases against the kernels' source executed on the host
        # (tests/emu).  Never set by the driver; the GPU tier always goes through libmcb200.so on a real device.
        from tests import emu
        return emu.load()
    return importlib.import_module("marching-cube-for-implicit-surfaces_b200")


@pytest.fixture(scope="session")
def mcb_emu():
    """The package's ctypes mirror bound to tests/emu/_build/libmcb200_emu.so (device code executed on the host)."""
    from tests import emu
    return emu.load()


@pytest.fixture(scope="session")
def refbind():
    """The unmodified reference (oracle/_ref) where its sources were there to build it; elsewhere its plain-C
    restatement, which tests/test_oracle.py pins to the reference's golden vectors (oracle/restated_ref.py)."""
    from oracle import refbind as R
    if R.available():
        return R
    from oracle import restated_ref
    if not restated_ref.available():
        pytest.skip("oracle/libmcoracle.so not built (run __graft_entry__.build())")
    return restated_ref


@pytest.fixture(scope="session")
def unmodified_reference():
    """The reference's own build, for what no restatement can stand in for (the restatement checked against it)."""
    from oracle import refbind as R
    if not R.available():
        pytest.skip("oracle/_ref/libmcref.so not built: the unmodified reference's sources are not part of the repository")
    return R


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", "cases.npz")
    return np.load(path, allow_pickle=False)
