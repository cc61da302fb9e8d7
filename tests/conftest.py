import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
if os.path.join(ROOT, "oracle") not in sys.path:
    sys.path.insert(0, os.path.join(ROOT, "oracle"))

PKG = "photoconsistency-visual-odometry_b200"
# config_files/ of a checkout of the original project, named by REF (the adapter build reads the same variable)
REF_CONFIG_DIR = os.path.join(os.environ["REF"], "config_files") if os.environ.get("REF") else ""


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def phovo():
    """The product package (its CUDA library is built in-tree if missing)."""
    mod = importlib.import_module(PKG)
    mod.build()
    return mod


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle binding (test infrastructure)."""
    import oracle_py
    oracle_py.build()
    return oracle_py


@pytest.fixture(scope="session")
def nr():
    import np_restatement
    return np_restatement
