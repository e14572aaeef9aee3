import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PKG = "3d_planetary_rt_model_b200"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def synth():
    return importlib.import_module(PKG + ".synth")


@pytest.fixture(scope="session")
def binding():
    return importlib.import_module(PKG + ".binding")


@pytest.fixture(scope="session")
def oraclebind():
    from oracle import oraclebind as ob
    ob.build()
    return ob


@pytest.fixture(scope="session")
def refbind():
    """the reference's own hot-path source built in place (oracle/_ref); absent => skip"""
    from oracle import refbind as rb
    if not rb.available("f64"):
        pytest.skip("oracle/_ref not built (needs the reference's source: B200RT_REFERENCE, see oracle/Makefile)")
    return rb
