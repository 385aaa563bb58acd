import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200")


@pytest.fixture(scope="session")
def orc():
    """The CPU checker: plain-C++ restatement of the reference (oracle/liboracle.so)."""
    import pyoracle
    if not os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so")):
        pyoracle.build()
    return pyoracle.Oracle("orc")


@pytest.fixture(scope="session")
def gpu_ctx():
    import lbfgspp_b200 as lb
    ctx = lb.Context(0)
    yield ctx
    ctx.close()
