import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


@pytest.fixture(scope="session")
def oracle():
    """The CPU checkers (test infrastructure).  Builds oracle/liboracle.so on first use."""
    from oracle import pyoracle as po
    if po.lib("oracle") is None:
        po.build(ref=os.path.isdir("/root/reference"))
        po._cache.clear()
    assert po.lib("oracle") is not None, "oracle/liboracle.so could not be built"
    return po


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    gdir = os.path.join(ROOT, "tests", "golden")

    def load(name):
        return np.load(os.path.join(gdir, name + ".npz"))
    return load


@pytest.fixture(scope="session")
def reference_digests():
    """Outputs of the unmodified reference on the parity tests' own inputs, as oracle.digests() entries
    (written by tests/golden/make_golden_parity.py)."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_digests.json")) as f:
        return json.load(f)
