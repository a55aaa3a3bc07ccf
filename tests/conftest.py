import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden():
    """Vectors produced by the unmodified reference Numba code (oracle/make_golden.py); the c3 group is
    stored in a file of its own to keep each file under 1 MB."""
    groups = {}
    for f in ("reference_numba_golden.npz", "reference_numba_golden_c3.npz"):
        z = np.load(os.path.join(ROOT, "tests", "golden", f))
        for key in z.files:
            g, name = key.split("/")
            groups.setdefault(g, {})[name] = z[key]
    return groups


@pytest.fixture(scope="session")
def golden_warp():
    """Vectors produced by the reference's UNMODIFIED Warp kernel source (oracle/make_golden_warp.py)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "reference_warp_golden.npz"))
    groups = {}
    for key in z.files:
        g, name = key.split("/")
        groups.setdefault(g, {})[name] = z[key]
    return groups


@pytest.fixture(scope="session")
def oracle():
    from oracle import hydro_oracle

    hydro_oracle.build()
    return hydro_oracle


@pytest.fixture(scope="session")
def built_lib():
    """The sm_100a library must exist (built by __graft_entry__.build())."""
    from silver2_isaacsim_b200 import _lib

    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    return _lib.load()
