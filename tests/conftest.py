import glob
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "fullsubnet-plus_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


@pytest.fixture(scope="session")
def built_lib():
    """Build (nvcc cross-compiles without a GPU) and load the in-tree C-ABI library."""
    import __graft_entry__ as ge
    ge.build()
    from fsnplus_b200 import _lib
    return _lib.load_library()


GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        """Arrays of <name>.npz, merged with those of its parts <name>.<part>.npz (a fixture split to keep files small)."""
        d = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
        for part in sorted(glob.glob(os.path.join(GOLDEN, glob.escape(name) + ".*.npz"))):
            d.update(np.load(part))
        return d
    return load
