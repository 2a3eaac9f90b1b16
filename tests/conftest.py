import os
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle_mod():
    from oracle import oracle as o

    if not os.path.exists(o.ORACLE_SO):
        o.build()
    return o


class Golden(dict):
    """The arrays of several .npz files behind the interface of one (`.files`, `[name]`)."""

    @property
    def files(self):
        return list(self)


@pytest.fixture(scope="session")
def golden():
    """The reference's outputs written by tests/gen_golden.py, split into files of under 1 MB each."""
    import glob

    import numpy as np

    g = Golden()
    for path in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "reference_vectors*.npz"))):
        with np.load(path) as f:
            g.update((k, f[k]) for k in f.files)
    return g


@pytest.fixture(scope="session")
def ref_lib(oracle_mod):
    """The unmodified reference, when its prebuilt .so travelled with the repo (None otherwise)."""
    return oracle_mod.load_ref()
