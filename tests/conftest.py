import os
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    """CPU oracle (test infrastructure only)."""
    from oracle.pyoracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def reference():
    """The compiled reference (oracle/_ref), or None where it was never built (no reference tree to build it from)."""
    from oracle.pyoracle import REF_SO, Reference, build
    if not REF_SO.exists():
        try:
            build()
        except Exception:
            pass
    return Reference() if REF_SO.exists() else None


@pytest.fixture(scope="session")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "vectors.npz"))


@pytest.fixture(scope="session")
def golden_planes():
    """Image::writeJPEG of the compiled reference on Images assembled from planes of doubles (tests/golden/make_planes_golden.py)"""
    return np.load(os.path.join(ROOT, "tests", "golden", "planes.npz"))


@pytest.fixture(scope="session")
def encoder():
    """GPU context through the C-ABI.  Raises (does not skip) when the library or the GPU is missing."""
    from jpgenc_b200.capi import Encoder
    e = Encoder(0)
    yield e
    e.close()


def table_fields(t):
    n = int(sum(t.counts))
    return (bytes(t.length), bytes(t.code_msb), bytes(t.counts), bytes(t.symbols[:n]))


def random_symbol_stats(rng, nsym, max_count):
    """a histogram with nsym distinct symbols and a first-occurrence order (unique keys), as K2 would deliver them"""
    import numpy as np
    syms = rng.choice(256, nsym, replace=False)
    count = np.zeros(256, np.uint32)
    first = np.full(256, np.iinfo(np.uint64).max, np.uint64)
    shape = rng.integers(0, 4)
    for rank, s in enumerate(rng.permutation(syms)):
        if shape == 0:
            count[s] = rng.integers(1, max_count)                     # arbitrary
        elif shape == 1:
            count[s] = rng.integers(1, 4)                             # many ties
        elif shape == 2:
            count[s] = max(1, int(max_count * 0.6 ** rank))           # geometric: the length limit of 15 binds
        else:
            count[s] = 1 << min(rank, 30)                             # powers of two: maximally deep tree
        first[s] = np.uint64(rank * 256 + int(rng.integers(0, 130)))
    return count, first
