import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200)")


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def ac_small(golden_dir):
    """tests/golden/ac_small.npz keyed '<case>/<field>' like the other golden files; it is stored one array per
    field (tests/golden/make_golden.py, save_by_field)."""
    g = np.load(os.path.join(golden_dir, "ac_small.npz"))
    names = g["names"]
    cases = {"names": names}
    for f in g.files:
        if f == "names" or f.endswith("_off"):
            continue
        v = g[f]
        if f"{f}_off" in g.files:
            off = g[f"{f}_off"]
            cases.update((f"{nm}/{f}", v[off[i]:off[i + 1]]) for i, nm in enumerate(names))
        else:
            cases.update((f"{nm}/{f}", v[i]) for i, nm in enumerate(names))
    return cases
