import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    with np.load(os.path.join(ROOT, "tests", "golden", "distance_golden.npz")) as z:
        g = dict(z)
    # the unexpanded L2 forms are the same cdist values as the expanded ones, stored once (make_golden.py)
    for case in ("small", "cfg1"):
        g[f"{case}_L2Unexpanded"] = g[f"{case}_L2Expanded"]
        g[f"{case}_L2SqrtUnexpanded"] = g[f"{case}_L2SqrtExpanded"]
    return g
