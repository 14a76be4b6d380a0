"""pytest configuration: registers the `gpu` marker and shared fixtures.

`-m "not gpu"` runs here on CPU (oracle vs golden vectors, host logic, C-ABI symbol export, gloo world_size-2);
`-m gpu` runs on a B200 and calls the CUDA path through the C-ABI.
"""
import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_sessionstart(session):
    """Build the native libraries when they are missing or stale (a clean checkout has no .so files: they are
    git-ignored).  This is the test harness building the product, not a fallback: the product itself only loads
    uninext_b200/lib/libmsda_b200.so and raises when it is absent (tests/test_cabi_symbols.py)."""
    try:
        from uninext_b200 import build as _b
        _b.build()
        from oracle import msda_oracle as _o
        _o.build()
    except Exception as exc:                       # no nvcc / gcc here: the tests that need the libraries will say so
        print(f"[conftest] native build skipped: {exc}")


def golden_names():
    """Op-level golden cases (module-level ones are named module_*.npz and loaded explicitly)."""
    names = (os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    return sorted(n for n in names if not n.startswith("module_"))


def load_golden(name):
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(params=golden_names())
def golden(request):
    case = load_golden(request.param)
    case["name"] = request.param
    return case
