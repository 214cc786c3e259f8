import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
# The reference (grid2op with its bundled data, test-suites and data_test fixtures) is found in $GRID2OP_B200_REF or in
# oracle/_ref, where build() installs it (oracle/reference.py).


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _first_dir(cands):
    for c in cands:
        if c and os.path.isdir(c):
            return c
    return None


def grid2op_root():
    """Directory that contains the reference's ``grid2op`` package (for its bundled grid files)."""
    return _first_dir([
        os.path.join(os.environ.get("GRID2OP_B200_REF", ""), "grid2op") if os.environ.get("GRID2OP_B200_REF") else None,
        os.path.join(REPO, "oracle", "_ref", "grid2op"),
        os.path.join(REPO, "baseline", "_ref", "grid2op"),
    ])


def env_grid(name):
    root = grid2op_root()
    if root is None:
        return None
    p = os.path.join(root, "data", name, "grid.json")
    return p if os.path.exists(p) else None


def data_test_dir():
    root = grid2op_root()
    return _first_dir([os.path.join(root, "data_test") if root else None])


def have_cuda():
    try:
        from grid2op_b200.engine import load_library
        return load_library().b200pf_device_count() > 0
    except Exception:
        return False


@pytest.fixture(scope="session")
def cuda_required():
    if not have_cuda():
        pytest.fail("CUDA device / libb200pf.so required for gpu-marked tests (no CPU fallback exists)")
