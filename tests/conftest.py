import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


def pytest_sessionstart(session):
    """The C-ABI library is a build artefact (git-ignored): build it in-tree if this checkout does not have it yet."""
    lib = os.path.join(ROOT, "sow_b200", "csrc", "libsow_b200.so")
    if not os.path.exists(lib):
        import __graft_entry__
        __graft_entry__.build()


class Golden:
    """Lazy view over tests/golden/<group>.npz with '/'-separated keys."""

    def __init__(self, group):
        self._d = np.load(os.path.join(GOLDEN_DIR, f"{group}.npz"), allow_pickle=False)

    def __getitem__(self, key):
        return self._d[key]

    def __contains__(self, key):
        return key in self._d.files

    def keys(self, prefix=""):
        return [k for k in self._d.files if k.startswith(prefix)]


@pytest.fixture(scope="session")
def golden_linear():
    return Golden("linear")


@pytest.fixture(scope="session")
def golden_merge():
    return Golden("merge")


@pytest.fixture(scope="session")
def golden_tt():
    return Golden("tt")


@pytest.fixture(scope="session")
def golden_loop():
    return Golden("loop")


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


def tt_matrix(g, case):
    """Input of a from_matrix / to_matrix case of tt.npz, which keeps only its shape and SHA-256: drawn again as
    tests/golden/make_golden.py drew it (torch.randn on the CPU after seed 0) and checked bit for bit."""
    import hashlib
    import torch
    shape = [int(d) for d in g[f"tt/{case}/shape"]]
    mat = torch.randn(*shape, generator=torch.Generator().manual_seed(0)).numpy()
    assert hashlib.sha256(mat.tobytes()).hexdigest() == str(g[f"tt/{case}/matrix_sha256"]), case
    return mat
