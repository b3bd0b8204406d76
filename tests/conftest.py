import contextlib
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")


def _load(name):
    z = np.load(os.path.join(GOLDEN, name))
    meta = json.loads(bytes(z["meta"]).decode())
    return z, meta


@pytest.fixture(scope="session")
def golden_retrieval():
    return _load("retrieval.npz")


@pytest.fixture(scope="session")
def golden_model():
    return _load("model.npz")


def golden_checksum(*arrays) -> float:
    """Same formula as oracle/make_golden.py::checksum."""
    s = 0.0
    for a in arrays:
        a = np.asarray(a, np.float64).ravel()
        s += float((a * (1.0 + (np.arange(a.size) % 7))).sum())
    return s


def golden_sha256(a) -> str:
    """Digest a golden array is stored as when the tests compare it bit for bit."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@contextlib.contextmanager
def golden_cpu_threads():
    """One CPU thread while computing what is compared bit for bit with tests/golden/: torch's CPU
    float32 products sum in another order when split over many threads (16 and more)."""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def golden_grad(z, key):
    """A reference gradient stored as a fixed sample (oracle/make_golden.py::compact_model):
    (flat indices, values, absolute maximum and L2 norm of the whole array, its shape)."""
    return (z[key + "/idx"].astype(np.int64), z[key + "/val"], float(z[key + "/absmax"]),
            float(z[key + "/norm"]), tuple(int(s) for s in z[key + "/shape"]))


@pytest.fixture(scope="session")
def have_gpu():
    import torch
    return torch.cuda.is_available()
