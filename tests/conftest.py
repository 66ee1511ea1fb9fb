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
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def reference_answers(key):
    """What the unmodified reference answered for one test's queries (tests/golden/reference_answers.json, written
    by tests/golden/make_reference_answers.py): small results as rows, large ones as digest() of a canonical form."""
    with open(os.path.join(GOLDEN, "reference_answers.json")) as f:
        return json.load(f)[key]


def digest(a):
    """sha256 of an array's dtype, shape and bytes: equal digests mean bit-identical arrays."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


@pytest.fixture(scope="session")
def ctx():
    """One b200 context on cuda:0, enqueueing on torch's current stream (so torch events see our kernels)."""
    import torch
    from duckdb_b200 import operators as ops

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    torch.cuda.set_device(0)
    c = ops.Context(0, torch.cuda.current_stream().cuda_stream)
    yield c
    c.close()

