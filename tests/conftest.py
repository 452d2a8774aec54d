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


def _cuda_present():
    try:
        import torch
        return bool(torch.cuda.is_available())
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    """A plain `pytest tests` on a machine without a CUDA device skips the `gpu` tests instead of
    failing them.  With a device nothing is skipped here: a missing or broken libsrs_ctr.so on a
    GPU box must fail loudly, not hide behind a skip."""
    if _cuda_present():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_golden_weights(name):
    """Rebuild canonical weights from a tests/golden/*.npz fixture."""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    W = {}
    for k in z.files:
        if k in ("user_ids", "user_rows"):
            continue
        W[k.replace("__", "/")] = z[k]
    table = np.zeros((30001, z["user_rows"].shape[1]), np.float32)
    table[z["user_ids"]] = z["user_rows"]
    W["userId_embedding"] = table
    return W


@pytest.fixture(scope="session")
def head_rows():
    from sparrowrecsys_b200.features import load_samples_csv
    return load_samples_csv(os.path.join(GOLDEN, "samples_head.csv"))


@pytest.fixture(scope="session")
def have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False
