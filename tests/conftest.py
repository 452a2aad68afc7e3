import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# a checkout of the unmodified Trustworthy-AI-Group/TransferAttack, for the tests marked `reference`
REF_ROOT = os.environ.get("TRANSFERATTACK_REFERENCE", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs a checkout of the unmodified reference in $TRANSFERATTACK_REFERENCE")


def pytest_collection_modifyitems(config, items):
    # `-m gpu` tests must never silently pass on a box without a GPU
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not (REF_ROOT and os.path.isdir(os.path.join(REF_ROOT, "transferattack"))):
            item.add_marker(pytest.mark.skip(reason="no reference checkout ($TRANSFERATTACK_REFERENCE)"))


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def bits_equal(a, b):
    """Bit-level equality for fp32 arrays with NaN == NaN (payload-insensitive) and +0 == -0 distinguished."""
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False
    return np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def n_diff_bits(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    na = np.isnan(a) & np.isnan(b)
    return int(((a.view(np.uint32) != b.view(np.uint32)) & ~na).sum())


def ulp_diff(a, b):
    a = np.ascontiguousarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.ascontiguousarray(b, np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a); b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)
