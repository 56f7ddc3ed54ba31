import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests", "golden"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    """`pytest tests` on a machine without CUDA: gpu-marked tests are skipped, not errors."""
    try:
        import torch
        have = torch.cuda.is_available()
    except Exception:
        have = False
    if have:
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def bits_equal(a, b):
    """Bitwise equality of float arrays, treating every NaN payload as equal."""
    a = np.asarray(a)
    b = np.asarray(b)
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    it = {4: np.int32, 8: np.int64}[a.dtype.itemsize]
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False
    return np.array_equal(a.view(it)[~na], b.view(it)[~nb])


def assert_bits_equal(a, b, what=""):
    a = np.asarray(a)
    b = np.asarray(b)
    assert a.dtype == b.dtype, f"{what}: dtype {a.dtype} != {b.dtype}"
    assert a.shape == b.shape, f"{what}: shape {a.shape} != {b.shape}"
    if not bits_equal(a, b):
        na, nb = np.isnan(a), np.isnan(b)
        nan_mismatch = int((na != nb).sum())
        both = ~(na | nb)
        diff = np.abs(a[both].astype(np.float64) - b[both].astype(np.float64))
        raise AssertionError(
            f"{what}: not bit-identical: {int((diff > 0).sum())} value mismatches "
            f"(max abs {diff.max() if diff.size else 0:.3e}), {nan_mismatch} NaN-pattern mismatches")


@pytest.fixture(scope="session")
def golden_sl():
    path = os.path.join(ROOT, "tests", "golden", "sl_golden.npz")
    return np.load(path)


@pytest.fixture(scope="session")
def reference_golden():
    """outputs of pysteps v1.21.3 on tests/golden/reference_cases.py (gen_reference_golden.py)"""
    import fingerprint
    return fingerprint.load(os.path.join(ROOT, "tests", "golden", "reference_golden.npz"))
