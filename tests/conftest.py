"""Shared fixtures.  GPU tests are marked ``gpu`` and call the product library
through its C ABI; everything else runs on the CPU (oracle, host logic, ABI)."""
import importlib
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "oracle"))

PKG_NAME = "software-defined-radio-course-project_b200"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu)")


def _has_gpu() -> bool:
    try:
        pkg = importlib.import_module(PKG_NAME)
        return pkg.binding.device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    # `-m gpu` on a box without a GPU must fail loudly, not skip: the product has no CPU path.
    pass


@pytest.fixture(scope="session")
def pkg():
    return importlib.import_module(PKG_NAME)


@pytest.fixture(scope="session")
def fm(pkg):
    """The product binding; GPU tests fail (not skip) if the library or device is missing."""
    pkg.binding.load()
    assert pkg.binding.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return pkg.binding


@pytest.fixture(scope="session")
def port():
    import pyoracle
    return pyoracle.Port()


@pytest.fixture(scope="session")
def reference():
    """The reference's own compiled code, or None: then tests/reference_vectors.py compares with what it
    computed, stored in tests/golden/reference_vectors.npz."""
    import warnings
    import pyoracle
    why = pyoracle.reference_missing_reason()
    if why is not None:
        warnings.warn(f"reference not available ({why}): comparing with the stored reference vectors")
        return None
    return pyoracle.Reference()


@pytest.fixture(scope="session")
def synth(pkg):
    return pkg.synth


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def assert_bits_equal(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    ne = np.nonzero(bits(a) != bits(b))[0] if a.ndim == 1 else np.argwhere(bits(a) != bits(b))
    assert len(ne) == 0, (f"{what}: {len(ne)} of {a.size} differ; first at {ne[0]}: "
                          f"{a[tuple(np.atleast_1d(ne[0]))]!r} vs {b[tuple(np.atleast_1d(ne[0]))]!r}")
