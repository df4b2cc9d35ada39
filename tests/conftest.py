"""Test configuration.

    python -m pytest tests -q -m "not gpu"    oracle vs golden vectors, host logic, C-ABI symbols (CPU)
    python -m pytest tests -q -m gpu          parity of the CUDA path against the oracle (B200)
"""

from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parent.parent
for p in (str(REPO), str(REPO / "anemoi-transform_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = REPO / "tests" / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "reference: needs the reference sources (ANEMOI_REFERENCE_SRC, see oracle/reference_import.py)")


def _ensure_library():
    """Build libat_b200.so if it is missing (nvcc cross-compiles without a GPU)."""
    from anemoi_transform_b200 import _cabi

    if not _cabi.library_path().exists():
        import importlib.util

        spec = importlib.util.spec_from_file_location("at_b200_build", REPO / "anemoi-transform_b200" / "build.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()


@pytest.fixture(scope="session")
def native_library():
    _ensure_library()
    from anemoi_transform_b200 import _cabi

    return _cabi.load()


@pytest.fixture(scope="session")
def cuda(native_library):
    import torch

    if not torch.cuda.is_available():
        pytest.fail("a test marked `gpu` ran without a CUDA device")
    return torch


@pytest.fixture(scope="session")
def golden_spatial():
    return dict(np.load(GOLDEN / "spatial_small.npz"))


@pytest.fixture(scope="session")
def golden_regrid():
    return dict(np.load(GOLDEN / "regrid_small.npz"))


@pytest.fixture(scope="session")
def golden_filters():
    d = dict(np.load(GOLDEN / "filters.npz"))
    d["order"] = json.loads(str(d["order"]))
    return d


def assert_same_values(actual: np.ndarray, expected: np.ndarray, what: str = ""):
    """Bit-exact on every non-NaN element and NaN in exactly the same places.

    (NaN payload / sign bits are not compared: x86 and the GPU canonicalise NaNs differently.)
    """
    actual, expected = np.asarray(actual), np.asarray(expected)
    assert actual.shape == expected.shape, (what, actual.shape, expected.shape)
    assert actual.dtype == expected.dtype, (what, actual.dtype, expected.dtype)
    nan_a, nan_e = np.isnan(actual), np.isnan(expected)
    assert np.array_equal(nan_a, nan_e), f"{what}: NaN positions differ ({nan_a.sum()} vs {nan_e.sum()})"
    view = {4: np.uint32, 8: np.uint64}[actual.dtype.itemsize]
    a, e = actual[~nan_a].view(view), expected[~nan_e].view(view)
    bad = np.nonzero(a != e)[0]
    assert bad.size == 0, f"{what}: {bad.size} of {a.size} elements differ bitwise, first at {bad[:5]}"


def assert_close_to_range(actual, expected, rel=1e-6, what="", circular=None):
    """|actual - expected| <= rel · (range of expected), NaN / inf in the same places.

    `circular`: period for angle-like fields (0 and 360 are the same direction)."""
    actual, expected = np.asarray(actual, dtype=np.float64), np.asarray(expected, dtype=np.float64)
    assert actual.shape == expected.shape, (what, actual.shape, expected.shape)
    assert np.array_equal(np.isnan(actual), np.isnan(expected)), f"{what}: NaN positions differ"
    inf = np.isinf(expected)
    assert np.array_equal(actual[inf], expected[inf]), f"{what}: infinities differ"
    ok = ~(np.isnan(expected) | inf)
    if not ok.any():
        return
    rng = float(expected[ok].max() - expected[ok].min()) or float(np.abs(expected[ok]).max()) or 1.0
    diff = np.abs(actual[ok] - expected[ok])
    if circular:
        diff = np.minimum(diff, circular - diff)
        rng = circular
    worst = diff.max()
    assert worst <= rel * rng, f"{what}: max |diff| {worst:.3e} > {rel:g} x range {rng:.3e}"


@pytest.fixture(scope="session")
def golden_filters_more():
    d = dict(np.load(GOLDEN / "filters_more.npz"))
    d["order"] = json.loads(str(d["order"]))
    return d
