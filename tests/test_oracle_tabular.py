"""oracle/tabular.py against the reference's superob: its outputs stored in
tests/golden/reference_checks.npz (oracle/make_golden.py), and live when ANEMOI_REFERENCE_SRC
points at the reference's sources."""

import numpy as np
import pytest
from conftest import GOLDEN

from anemoi_transform_b200 import synthetic as syn
from oracle import make_golden as mg
from oracle import reference_import
from oracle import tabular as ot


def _oracle(obs, grid):
    clean = obs.dropna(subset=["latitude"])
    binned = ot.assign_nearest_grid(clean, grid, 3600)
    result = ot.superob(obs.copy(), grid, 3600, take_nearest=["date"], groupby=["reporttype"])
    return clean, binned, result


def test_superob_restatement_equals_the_reference():
    grid, obs = mg.superob_case(syn)
    stored = np.load(GOLDEN / "reference_checks.npz")
    clean, binned, got = _oracle(obs, grid)
    assert binned.equals(mg.stored_frame(stored, "binned", base=clean))
    want = mg.stored_frame(stored, "superob")
    assert list(want.columns) == list(got.columns) and len(want) == len(got)
    assert want.equals(got.reset_index(drop=True))


@pytest.mark.reference
@pytest.mark.skipif(not reference_import.available(), reason="reference sources not present")
def test_superob_restatement_equals_the_reference_live(monkeypatch):
    reference_import.load()
    import importlib

    ref_support = importlib.import_module("anemoi.transform.filters.tabular.support.superob")
    ref_filter = importlib.import_module("anemoi.transform.filters.tabular.superob")
    grid, obs = mg.superob_case(syn)
    monkeypatch.setattr(ref_filter, "define_grid", lambda name: grid)  # the named-grid download is not the arithmetic
    clean, mine, got = _oracle(obs, grid)
    binned = ref_support.assign_nearest_grid(clean, grid, 3600)
    assert binned.equals(mine)
    want = ref_filter.SuperOb(grid="o6", **mg.SUPEROB_ARGS).forward(obs.copy())
    assert list(want.columns) == list(got.columns) and len(want) == len(got)
    assert want.reset_index(drop=True).equals(got.reset_index(drop=True))
    stored = np.load(GOLDEN / "reference_checks.npz")
    assert binned.equals(mg.stored_frame(stored, "binned", base=clean))
    assert want.reset_index(drop=True).equals(mg.stored_frame(stored, "superob"))
