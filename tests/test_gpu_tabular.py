"""SURVEY §8(f) rank 3 remainder: `superob` (tabular kNN in the lat-lon plane) and
`icon_refinement_level` (nearest-neighbour gather to ICON cell centres)."""

import numpy as np
import pytest
from conftest import assert_same_values

from anemoi_transform_b200 import ekd
from anemoi_transform_b200 import synthetic as syn
from oracle import tabular as ot

pytestmark = pytest.mark.gpu


def test_superob_equals_the_ckdtree_pandas_restatement(cuda):
    from anemoi_transform_b200.filters import create_filter_by_name as F
    from anemoi_transform_b200.filters.tabular.assign_to_grid import define_grid
    from anemoi_transform_b200.filters.tabular.superob import assign_nearest_grid

    grid = define_grid("o6")
    obs = ot.synthetic_observations(20000, seed=1)
    obs.loc[::777, "longitude"] = np.nan
    clean = obs.dropna(subset=["date", "latitude", "longitude"])
    mine, want = assign_nearest_grid(clean, grid, 3600), ot.assign_nearest_grid(clean, grid, 3600)
    assert np.array_equal(mine["distance"].to_numpy(), want["distance"].to_numpy())  # bitwise cKDTree's
    differ = mine["spatial_index"].to_numpy() != want["spatial_index"].to_numpy()
    assert differ.sum() == 0  # random observations: no exact ties
    out = F("superob", grid="o6", timeslot_length=3600, columns_to_take_nearest=["date"], columns_to_groupby=["reporttype"]).forward(obs.copy())
    ref = ot.superob(obs.copy(), grid, 3600, take_nearest=["date"], groupby=["reporttype"])
    assert list(out.columns) == list(ref.columns)
    assert out.reset_index(drop=True).equals(ref.reset_index(drop=True))
    # "native" and empty inputs pass through
    assert F("superob", grid="native", timeslot_length=60).forward(obs) is obs
    assert len(F("superob", grid="o6", timeslot_length=60).forward(obs.iloc[:0])) == 0


def test_superob_matches_the_reference_outputs(cuda, monkeypatch):
    """The reference's binning and superob result (tests/golden/reference_checks.npz)."""
    from conftest import GOLDEN

    from anemoi_transform_b200.filters import create_filter_by_name as F
    from anemoi_transform_b200.filters.tabular import superob
    from oracle import make_golden as mg

    stored = np.load(GOLDEN / "reference_checks.npz")
    grid, obs = mg.superob_case(syn)
    clean = obs.dropna(subset=["latitude"])
    binned, want = mg.stored_frame(stored, "binned", base=clean), mg.stored_frame(stored, "superob")
    mine = superob.assign_nearest_grid(clean, grid, 3600)
    for c in ("grid_index", "spatial_index", "distance"):
        assert np.array_equal(mine[c].to_numpy(), binned[c].to_numpy()), c
    monkeypatch.setattr(superob, "define_grid", lambda name: grid)
    out = F("superob", grid="o6", **mg.SUPEROB_ARGS).forward(obs.copy())
    assert list(out.columns) == list(want.columns)
    assert out.reset_index(drop=True).equals(want)


def test_icon_refinement_level_gathers_the_nearest_cells(cuda, tmp_path):
    from scipy.spatial import cKDTree

    from anemoi_transform_b200.filters import create_filter_by_name as F
    from oracle import spatial as osp

    # an "ICON grid file": cell centres in radians with a refinement level per cell
    rng = np.random.default_rng(0)
    n_cells = 5000
    clat = np.arcsin(rng.uniform(-1, 1, n_cells))
    clon = rng.uniform(-np.pi, np.pi, n_cells)
    level = rng.integers(0, 4, n_cells)
    np.savez(tmp_path / "icon.npz", clat=clat, clon=clon, refinement_level_c=level)
    s_lat, s_lon = syn.regular_latlon(2.0)
    values = [syn.synthetic_field("t", s_lat.size, k, 0.002 if k == 1 else 0.0) for k in range(5)]
    values[3] = values[3].astype(np.float64)
    data = ekd.from_source("list-of-dicts", [dict(param="t", levelist=850, step=k, values=v, latitudes=s_lat, longitudes=s_lon) for k, v in enumerate(values)])
    for lev in (None, 2):
        flt = F("icon_refinement_level", grid=str(tmp_path / "icon.npz"), refinement_level_c=lev)
        keep = slice(None) if lev is None else level <= lev
        t_lat, t_lon = np.rad2deg(clat[keep]), np.rad2deg(clon[keep])
        assert np.array_equal(flt.latitudes, t_lat) and np.array_equal(flt.longitudes, t_lon)
        out = flt.forward(data)
        dist, idx = cKDTree(np.array(osp.latlon_to_xyz(s_lat, s_lon)).T).query(np.array(osp.latlon_to_xyz(t_lat, t_lon)).T)
        mine = flt.nearest_grid_points
        # equal wherever the nearest source is unique; a tie still returns a source at that distance
        sx = np.array(osp.latlon_to_xyz(s_lat, s_lon)).T
        tx = np.array(osp.latlon_to_xyz(t_lat, t_lon)).T
        assert np.array_equal(np.sqrt(((sx[mine] - tx) ** 2).sum(axis=1)), dist) or np.allclose(np.linalg.norm(sx[mine] - tx, axis=1), dist, rtol=0, atol=1e-15)
        for k, f in enumerate(out):
            assert_same_values(f.to_numpy(), values[k][mine], f"field {k}")
            assert np.array_equal(f.grid_points()[0], t_lat)
        assert (mine != idx).mean() < 0.01
