"""The first-order conservative scheme (`method="structured-conservative"`): the numpy
restatement oracle/conservative_matrix.py that the device builder `at_conservative_matrix_*`
follows, pinned by a brute force over every pair of boxes and by the scheme's defining
properties, and the host's refusals.  CPU only."""

import numpy as np
import pytest
from scipy.sparse import csr_array

from anemoi_transform_b200 import synthetic as syn
from anemoi_transform_b200.regrid_files import box_z_edges, make_conservative_matrix, structured_grid_rows
from oracle import conservative_matrix as oc
from oracle import structured_matrix as om


def _cell_centred(step):
    lat = 90.0 - step / 2 - step * np.arange(int(round(180 / step)))
    lon = step / 2 + step * np.arange(int(round(360 / step)))
    return np.repeat(lat, lon.size), np.tile(lon, lat.size)


def _one_point_rows(south_to_north=True):
    """A hand-made global reduced grid with rows of 1, 2, 3 and 5 points, south → north, first
    longitudes off zero (a 1-point row's box is its whole band)."""
    row_lat, pl, lon0 = [-60.0, -20.0, 25.0, 70.0], [1, 2, 3, 5], [10.0, 0.0, 100.0, 350.0]
    if not south_to_north:
        row_lat, pl, lon0 = row_lat[::-1], pl[::-1], lon0[::-1]
    lat = np.repeat(row_lat, pl)
    lon = np.concatenate([l0 + np.arange(p) * (360.0 / p) for l0, p in zip(lon0, pl)])
    return lat, lon


def _rows(lat, lon):
    rows = om.structured_rows(lat, lon)
    om.check_global(rows)
    return rows


def _brute_force(s_lat, s_lon, t_lat, t_lon):
    """Dense [n_tgt, n_src] weights: every (target box, source box) pair intersected
    explicitly, longitude intervals compared at shifts of -360, 0 and 360 degrees."""

    def boxes(lat, lon):
        lats = np.unique(lat)[::-1]
        edges = np.concatenate(([90.0], (lats[:-1] + lats[1:]) / 2.0, [-90.0]))
        z = np.sin(np.deg2rad(edges))
        k = np.searchsorted(-lats, -lat)
        width = 360.0 / np.bincount(k)[k]
        return z[k], z[k + 1], np.mod(lon - width / 2.0, 360.0), width

    zn_t, zs_t, w_t, d_t = boxes(t_lat, t_lon)
    zn_s, zs_s, w_s, d_s = boxes(s_lat, s_lon)
    m = np.zeros((t_lat.size, s_lat.size))
    for t in range(t_lat.size):
        for s in range(s_lat.size):
            dz = min(zn_t[t], zn_s[s]) - max(zs_t[t], zs_s[s])
            if dz <= 0.0:
                continue
            lon = sum(max(0.0, min(w_t[t] + d_t[t], w_s[s] + shift + d_s[s]) - max(w_t[t], w_s[s] + shift)) for shift in (-360.0, 0.0, 360.0))
            m[t, s] = dz / (zn_t[t] - zs_t[t]) * lon / d_t[t]
    return m


TINY = {
    "o4": lambda: syn.octahedral(4),
    "30deg": lambda: syn.regular_latlon(30.0),
    "15deg-cell-centred": lambda: _cell_centred(15.0),
    "1-2-3-5-points": _one_point_rows,
}


@pytest.mark.parametrize(
    "source,target",
    [("o4", "30deg"), ("30deg", "o4"), ("15deg-cell-centred", "o4"), ("o4", "15deg-cell-centred"), ("1-2-3-5-points", "30deg"), ("o4", "1-2-3-5-points"), ("1-2-3-5-points", "1-2-3-5-points")],
)
def test_oracle_equals_a_brute_force_over_every_pair_of_boxes(source, target):
    s_lat, s_lon = TINY[source]()
    t_lat, t_lon = TINY[target]()
    d, i, p, shape = oc.conservative_matrix(_rows(s_lat, s_lon), _rows(t_lat, t_lon), weights_dtype=np.float64)
    got = csr_array((d, i, p), shape=shape)
    assert got.has_canonical_format  # columns ascending and unique in every row
    want = _brute_force(s_lat, s_lon, t_lat, t_lon)
    assert np.abs(got.toarray() - want).max() <= 1e-12
    assert (d > 0).all()  # no explicit zeros


@pytest.mark.parametrize(
    "source,target",
    [(lambda: syn.octahedral(48), lambda: syn.regular_latlon(2.5)), (lambda: syn.regular_latlon(1.0), lambda: syn.octahedral(24)), (_one_point_rows, lambda: syn.octahedral(16)), (lambda: syn.octahedral(16), _one_point_rows)],
)
def test_rows_sum_to_one_within_float32_rounding(source, target):
    d, i, p, shape = oc.conservative_matrix(_rows(*source()), _rows(*target()))
    assert d.dtype == np.float32 and i.dtype == np.int32 and p.dtype == np.int32
    sums = np.add.reduceat(d.astype(np.float64), p[:-1])
    assert (np.abs(sums - 1.0) <= np.diff(p) * 2.0**-24 + 1e-12).all()


@pytest.mark.parametrize("grid", [lambda: syn.octahedral(24), lambda: syn.regular_latlon(2.0)])
def test_a_grid_onto_itself_is_the_identity(grid):
    lat, lon = grid()
    rows = _rows(lat, lon)
    d, i, p, shape = oc.conservative_matrix(rows, rows)
    assert np.array_equal(p, np.arange(lat.size + 1)) and np.array_equal(i, np.arange(lat.size))
    assert (d == np.float32(1.0)).all()


def test_a_nested_grid_takes_its_two_by_two_sub_boxes():
    s_lat, s_lon = _cell_centred(1.0)
    t_lat, t_lon = _cell_centred(2.0)
    s_rows, t_rows = _rows(s_lat, s_lon), _rows(t_lat, t_lon)
    d, i, p, shape = oc.conservative_matrix(s_rows, t_rows)
    assert np.array_equal(p, 4 * np.arange(t_lat.size + 1))
    zn_s, zs_s = oc.box_tables(s_rows)
    zn_t, zs_t = oc.box_tables(t_rows)
    t = np.arange(t_lat.size)
    r, c = t // 180, t % 180  # 2° rows of 180 boxes; 1° rows of 360
    want_cols = np.stack([720 * r + 2 * c, 720 * r + 2 * c + 1, 720 * r + 360 + 2 * c, 720 * r + 361 + 2 * c], axis=1)
    assert np.array_equal(i.reshape(-1, 4), want_cols)
    dz_t = zn_t[r] - zs_t[r]
    half = [(zn_s[2 * r] - zs_s[2 * r]) / dz_t * 0.5, (zn_s[2 * r + 1] - zs_s[2 * r + 1]) / dz_t * 0.5]
    want = np.stack([half[0], half[0], half[1], half[1]], axis=1).astype(np.float32)
    ulps = np.abs(d.reshape(-1, 4).view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1


def _positive_smooth(lat, lon):
    p, l = np.deg2rad(lat), np.deg2rad(lon)
    x, y, z = np.cos(p) * np.cos(l), np.cos(p) * np.sin(l), np.sin(p)
    return 5.0 + x + 2 * y + 3 * z + x * y + z * z


def _box_areas(rows):
    zn, zs = oc.box_tables(rows)
    area = np.empty(int(rows[3].sum()))
    for k in range(rows[0].size):
        area[rows[2][k] : rows[2][k] + rows[3][k]] = (zn[k] - zs[k]) * (2.0 * np.pi / rows[3][k])
    return area


@pytest.mark.parametrize("source,target", [(lambda: syn.octahedral(48), lambda: syn.regular_latlon(2.5)), (lambda: syn.regular_latlon(1.0), lambda: syn.octahedral(24))])
def test_the_area_integral_is_kept(source, target):
    s_lat, s_lon = source()
    t_lat, t_lon = target()
    s_rows, t_rows = _rows(s_lat, s_lon), _rows(t_lat, t_lon)
    m = csr_array(oc.conservative_matrix(s_rows, t_rows)[:3], shape=(t_lat.size, s_lat.size))
    x = _positive_smooth(s_lat, s_lon)
    y = m @ x
    a_s, a_t = _box_areas(s_rows), _box_areas(t_rows)
    assert abs(a_s.sum() - 4 * np.pi) < 1e-12 and abs(a_t.sum() - 4 * np.pi) < 1e-12  # the boxes tile the sphere
    assert abs((a_t * y).sum() - (a_s * x).sum()) <= 2e-6 * (a_s * x).sum()


def test_host_z_tables_are_the_oracles():
    for lat, lon in (syn.octahedral(32), syn.regular_latlon(1.5), _one_point_rows()):
        rows = structured_grid_rows(lat, lon)
        z = box_z_edges(rows[0])
        zn, zs = oc.box_tables(om.structured_rows(lat, lon))
        assert np.array_equal(z[:-1], zn) and np.array_equal(z[1:], zs)


def test_the_host_refuses_grids_the_scheme_cannot_take():
    s_lat, s_lon = syn.octahedral(16)
    t_lat, t_lon = syn.regular_latlon(10.0)
    rng = np.random.default_rng(0)
    shuffle_s, shuffle_t = rng.permutation(s_lat.size), rng.permutation(t_lat.size)
    with pytest.raises(NotImplementedError, match="structured-conservative.*source"):
        make_conservative_matrix(s_lat[shuffle_s], s_lon[shuffle_s], t_lat, t_lon)
    with pytest.raises(NotImplementedError, match="structured-conservative.*target"):
        make_conservative_matrix(s_lat, s_lon, t_lat[shuffle_t], t_lon[shuffle_t])
    b_lat, b_lon = syn.regular_latlon(2.0)
    band = np.abs(b_lat) <= 60.0
    with pytest.raises(ValueError, match="source grid is not global"):
        make_conservative_matrix(b_lat[band], b_lon[band], t_lat, t_lon)
    with pytest.raises(ValueError, match="target grid is not global"):
        make_conservative_matrix(s_lat, s_lon, b_lat[band], b_lon[band])
    with pytest.raises(ValueError, match=r"\[-90, 90\]"):
        make_conservative_matrix(s_lat, s_lon, np.repeat([95.0, 45.0, 0.0, -45.0, -90.0], 4), np.tile(np.arange(4) * 90.0, 5))


def test_host_api_without_a_gpu_fails_loudly(native_library):
    import torch

    from anemoi_transform_b200._cabi import NativeLibraryError

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible: the builder runs (tests/test_gpu_conservative_matrix.py)")
    with pytest.raises(NativeLibraryError):
        make_conservative_matrix(*syn.octahedral(16), *syn.regular_latlon(10.0))
