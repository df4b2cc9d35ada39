"""The structured-grid stencils (`method="structured-bilinear" | "structured-bicubic"`): row
detection (`regrid_files.structured_grid_rows`, restated by oracle/structured_matrix.py::structured_rows)
and the numpy restatement of the weights the device builder `at_structured_matrix` follows,
pinned by the scheme's defining properties.  CPU only."""

import numpy as np
import pytest
from scipy.sparse import csr_array

from anemoi_transform_b200 import synthetic as syn
from anemoi_transform_b200.regrid_files import make_structured_matrix, structured_grid_rows
from oracle import structured_matrix as om


def _smooth(lat, lon):
    """x + 2y + 3z + xy + z² on the unit sphere: smooth, with no special value at the poles."""
    p, l = np.deg2rad(lat), np.deg2rad(lon)
    x, y, z = np.cos(p) * np.cos(l), np.cos(p) * np.sin(l), np.sin(p)
    return x + 2 * y + 3 * z + x * y + z * z


def _cell_centred(step):
    lat = 90.0 - step / 2 - step * np.arange(int(round(180 / step)))
    lon = step / 2 + step * np.arange(int(round(360 / step)))
    return np.repeat(lat, lon.size), np.tile(lon, lat.size)


def _full_gaussian(n):
    lat = syn.gaussian_latitudes(n)
    return np.repeat(lat, 4 * n), np.tile(np.arange(4 * n) * (360.0 / (4 * n)), lat.size)


def _south_to_north(lat, lon):
    """The same grid with its rows stored south → north (each row still west → east)."""
    starts = np.flatnonzero(np.concatenate(([True], lat[1:] != lat[:-1])))
    bounds = np.append(starts, lat.size)
    order = np.concatenate([np.arange(a, b) for a, b in zip(bounds[-2::-1], bounds[:0:-1])])
    return lat[order], lon[order]


GRIDS = {
    "o16": lambda: syn.octahedral(16),
    "o16-south-to-north": lambda: _south_to_north(*syn.octahedral(16)),
    "n320-like": syn.n320_like,
    "regular-2deg-with-poles": lambda: syn.regular_latlon(2.0),
    "regular-cell-centred": lambda: _cell_centred(3.0),
    "full-gaussian-n24": lambda: _full_gaussian(24),
}


@pytest.mark.parametrize("name", sorted(GRIDS))
def test_row_detection_accepts_global_structured_grids(name):
    lat, lon = GRIDS[name]()
    rows = structured_grid_rows(lat, lon)
    assert rows is not None
    want = om.structured_rows(lat, lon)
    for a, b in zip(rows, want):
        assert a.dtype == b.dtype and np.array_equal(a, b)
    row_lat, lon0, first, count = rows
    assert (np.diff(row_lat) < 0).all() and count.sum() == lat.size
    assert np.array_equal(lat[first], row_lat) and np.array_equal(lon[first], lon0)
    om.check_global(rows)


def test_row_detection_rejects_what_is_not_a_structured_grid():
    lat, lon = syn.octahedral(16)
    shuffle = np.random.default_rng(0).permutation(lat.size)
    assert structured_grid_rows(lat[shuffle], lon[shuffle]) is None
    # rows that cover half the circle: 90 points 2° apart are not 360/90 = 4° apart
    h_lat, h_lon = syn.regular_latlon(2.0)
    half = h_lon < 180.0
    assert structured_grid_rows(h_lat[half], h_lon[half]) is None
    # one row's points out of place
    bad = lon.copy()
    bad[100] += 0.5
    assert structured_grid_rows(lat, bad) is None
    # non-monotone row latitudes: two rows swapped
    r_lat, r_lon = syn.regular_latlon(10.0)
    n_lon = 36
    swapped = np.concatenate([r_lat[: 3 * n_lon], r_lat[4 * n_lon : 5 * n_lon], r_lat[3 * n_lon : 4 * n_lon], r_lat[5 * n_lon :]])
    assert structured_grid_rows(swapped, r_lon) is None
    # a row latitude repeated further down
    repeated = np.concatenate([r_lat, r_lat[n_lon : 2 * n_lon]])
    assert structured_grid_rows(repeated, np.concatenate([r_lon, r_lon[:n_lon]])) is None
    for rows in (structured_grid_rows(lat[shuffle], lon[shuffle]), om.structured_rows(lat[shuffle], lon[shuffle])):
        assert rows is None


def test_a_latitude_band_is_not_global():
    lat, lon = syn.regular_latlon(2.0)
    band = np.abs(lat) <= 60.0
    rows = structured_grid_rows(lat[band], lon[band])
    assert rows is not None  # structured, but it does not reach the poles
    with pytest.raises(ValueError, match="not global"):
        om.check_global(rows)
    for method in ("structured-bilinear", "structured-bicubic"):
        with pytest.raises(ValueError, match="not global"):
            make_structured_matrix(lat[band], lon[band], *syn.octahedral(16), method)


@pytest.mark.parametrize("stencil", [2, 4])
@pytest.mark.parametrize("source", ["o24", "regular-2deg-with-poles", "regular-cell-centred", "n320-like"])
def test_rows_sum_to_one_and_source_points_are_reproduced(stencil, source):
    s_lat, s_lon = syn.octahedral(24) if source == "o24" else GRIDS[source]()
    rows = om.structured_rows(s_lat, s_lon)
    t_lat, t_lon = syn.regular_latlon(1.0)
    t_lat, t_lon = np.concatenate([t_lat, [90.0, -90.0, 89.99, -89.99]]), np.concatenate([t_lon, [0.0, 17.0, 200.0, 359.99]])
    d, i, p, shape = om.structured_matrix(rows, t_lat, t_lon, stencil, weights_dtype=np.float64)
    m = csr_array((d, i, p), shape=shape)
    assert np.abs(m.sum(axis=1) - 1.0).max() <= 1e-15
    assert (np.diff(i.reshape(-1, stencil * stencil), axis=1) >= 0).all()  # sorted within a row
    # a target on a source point takes exactly that point's value (float32 matrix, float32 field)
    pick = np.random.default_rng(1).choice(s_lat.size, 3000, replace=False)
    d, i, p, shape = om.structured_matrix(rows, s_lat[pick], s_lon[pick], stencil)
    v = np.random.default_rng(2).standard_normal(s_lat.size).astype(np.float32)
    got = csr_array((d, i, p), shape=shape) @ v
    assert np.array_equal(got.view(np.uint32), v[pick].view(np.uint32))
    assert (d == 0).any()  # the explicit zeros are kept


def test_error_on_a_smooth_field_falls_with_resolution_and_bicubic_beats_bilinear():
    t_lat, t_lon = syn.regular_latlon(2.5)
    bounds = {2: [8e-3, 2e-3, 8e-4], 4: [4e-5, 1.6e-5, 7e-6]}
    errors = {2: [], 4: []}
    for n in (24, 48, 96):
        s_lat, s_lon = syn.octahedral(n)
        rows = om.structured_rows(s_lat, s_lon)
        for stencil in (2, 4):
            m = csr_array(om.structured_matrix(rows, t_lat, t_lon, stencil, weights_dtype=np.float64)[:3], shape=(t_lat.size, s_lat.size))
            errors[stencil].append(np.abs(m @ _smooth(s_lat, s_lon) - _smooth(t_lat, t_lon)).max())
    for stencil in (2, 4):
        assert all(e <= b for e, b in zip(errors[stencil], bounds[stencil])), (stencil, errors[stencil])
        assert errors[stencil][0] > errors[stencil][1] > errors[stencil][2]
    assert all(c < 0.05 * b for c, b in zip(errors[4], errors[2]))
    d = om.structured_matrix(om.structured_rows(*syn.octahedral(48)), t_lat, t_lon, 4, weights_dtype=np.float64)[0]
    assert d.min() < -0.1  # cubic weights go negative; no limiter


@pytest.mark.parametrize("stencil", [2, 4])
@pytest.mark.parametrize("source", ["o24", "regular-2deg-with-poles"])
def test_targets_poleward_of_the_outermost_rows_are_continuous(stencil, source):
    """Across the pole the stencil takes the outermost rows seen from the other side: values
    approach the field's own towards ±90°, without a jump where the stencil changes rows."""
    s_lat, s_lon = syn.octahedral(24) if source == "o24" else syn.regular_latlon(2.0)
    rows = om.structured_rows(s_lat, s_lon)
    f = _smooth(s_lat, s_lon)
    outer = rows[0][0]
    for lon in (0.0, 33.3, 181.0, 300.25):
        for sign in (1.0, -1.0):
            lats = sign * np.concatenate([np.linspace(rows[0][2], 90.0, 400), [outer - 1e-9, outer, outer + 1e-9]])
            lats = np.minimum(np.maximum(lats, -90.0), 90.0)
            d, i, p, shape = om.structured_matrix(rows, lats, np.full(lats.size, lon), stencil, weights_dtype=np.float64)
            got = csr_array((d, i, p), shape=shape) @ f
            want = _smooth(lats, np.full(lats.size, lon))
            assert np.abs(got - want).max() < (0.02 if stencil == 2 else 2e-4)
            assert np.abs(np.diff(got[:400])).max() < 0.01  # no jump along the sweep
            assert np.abs(got[-3] - got[-2]) < 1e-8 and np.abs(got[-1] - got[-2]) < 1e-8


def test_targets_outside_the_sphere_and_non_structured_sources_are_refused_on_the_host():
    s_lat, s_lon = syn.octahedral(16)
    with pytest.raises(ValueError, match=r"\[-90, 90\]"):
        make_structured_matrix(s_lat, s_lon, [90.5], [0.0], "structured-bicubic")
    with pytest.raises(ValueError, match=r"\[-90, 90\]"):
        make_structured_matrix(s_lat, s_lon, [np.nan], [0.0], "structured-bilinear")
    shuffle = np.random.default_rng(0).permutation(s_lat.size)
    with pytest.raises(NotImplementedError, match="structured-bilinear"):
        make_structured_matrix(s_lat[shuffle], s_lon[shuffle], [0.0], [0.0], "structured-bilinear")
    with pytest.raises(ValueError, match="not one of"):
        make_structured_matrix(s_lat, s_lon, [0.0], [0.0], "structured-linear")


def test_host_api_without_a_gpu_fails_loudly_and_detection_still_works(native_library):
    import torch

    from anemoi_transform_b200._cabi import NativeLibraryError

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible: the builder runs (tests/test_gpu_structured_matrix.py)")
    s_lat, s_lon = syn.octahedral(16)
    assert structured_grid_rows(s_lat, s_lon) is not None
    with pytest.raises(NativeLibraryError):
        make_structured_matrix(s_lat, s_lon, *syn.regular_latlon(10.0), "structured-bicubic")
