"""HEALPix grids (`synthetic.healpix`, `grids.lookup`, `regrid_files.healpix_grid_of`) and the
pixel-exact conservative oracle oracle/healpix_conservative.py, pinned by its defining
properties and by an independent Monte-Carlo estimate (CPU)."""

import math

import numpy as np
import pytest
from scipy.sparse import csr_array

from anemoi_transform_b200 import synthetic as syn
from anemoi_transform_b200.filters.fields.regrid import as_griddata
from anemoi_transform_b200.grids import lookup
from anemoi_transform_b200.regrid_files import healpix_grid_of
from oracle import healpix as hp
from oracle import healpix_conservative as hc


def test_closed_form_centres():
    for n in (1, 2, 3, 4, 16):
        lat, lon = syn.healpix(n)
        z = np.sin(np.deg2rad(lat))
        assert lat.size == 12 * n * n
        assert z[0] == pytest.approx(1 - 1 / (3 * n * n), abs=1e-15) and lon[0] == 45.0
        starts = np.flatnonzero(np.concatenate(([True], lat[1:] != lat[:-1])))
        counts = np.diff(np.append(starts, lat.size))
        assert counts.size == 4 * n - 1
        expect = [4 * i if i < n else (4 * n if i <= 3 * n else 4 * (4 * n - i)) for i in range(1, 4 * n)]
        assert counts.tolist() == expect
        assert lat[starts[2 * n - 1]] == 0.0  # ring 2n is the equator
        assert (lon >= 0).all() and (lon < 360).all()
        zo, phio = hp.centres(n)
        np.testing.assert_allclose(z, zo, atol=1e-14)
        np.testing.assert_allclose(np.deg2rad(lon), phio, atol=1e-13)


@pytest.mark.parametrize("n", [1, 2, 4, 64, 1024])
def test_ring_nested_round_trips(n):
    all_ = np.arange(12 * n * n)
    r2n = syn.healpix_ring2nest(n, all_)
    assert (syn.healpix_nest2ring(n, r2n) == all_).all()
    assert np.unique(r2n).size == all_.size
    sample = all_ if n <= 64 else np.random.default_rng(n).choice(all_, 4000, replace=False)
    assert (hp.nest2ring(n, sample) == syn.healpix_nest2ring(n, sample)).all()
    lat_r, lon_r = syn.healpix(n, "ring")
    lat_n, lon_n = syn.healpix(n, "nested")
    ring = syn.healpix_nest2ring(n, all_)
    assert np.array_equal(lat_n, lat_r[ring]) and np.array_equal(lon_n, lon_r[ring])


@pytest.mark.parametrize("n", [1, 2, 4, 8, 64])
def test_ang2pix_inverts_pix2ang(n):
    z, phi = hp.centres(n)
    assert (hp.ang2pix_ring(n, z, phi) == np.arange(12 * n * n)).all()
    nest = hp.ang2pix_nest(n, z, phi)
    assert (hp.nest2ring(n, nest) == np.arange(12 * n * n)).all()


@pytest.mark.parametrize("n", [1, 3, 8, 48])
def test_every_pixel_area(n):
    for r in range(12 * n * n):
        i, p = hp.ring_of(n, r)
        assert hp.shoelace(hp.diamond(n, i, p, 0.0, 0.0)) == pytest.approx(2.0 / (n * n), rel=1e-15)


def _areas(grid):
    if grid[0] == "healpix":
        return np.full(12 * grid[1] ** 2, 2.0 / grid[1] ** 2)
    zn, zs, _, first, count = grid[1:]
    a = np.empty(int(count.sum()))
    for k in range(len(zn)):
        a[first[k] : first[k] + count[k]] = 12.0 * (zn[k] - zs[k]) / count[k]
    return a


def _grid(name, target):
    if name.startswith("H"):
        return hc.healpix_grid(int(name[1:]))
    lat, lon = syn.regular_latlon(10.0) if name == "10deg" else syn.octahedral(16)
    return hc.box_grid(lat, lon, target)


@pytest.mark.parametrize("a,b", [("H8", "10deg"), ("H16", "O16"), ("H12", "H8")])
def test_rows_sum_to_one_and_area_is_kept(a, b):
    for s, t in ((a, b), (b, a)):
        src, tgt = _grid(s, False), _grid(t, True)
        d, i, p, shape = hc.matrix(src, tgt, weights_dtype=np.float64)
        m = csr_array((d, i, p), shape=shape)
        np.testing.assert_allclose(m.sum(axis=1), 1.0, rtol=0, atol=1e-12)
        np.testing.assert_allclose(_areas(tgt) @ m, _areas(src), rtol=1e-9, atol=0)
        for r in range(shape[0]):
            assert (np.diff(i[p[r] : p[r + 1]]) > 0).all()


@pytest.mark.parametrize("k", [2, 3])
def test_nesting_is_exact(k):
    n = 4
    d, i, p, _ = hc.matrix(hc.healpix_grid(n), hc.healpix_grid(k * n))
    assert (np.diff(p) == 1).all() and (d == np.float32(1.0)).all()
    d, i, p, _ = hc.matrix(hc.healpix_grid(k * n), hc.healpix_grid(n))
    assert (np.diff(p) == k * k).all() and (d == np.float32(1.0 / (k * k))).all()


def _monte_carlo(src_class, tgt_class, n_src, n_tgt, m, n_points=10_000_000, seed=0):
    rng = np.random.default_rng(seed)
    z = rng.uniform(-1.0, 1.0, n_points)
    phi = rng.uniform(0.0, 2 * np.pi, n_points)
    s, t = src_class(z, phi), tgt_class(z, phi)
    joint = csr_array((np.ones(n_points), (t, s)), shape=(n_tgt, n_src)).toarray()
    count_t = joint.sum(axis=1, keepdims=True)
    frac = joint / count_t
    sigma = np.sqrt(np.maximum(frac * (1 - frac), 1.0 / count_t) / count_t)
    w = m.toarray()
    assert (np.abs(w - frac) <= 5 * sigma + 1e-7).all(), np.abs((w - frac) / sigma).max()


def _box_classifier(lat, lon):
    rows = hc.structured_rows(lat, lon)
    z_edges = np.concatenate(([1.0], hc.box_tables(rows)[1]))

    def classify(z, phi):
        k = np.searchsorted(-z_edges, -z, side="right") - 1
        k = np.clip(k, 0, rows[0].size - 1)
        n, lon0, first = rows[3][k], rows[1][k], rows[2][k]
        d = 360.0 / n
        c = np.floor(np.mod(np.rad2deg(phi) - (lon0 - d / 2.0), 360.0) / d).astype(np.int64) % n
        return first + c

    return classify


def test_monte_carlo_h4_to_30deg():
    lat, lon = syn.regular_latlon(30.0)
    src, tgt = hc.healpix_grid(4), hc.box_grid(lat, lon, True)
    d, i, p, shape = hc.matrix(src, tgt, weights_dtype=np.float64)
    _monte_carlo(lambda z, phi: hp.ang2pix_ring(4, z, phi), _box_classifier(lat, lon), shape[1], shape[0], csr_array((d, i, p), shape=shape))


def test_monte_carlo_o8_to_h4():
    lat, lon = syn.octahedral(8)
    src, tgt = hc.box_grid(lat, lon, False), hc.healpix_grid(4)
    d, i, p, shape = hc.matrix(src, tgt, weights_dtype=np.float64)
    _monte_carlo(_box_classifier(lat, lon), lambda z, phi: hp.ang2pix_ring(4, z, phi), shape[1], shape[0], csr_array((d, i, p), shape=shape))


def test_lookup_forms():
    ring = syn.healpix(8)
    nested = syn.healpix(8, "nested")
    for spec in ("H8", "h8", {"grid": "H8"}, {"grid": "H8", "ordering": "ring"}):
        g = lookup(spec)
        assert np.array_equal(g["latitudes"], ring[0]) and np.array_equal(g["longitudes"], ring[1])
    g = as_griddata({"grid": "H8", "ordering": "nested"})
    assert np.array_equal(g["latitudes"], nested[0]) and np.array_equal(g["longitudes"], nested[1])
    for bare, spec in (("O16", {"grid": "O16"}), ([10, 10], {"grid": [10, 10]})):
        a, b = lookup(bare), as_griddata(spec)
        assert np.array_equal(a["latitudes"], b["latitudes"]) and np.array_equal(a["longitudes"], b["longitudes"])


def test_lookup_refusals():
    with pytest.raises(ValueError, match="power-of-two"):
        lookup({"grid": "H12", "ordering": "nested"})
    with pytest.raises(ValueError, match="ordering"):
        lookup({"grid": "H8", "ordering": "peano"})
    with pytest.raises(ValueError, match="nside"):
        lookup("H20000")
    with pytest.raises(ValueError, match="'area'"):
        lookup({"grid": "H8", "area": [90, 0, -90, 360]})
    with pytest.raises(ValueError, match="'ordering'"):
        lookup({"grid": "O16", "ordering": "nested"})
    with pytest.raises(ValueError, match="Invalid grid"):
        as_griddata({"ordering": "ring"})


def test_healpix_grid_of():
    assert healpix_grid_of(*syn.healpix(16)) == (16, "ring")
    assert healpix_grid_of(*syn.healpix(16, "nested")) == (16, "nested")
    assert healpix_grid_of(*syn.healpix(12)) == (12, "ring")
    lat, lon = syn.healpix(16)
    assert healpix_grid_of(lat, lon - 360.0) == (16, "ring")  # longitudes compared mod 360
    spacing = math.degrees(math.sqrt(4 * math.pi / lat.size))
    assert healpix_grid_of(lat + 1e-8 * spacing, lon) == (16, "ring")
    assert healpix_grid_of(lat + 1e-4 * spacing, lon) is None
    order = np.random.default_rng(0).permutation(lat.size)
    assert healpix_grid_of(lat[order], lon[order]) is None
    assert healpix_grid_of(*syn.octahedral(16)) is None
    assert healpix_grid_of(lat[:-1], lon[:-1]) is None


def test_builder_refuses_grids_it_cannot_take(monkeypatch):
    from anemoi_transform_b200 import device
    from anemoi_transform_b200.regrid_files import make_healpix_conservative_matrix

    monkeypatch.setattr(device, "require_cuda", lambda: pytest.fail("reached the device"))
    h8 = syn.healpix(8)
    with pytest.raises(ValueError, match="structured-conservative"):
        make_healpix_conservative_matrix(*syn.octahedral(8), *syn.octahedral(16))
    lat, lon = syn.regular_latlon(10.0)
    band = np.abs(lat) <= 60
    with pytest.raises(ValueError, match="not global"):
        make_healpix_conservative_matrix(*h8, lat[band], lon[band])
    rng = np.random.default_rng(1)
    with pytest.raises(NotImplementedError, match="structured"):
        make_healpix_conservative_matrix(rng.uniform(-90, 90, 100), rng.uniform(0, 360, 100), *h8)
