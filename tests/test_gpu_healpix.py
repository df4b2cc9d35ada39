"""`method="healpix-conservative"` (`at_healpix_conservative_count` / `_fill`) against the
restatement oracle/healpix_conservative.py bit for bit, nested HEALPix grids through
`at_healpix_reorder`, the structured stencils on HEALPix sources, and the `regrid` recipe on
numpy and GRIB-backed FieldLists."""

import ctypes

import numpy as np
import pytest
from conftest import assert_same_values
from grib_fields import GribMessageField
from scipy.sparse import csr_array

from anemoi_transform_b200 import ekd
from anemoi_transform_b200 import synthetic as syn
from oracle import grib as ogrib
from oracle import grib_ccsds as ogc
from oracle import healpix_conservative as hc
from oracle.spmm_missing import ALL, csr_matvec_missing

pytestmark = pytest.mark.gpu

METHOD = "healpix-conservative"


@pytest.fixture(scope="module")
def F(cuda):
    from anemoi_transform_b200.filters import create_filter_by_name

    return create_filter_by_name


def _one_point_rows():
    """Rows of 1, 2, 3 and 5 points, stored south → north, first longitudes off zero."""
    row_lat, pl, lon0 = [-60.0, -20.0, 25.0, 70.0], [1, 2, 3, 5], [10.0, 0.0, 100.0, 350.0]
    return np.repeat(row_lat, pl), np.concatenate([l0 + np.arange(p) * (360.0 / p) for l0, p in zip(lon0, pl)])


def _points(name):
    """Point lists and the oracle's grid description (source and target forms)."""
    if name.startswith("H"):
        nside, _, ordering = name[1:].partition("-")
        ordering = ordering or "ring"
        lat, lon = syn.healpix(int(nside), ordering)
        return lat, lon, hc.healpix_grid(int(nside), ordering), hc.healpix_grid(int(nside), ordering)
    if name == "1235":
        lat, lon = _one_point_rows()
    elif name.startswith("O"):
        lat, lon = syn.octahedral(int(name[1:]))
    else:
        lat, lon = syn.regular_latlon(float(name.rstrip("deg")))
    return lat, lon, hc.box_grid(lat, lon, False), hc.box_grid(lat, lon, True)


def _build(source, target):
    from anemoi_transform_b200.regrid_files import make_healpix_conservative_matrix

    s_lat, s_lon, s_grid, _ = _points(source)
    t_lat, t_lon, _, t_grid = _points(target)
    got = make_healpix_conservative_matrix(s_lat, s_lon, t_lat, t_lon)
    return got, s_grid, t_grid


def _assert_rows_equal(got, want, rows):
    d, i, p, _ = got
    wd, wi, wp, _ = want
    for k, r in enumerate(rows):
        a, b = slice(p[r], p[r + 1]), slice(wp[k], wp[k + 1])
        assert np.array_equal(i[a], wi[b]), f"row {r}: columns differ"
        assert np.array_equal(d[a].view(np.uint32), wd[b].view(np.uint32)), f"row {r}: weights differ bitwise"


CASES = [
    ("H8", "10deg"),
    ("5deg", "H16-nested"),
    ("O96", "H64"),
    ("O96", "H64-nested"),
    ("H128-nested", "O96"),
    ("H32", "H48"),
    ("H48", "H32"),
    ("1235", "H8"),
    ("H8", "1235"),
]


@pytest.mark.parametrize("source,target", CASES)
def test_device_matrix_is_bitwise_the_oracle(cuda, source, target):
    got, s_grid, t_grid = _build(source, target)
    want = hc.matrix(s_grid, t_grid)
    assert got[3] == want[3]
    d, i, p, _ = got
    assert d.dtype == np.float32 and i.dtype == np.int32 and p.dtype == np.int32
    assert np.array_equal(p, want[2]) and np.array_equal(i, want[1])
    bad = np.flatnonzero(d.view(np.uint32) != want[0].view(np.uint32))
    assert bad.size == 0, f"{bad.size} weights differ bitwise, first at entries {bad[:5]}"
    for r in range(got[3][0]):
        assert (np.diff(i[p[r] : p[r + 1]]) > 0).all()


def _areas(lat, lon):
    from anemoi_transform_b200.regrid_files import healpix_grid_of

    hp = healpix_grid_of(lat, lon)
    if hp is not None:
        return np.full(lat.size, 4.0 * np.pi / lat.size)
    grid = hc.box_grid(lat, lon, False)
    zn, zs, _, first, count = grid[1:]
    a = np.empty(lat.size)
    for k in range(len(zn)):
        a[first[k] : first[k] + count[k]] = (zn[k] - zs[k]) * 2.0 * np.pi / count[k]
    return a


@pytest.mark.parametrize("source,target", [("H1024-nested", "O96"), ("O1280", "H256")])
def test_full_size_matches_the_oracle_on_a_sample_and_keeps_the_area_integral(cuda, source, target):
    got, s_grid, t_grid = _build(source, target)
    rows = np.sort(np.random.default_rng(2000).choice(got[3][0], 2000, replace=False))
    _assert_rows_equal(got, hc.matrix(s_grid, t_grid, rows=rows), rows)
    s_lat, s_lon = _points(source)[:2]
    t_lat, t_lon = _points(target)[:2]
    m = csr_array(got[:3], shape=got[3])
    ph, la = np.deg2rad(s_lat), np.deg2rad(s_lon)
    x = 5.0 + np.cos(ph) * np.cos(la) + 3.0 * np.sin(ph) + np.cos(ph) ** 2 * np.sin(3 * la)
    a_s, a_t = _areas(s_lat, s_lon), _areas(t_lat, t_lon)
    assert abs((a_t * (m @ x)).sum() - (a_s * x).sum()) <= 2e-6 * (a_s * x).sum()


def test_nested_matrices_are_the_ring_matrices_permuted(cuda):
    n = 32
    r2n = syn.healpix_ring2nest(n, np.arange(12 * n * n))
    ring, _, _ = _build(f"H{n}", "O32")
    nested, _, _ = _build(f"H{n}-nested", "O32")
    a = csr_array(ring[:3], shape=ring[3])
    b = csr_array(nested[:3], shape=nested[3])
    perm = csr_array((np.ones(r2n.size), (r2n, np.arange(r2n.size))), shape=(r2n.size, r2n.size))  # ring column c → nested r2n[c]
    want = (a @ perm.T).tocsr()
    want.sort_indices()
    assert np.array_equal(b.indptr, want.indptr) and np.array_equal(b.indices, want.indices)
    assert np.array_equal(b.data.astype(np.float32).view(np.uint32), want.data.astype(np.float32).view(np.uint32))

    ring, _, _ = _build("O32", f"H{n}")
    nested, _, _ = _build("O32", f"H{n}-nested")
    n2r = syn.healpix_nest2ring(n, np.arange(12 * n * n))
    for t in (0, 5, 777, 6000, 12287):
        r = n2r[t]
        assert np.array_equal(nested[1][nested[2][t] : nested[2][t + 1]], ring[1][ring[2][r] : ring[2][r + 1]])
        assert np.array_equal(nested[0][nested[2][t] : nested[2][t + 1]].view(np.uint32), ring[0][ring[2][r] : ring[2][r + 1]].view(np.uint32))


@pytest.mark.parametrize("method", ["structured-bilinear", "structured-bicubic"])
def test_structured_stencils_on_ring_and_nested_sources(cuda, method):
    from anemoi_transform_b200.grids import lookup
    from anemoi_transform_b200.regrid_files import make_structured_matrix

    n = 32
    t_lat, t_lon = syn.octahedral(24)
    g = lookup(f"H{n}")
    d, i, p, shape = make_structured_matrix(g["latitudes"], g["longitudes"], t_lat, t_lon, method)
    assert np.abs(csr_array((d, i, p), shape=shape).sum(axis=1) - 1.0).max() < 1e-5
    g = lookup({"grid": f"H{n}", "ordering": "nested"})
    dn, in_, pn, shape_n = make_structured_matrix(g["latitudes"], g["longitudes"], t_lat, t_lon, method)
    assert shape_n == shape and np.array_equal(pn, p)
    r2n = syn.healpix_ring2nest(n, i)
    for r in range(shape[0]):
        o = np.argsort(r2n[p[r] : p[r + 1]], kind="stable")
        assert np.array_equal(in_[pn[r] : pn[r + 1]], r2n[p[r] : p[r + 1]][o])
        assert np.array_equal(dn[pn[r] : pn[r + 1]].view(np.uint32), d[p[r] : p[r + 1]][o].view(np.uint32))


def _oracle_csr(source, target):
    _, _, s_grid, _ = _points(source)
    _, _, _, t_grid = _points(target)
    d, i, p, shape = hc.matrix(s_grid, t_grid)
    return csr_array((d, i, p), shape=shape)


IN_GRID = {"grid": "H64", "ordering": "nested"}


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("missing", [None, "missing-if-all-missing"])
def test_regrid_numpy_fieldlists(F, dtype, missing):
    s_lat, s_lon = syn.healpix(64, "nested")
    m = _oracle_csr("H64-nested", "O32")
    values = [syn.synthetic_field("t", s_lat.size, s, 0.003 if missing and s % 2 else 0.0).astype(dtype) for s in range(5)]
    data = ekd.from_source("list-of-dicts", [dict(values=v, latitudes=s_lat, longitudes=s_lon, param="t", levelist=850, step=k) for k, v in enumerate(values)])
    kw = {} if missing is None else {"missing_values": missing}
    out = F("regrid", in_grid=IN_GRID, out_grid="O32", method=METHOD, **kw).forward(data)
    t_lat, t_lon = syn.octahedral(32)
    if missing is not None:  # skip the missing sources, renormalise what is left
        want = csr_matvec_missing(m.indptr, m.indices, m.data, np.stack(values, axis=1), ALL)
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), m @ values[k] if missing is None else want[:, k], f"field {k}")
        assert np.array_equal(f.grid_points()[0], t_lat) and np.array_equal(f.grid_points()[1], t_lon)
    if missing is not None:
        assert np.isnan(m @ values[1]).any() and not np.isnan(out[1].to_numpy()).any()


@pytest.mark.parametrize("packing", ["simple", "ccsds"])
def test_regrid_grib_fieldlists_on_the_packed_route(F, packing):
    s_lat, s_lon = syn.healpix(64, "nested")
    n_src = s_lat.size
    m = _oracle_csr("H64-nested", "O32")
    rng = np.random.default_rng(64)
    encode = ogrib.encode_grib2 if packing == "simple" else ogc.encode_grib2
    msgs = [encode(np.cumsum(rng.normal(0.0, 0.1, n_src)) + 280.0, 16, 1) for _ in range(6)]
    fields = [GribMessageField(msg, n_src, dict(param="t", levelist=850, step=k), latitudes=s_lat, longitudes=s_lon) for k, msg in enumerate(msgs)]
    out = F("regrid", in_grid=IN_GRID, out_grid="O32", method=METHOD).forward(ekd.SimpleFieldList(fields))
    for k, f in enumerate(out):
        host = ogc.decode(msgs[k], n_points=n_src)
        assert_same_values(f.to_numpy(), m @ host, f"{packing} field {k}")
    assert sum(f.decodes for f in fields) == 0  # decoded on the device


def test_fused_regrid_clip_equals_the_unfused_chain(F):
    from anemoi_transform_b200.fusion import FusedRegrid
    from anemoi_transform_b200.source import FieldListSource

    s_lat, s_lon = syn.healpix(64, "nested")
    values = [syn.synthetic_field("t", s_lat.size, 30 + s) for s in range(4)]
    data = ekd.from_source("list-of-dicts", [dict(values=v, latitudes=s_lat, longitudes=s_lon, param="t", levelist=850, step=k) for k, v in enumerate(values)])
    filters = [F("regrid", in_grid=IN_GRID, out_grid="O32", method=METHOD), F("clip", param="t", minimum=270.0, maximum=290.0)]
    pipe = FieldListSource(dataset=data)
    for f in filters:
        pipe = pipe | f
    plan = pipe.execution_plan()
    assert isinstance(plan[1], FusedRegrid)
    fused = pipe.forward(None)
    assert plan[1].last_forward_was_fused
    unfused = data
    for f in filters:
        unfused = f.forward(unfused)
    for a, b in zip(fused, unfused):
        assert_same_values(a.to_numpy(flatten=True), b.to_numpy(flatten=True), "fused")


def test_named_h1024_nested_to_o96_runs(F):
    regrid = F("regrid", in_grid={"grid": "H1024", "ordering": "nested"}, out_grid="O96", method=METHOD)
    s_lat, _ = syn.healpix(1024, "nested")
    x = np.ones(s_lat.size, dtype=np.float32)
    out = regrid.forward(ekd.from_source("list-of-dicts", [dict(values=x, latitudes=s_lat, longitudes=_, param="t", levelist=0)]))
    np.testing.assert_allclose(out[0].to_numpy(), 1.0, atol=1e-5)


def test_c_entries_check_their_arguments(cuda, native_library):
    from anemoi_transform_b200 import _cabi

    lib = native_library
    counts = cuda.full((768,), -7, dtype=cuda.int32, device="cuda")
    null5 = [None] * 5
    cp = ctypes.c_void_p(counts.data_ptr())
    cases = [
        ((0, 0, *null5, 0, 768, 8, 0, *null5, 0, 768), "rows"),  # a structured source without tables
        ((8, 1, *null5, 0, 768, 12, 1, *null5, 0, 1728), "power-of-two"),
        ((8, 2, *null5, 0, 768, 8, 0, *null5, 0, 768), "ordering"),
        ((8, 0, *null5, 0, 700, 8, 0, *null5, 0, 768), "points"),
        ((20000, 0, *null5, 0, 768, 8, 0, *null5, 0, 768), "nside"),
    ]
    cuda.cuda.synchronize()
    for args, message in cases:
        assert lib.at_healpix_conservative_count(*args, cp, None) == _cabi.AT_ERR_INVALID, args
        assert message in lib.at_last_error().decode(), (args, lib.at_last_error())
    assert lib.at_healpix_reorder(12, 1, None, 1, None, None) == _cabi.AT_ERR_INVALID
    cuda.cuda.synchronize()
    assert (counts == -7).all()
