"""`at_conservative_matrix_count` / `_fill` (first-order conservative weights built on the
device) against the numpy restatement oracle/conservative_matrix.py::conservative_matrix, bit
for bit, and the `regrid(in_grid=…, out_grid=…, method="structured-conservative")` recipe on the
streamed, resident and fused routes."""

import ctypes

import numpy as np
import pytest
from conftest import assert_same_values
from scipy.sparse import csr_array

from anemoi_transform_b200 import ekd
from anemoi_transform_b200 import synthetic as syn
from oracle import conservative_matrix as oc
from oracle import structured_matrix as om

pytestmark = pytest.mark.gpu

METHOD = "structured-conservative"


@pytest.fixture(scope="module")
def F(cuda):
    from anemoi_transform_b200.filters import create_filter_by_name

    return create_filter_by_name


def _south_to_north(lat, lon):
    starts = np.flatnonzero(np.concatenate(([True], lat[1:] != lat[:-1])))
    bounds = np.append(starts, lat.size)
    order = np.concatenate([np.arange(a, b) for a, b in zip(bounds[-2::-1], bounds[:0:-1])])
    return lat[order], lon[order]


def _one_point_rows():
    """Rows of 1, 2, 3 and 5 points, stored south → north, first longitudes off zero."""
    row_lat, pl, lon0 = [-60.0, -20.0, 25.0, 70.0], [1, 2, 3, 5], [10.0, 0.0, 100.0, 350.0]
    return np.repeat(row_lat, pl), np.concatenate([l0 + np.arange(p) * (360.0 / p) for l0, p in zip(lon0, pl)])


def _grid(name):
    if name == "1235-south-to-north":
        return _one_point_rows()
    if name == "1235-north-to-south":
        return _south_to_north(*_one_point_rows())
    if name.startswith("o"):
        return syn.octahedral(int(name[1:]))
    if name == "n320":
        return syn.n320_like()
    return syn.regular_latlon(float(name.rstrip("deg")))


CASES = [
    ("o48", "2.5deg"),
    ("1deg", "o96"),
    ("o1280", "n320"),
    ("0.25deg", "o96"),
    ("o320", "10deg"),
    ("1235-south-to-north", "o16"),
    ("1235-north-to-south", "o16"),
    ("o16", "1235-south-to-north"),
    ("o16", "1235-north-to-south"),
    ("o96", "o96"),
]


@pytest.mark.parametrize("source,target", CASES)
def test_device_conservative_matrix_is_bitwise_the_oracle(cuda, source, target):
    from anemoi_transform_b200.regrid_files import make_conservative_matrix

    s_lat, s_lon = _grid(source)
    t_lat, t_lon = _grid(target)
    d, i, p, shape = make_conservative_matrix(s_lat, s_lon, t_lat, t_lon)
    want = oc.conservative_matrix(om.structured_rows(s_lat, s_lon), om.structured_rows(t_lat, t_lon))
    assert shape == want[3] == (t_lat.size, s_lat.size)
    assert d.dtype == np.float32 and i.dtype == np.int32 and p.dtype == np.int32
    assert np.array_equal(p, want[2]) and np.array_equal(i, want[1])
    bad = np.flatnonzero(d.view(np.uint32) != want[0].view(np.uint32))
    assert bad.size == 0, f"{bad.size} weights differ bitwise, first at entries {bad[:5]}"
    if (source, target) == ("o320", "10deg"):
        assert np.diff(p).max() > 1024  # equatorial rows longer than a CTA of the SpMM stages
    if source == target:
        assert np.array_equal(p, np.arange(t_lat.size + 1)) and (d == 1.0).all()


def _box_areas(rows):
    zn, zs = oc.box_tables(rows)
    area = np.empty(int(rows[3].sum()))
    for k in range(rows[0].size):
        area[rows[2][k] : rows[2][k] + rows[3][k]] = (zn[k] - zs[k]) * (2.0 * np.pi / rows[3][k])
    return area


def test_full_size_o1280_to_n320_keeps_the_area_integral(cuda):
    from anemoi_transform_b200.regrid_files import make_conservative_matrix

    s_lat, s_lon = syn.octahedral(1280)
    t_lat, t_lon = syn.n320_like()
    d, i, p, shape = make_conservative_matrix(s_lat, s_lon, t_lat, t_lon)
    m = csr_array((d, i, p), shape=shape)
    ph, la = np.deg2rad(s_lat), np.deg2rad(s_lon)
    x = 5.0 + np.cos(ph) * np.cos(la) + 3.0 * np.sin(ph) + np.cos(ph) ** 2 * np.sin(3 * la)
    y = m @ x
    a_s, a_t = _box_areas(om.structured_rows(s_lat, s_lon)), _box_areas(om.structured_rows(t_lat, t_lon))
    assert abs((a_t * y).sum() - (a_s * x).sum()) <= 2e-6 * (a_s * x).sum()
    assert np.abs(m.sum(axis=1) - 1.0).max() <= 1e-5


def _fieldlist(values, lat, lon):
    return ekd.from_source("list-of-dicts", [dict(values=v, latitudes=lat, longitudes=lon, param="tp", levelist=0, step=k) for k, v in enumerate(values)])


def _values(n, dtype):
    vals = [syn.synthetic_field("t", n, s, 0.003 if s % 3 == 0 else 0.0) for s in range(7)]
    return [v.astype(dtype) for v in vals]


@pytest.mark.parametrize("grids", [("O96", [1.0, 1.0]), ("O320", [10.0, 10.0])], ids=["o96-1deg", "o320-10deg"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("route", ["streamed", "resident"])
def test_recipes_equal_the_oracle_matrix_per_field(F, grids, dtype, route):
    from anemoi_transform_b200.device import results_stay_on_device
    from anemoi_transform_b200.fields import device_column_of

    in_grid, out_grid = grids
    s_lat, s_lon = syn.octahedral(int(in_grid[1:]))
    t_lat, t_lon = syn.regular_latlon(out_grid[0])
    m = oc.conservative_csr(s_lat, s_lon, t_lat, t_lon)
    values = _values(s_lat.size, dtype)
    data = _fieldlist(values, s_lat, s_lon)
    regrid = F("regrid", in_grid=in_grid, out_grid=out_grid, method=METHOD)
    if route == "streamed":
        out = regrid.forward(data)
    else:
        with results_stay_on_device():
            out = regrid.forward(data)
        assert all(device_column_of(f) is not None for f in out)
    assert len(out) == len(values)
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), m @ values[k], f"{grids} {route} field {k}")
        assert np.array_equal(f.grid_points()[0], t_lat) and np.array_equal(f.grid_points()[1], t_lon)
    assert regrid.interpolator.matrix.shape == m.shape


def test_a_written_matrix_file_reloads(F, tmp_path):
    from anemoi_transform_b200.regrid_files import make_conservative_matrix

    s_lat, s_lon = syn.octahedral(48)
    t_lat, t_lon = syn.regular_latlon(2.5)
    make_conservative_matrix(s_lat, s_lon, t_lat, t_lon, output=str(tmp_path / "m.npz"))
    values = _values(s_lat.size, np.float32)
    out = F("regrid", matrix=str(tmp_path / "m.npz")).forward(_fieldlist(values, s_lat, s_lon))
    m = oc.conservative_csr(s_lat, s_lon, t_lat, t_lon)
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), m @ values[k], f"field {k}")


def _mixed_fields(s_lat, s_lon):
    specs = [("t", 850), ("u", 850), ("v", 850), ("q", 850), ("u", 500), ("v", 500), ("t", 500), ("q", 500), ("lsm", 0)]
    values = []
    for i, (p, _) in enumerate(specs):
        if p == "lsm":
            values.append(np.random.default_rng(i).uniform(0.0, 1.0, s_lat.size).astype(np.float32))
        else:
            values.append(syn.synthetic_field(p, s_lat.size, 80 + i, 0.002 if i % 4 == 0 else 0.0))
    return ekd.from_source("list-of-dicts", [dict(values=v, latitudes=s_lat, longitudes=s_lon, param=p, levelist=lev) for v, (p, lev) in zip(values, specs)])


def test_conservative_regrid_fuses_with_its_followers(F):
    """`regrid(structured-conservative) | uv_to_ddff | q_to_r | clip | apply_mask` is one launch
    (rows of varying length on the fused SpMM) and bitwise the filters run one after the other."""
    from anemoi_transform_b200.fusion import FusedRegrid
    from anemoi_transform_b200.source import FieldListSource

    s_lat, s_lon = syn.octahedral(48)
    data = _mixed_fields(s_lat, s_lon)
    filters = [
        F("regrid", in_grid="O48", out_grid=[5.0, 5.0], method=METHOD),
        F("uv_to_ddff"),
        F("q_to_r", return_inputs="none"),
        F("clip", param="r", minimum=5.0),
        F("apply_mask", mask_param="lsm", threshold=0.5, threshold_operator=">", param=["ws", "r"]),
    ]
    pipe = FieldListSource(dataset=data)
    for f in filters:
        pipe = pipe | f
    plan = pipe.execution_plan()
    assert len(plan) == 2 and isinstance(plan[1], FusedRegrid)
    fused = pipe.forward(None)
    assert plan[1].last_forward_was_fused
    unfused = data
    for f in filters:
        unfused = f.forward(unfused)
    assert [(f.metadata("param"), f.metadata("levelist")) for f in fused] == [(f.metadata("param"), f.metadata("levelist")) for f in unfused]
    for a, b in zip(fused, unfused):
        assert_same_values(a.to_numpy(flatten=True), b.to_numpy(flatten=True), str(a.metadata("param")))
        assert np.array_equal(a.grid_points()[0], b.grid_points()[0])
    assert "ws" in [f.metadata("param") for f in fused] and "r" in [f.metadata("param") for f in fused]


def test_refusals(F, cuda, native_library):
    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.regrid_files import box_z_edges, structured_grid_rows

    # a target that is not a structured grid, a source that is not global; grid-box-average stays MIR's
    s_lat, s_lon = syn.octahedral(32)
    t_lat, t_lon = syn.regular_latlon(10.0)
    shuffle = np.random.default_rng(5).permutation(t_lat.size)
    values = [np.zeros(s_lat.size, np.float32)]
    with pytest.raises(NotImplementedError, match=f"{METHOD}.*target"):
        F("regrid", in_grid="O32", out_grid=dict(latitudes=t_lat[shuffle], longitudes=t_lon[shuffle]), method=METHOD).forward(_fieldlist(values, s_lat, s_lon))
    b_lat, b_lon = syn.regular_latlon(2.0)
    band = np.abs(b_lat) <= 60.0
    with pytest.raises(ValueError, match="not global"):
        F("regrid", out_grid="O16", method=METHOD).forward(_fieldlist([np.zeros(int(band.sum()), np.float32)], b_lat[band], b_lon[band]))
    with pytest.raises(NotImplementedError, match="not built locally"):
        F("regrid", in_grid="O32", out_grid=[10.0, 10.0], method="grid-box-average")

    # the C entries check their arguments and answer with a status, not a launch
    def device_tables(lat, lon):
        rows = structured_grid_rows(lat, lon)
        z = box_z_edges(rows[0])
        return [cuda.from_numpy(np.ascontiguousarray(a)).cuda() for a in (z[:-1], z[1:], *rows[1:])], rows[0].size

    src, n_src_rows = device_tables(s_lat, s_lon)
    tgt, n_tgt_rows = device_tables(t_lat, t_lon)
    sp, tp = [ctypes.c_void_p(t.data_ptr()) for t in src], [ctypes.c_void_p(t.data_ptr()) for t in tgt]
    n_src, n_tgt = s_lat.size, t_lat.size
    counts = cuda.full((n_tgt,), -7, dtype=cuda.int32, device="cuda")
    indptr = cuda.zeros((n_tgt + 1,), dtype=cuda.int32, device="cuda")
    data = cuda.full((1 << 16,), -7.0, dtype=cuda.float32, device="cuda")
    idx = cuda.full((1 << 16,), -7, dtype=cuda.int32, device="cuda")
    good = dict(src=sp, n_src_rows=n_src_rows, n_src=n_src, tgt=tp, n_tgt_rows=n_tgt_rows, n_tgt=n_tgt, counts=ctypes.c_void_p(counts.data_ptr()),
                indptr=ctypes.c_void_p(indptr.data_ptr()), nnz=1000, data=ctypes.c_void_p(data.data_ptr()), idx=ctypes.c_void_p(idx.data_ptr()))  # fmt: skip
    grid_cases = [
        (dict(n_src_rows=1), "rows"),
        (dict(n_tgt_rows=1), "rows"),
        (dict(n_src=10), "rows"),
        (dict(n_src=1 << 31), "int32"),
        (dict(n_tgt=1 << 31), "int32"),
        (dict(src=[sp[0], None, *sp[2:]]), "null"),
        (dict(tgt=[*tp[:4], None]), "null"),
    ]
    count_cases = grid_cases + [(dict(counts=None), "null")]
    fill_cases = grid_cases + [(dict(nnz=1 << 31), "int32"), (dict(nnz=-1), "int32"), (dict(indptr=None), "null"), (dict(data=None), "null"), (dict(idx=None), "null")]
    lib = native_library

    def grid_args(a):
        return (*a["src"], a["n_src_rows"], a["n_src"], *a["tgt"], a["n_tgt_rows"], a["n_tgt"])

    cuda.cuda.synchronize()
    for name, cases in (("count", count_cases), ("fill", fill_cases)):
        for change, message in cases:
            a = {**good, **change}
            if name == "count":
                rc = lib.at_conservative_matrix_count(*grid_args(a), a["counts"], None)
            else:
                rc = lib.at_conservative_matrix_fill(*grid_args(a), a["indptr"], a["nnz"], a["data"], a["idx"], None)
            assert rc == _cabi.AT_ERR_INVALID, (name, change)
            assert message in lib.at_last_error().decode(), (name, change, lib.at_last_error())
    cuda.cuda.synchronize()
    assert (counts == -7).all() and (data == -7.0).all() and (idx == -7).all()  # nothing was launched

    # and the same arguments, put right, build the matrix
    assert lib.at_conservative_matrix_count(*grid_args(good), good["counts"], None) == _cabi.AT_OK
    indptr[1:] = cuda.cumsum(counts, 0, dtype=cuda.int32)
    nnz = int(indptr[-1])
    assert lib.at_conservative_matrix_fill(*grid_args(good), good["indptr"], nnz, good["data"], good["idx"], None) == _cabi.AT_OK
    cuda.cuda.synchronize()
    want = oc.conservative_matrix(om.structured_rows(s_lat, s_lon), om.structured_rows(t_lat, t_lon))
    assert np.array_equal(indptr.cpu().numpy(), want[2])
    assert np.array_equal(idx[:nnz].cpu().numpy(), want[1]) and np.array_equal(data[:nnz].cpu().numpy().view(np.uint32), want[0].view(np.uint32))
    assert (idx[nnz:] == -7).all()
