"""`at_structured_matrix` (structured bilinear / bicubic weights built on the device) against the
numpy restatement oracle/structured_matrix.py::structured_matrix, bit for bit, and the
`regrid(in_grid=…, out_grid=…, method="structured-bilinear" | "structured-bicubic")` recipes
on the streamed, resident and fused routes."""

import ctypes

import numpy as np
import pytest
from conftest import assert_same_values

from anemoi_transform_b200 import ekd
from anemoi_transform_b200 import synthetic as syn
from oracle import structured_matrix as om

pytestmark = pytest.mark.gpu

METHODS = {"structured-bilinear": 2, "structured-bicubic": 4}


@pytest.fixture(scope="module")
def F(cuda):
    from anemoi_transform_b200.filters import create_filter_by_name

    return create_filter_by_name


def _grid(name):
    if name.startswith("o"):
        return syn.octahedral(int(name[1:]))
    if name == "n320":
        return syn.n320_like()
    return syn.regular_latlon(float(name.rstrip("deg")))


def _with_edge_targets(t_lat, t_lon, rows):
    """Poles, source row latitudes hit exactly, the 360 -> 0 seam, λ = 720.5 and -0.0."""
    row_lat = rows[0]
    lat = [90.0, -90.0, 90.0, -90.0, row_lat[0], row_lat[1], row_lat[row_lat.size // 2], row_lat[-1], 0.0, 10.0, -0.0, 45.0]
    lon = [0.0, 123.4, 359.9999, -0.0, 0.0, 359.99999999, 720.5, 180.0, 360.0 - 1e-9, 720.5, -0.0, -0.0]
    return np.concatenate([t_lat, lat]), np.concatenate([t_lon, lon])


@pytest.mark.parametrize("method", sorted(METHODS))
@pytest.mark.parametrize("source,target", [("o48", "2.5deg"), ("1deg", "o96"), ("o1280", "n320"), ("o1280", "0.25deg")])
def test_device_structured_matrix_is_bitwise_the_oracle(cuda, method, source, target):
    from anemoi_transform_b200.regrid_files import make_structured_matrix

    s_lat, s_lon = _grid(source)
    rows = om.structured_rows(s_lat, s_lon)
    t_lat, t_lon = _with_edge_targets(*_grid(target), rows)
    d, i, p, shape = make_structured_matrix(s_lat, s_lon, t_lat, t_lon, method)
    want = om.structured_matrix(rows, t_lat, t_lon, METHODS[method])
    assert shape == want[3] == (t_lat.size, s_lat.size)
    assert d.dtype == np.float32 and i.dtype == np.int32 and p.dtype == np.int32
    assert np.array_equal(p, want[2]) and np.array_equal(i, want[1])
    bad = np.flatnonzero(d.view(np.uint32) != want[0].view(np.uint32))
    assert bad.size == 0, f"{bad.size} weights differ bitwise, first at entries {bad[:5]}"
    assert (d == 0).any()  # the explicit zeros are kept


def _fieldlist(values, lat, lon):
    return ekd.from_source("list-of-dicts", [dict(values=v, latitudes=lat, longitudes=lon, param="t", levelist=850, step=k) for k, v in enumerate(values)])


def _values(n, dtype):
    vals = [syn.synthetic_field("t", n, s, 0.003 if s % 3 == 0 else 0.0) for s in range(7)]
    return [v.astype(dtype) for v in vals]


@pytest.mark.parametrize("method", sorted(METHODS))
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("route", ["streamed", "resident"])
def test_o96_recipes_equal_the_oracle_matrix_per_field(F, method, dtype, route):
    from anemoi_transform_b200.device import results_stay_on_device
    from anemoi_transform_b200.fields import device_column_of

    s_lat, s_lon = syn.octahedral(96)
    t_lat, t_lon = syn.regular_latlon(1.5)
    m = om.structured_csr(s_lat, s_lon, t_lat, t_lon, METHODS[method])
    values = _values(s_lat.size, dtype)
    data = _fieldlist(values, s_lat, s_lon)
    regrid = F("regrid", in_grid="O96", out_grid=[1.5, 1.5], method=method)
    if route == "streamed":
        out = regrid.forward(data)
    else:
        with results_stay_on_device():
            out = regrid.forward(data)
        assert all(device_column_of(f) is not None for f in out)  # kept in HBM for a follower
    assert len(out) == len(values)
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), m @ values[k], f"{method} {route} field {k}")
        assert np.array_equal(f.grid_points()[0], t_lat) and np.array_equal(f.grid_points()[1], t_lon)
    assert regrid.interpolator.matrix.shape == m.shape


def _mixed_fields(s_lat, s_lon):
    specs = [("t", 850), ("u", 850), ("v", 850), ("q", 850), ("u", 500), ("v", 500), ("t", 500), ("q", 500), ("lsm", 0)]
    values = []
    for i, (p, _) in enumerate(specs):
        if p == "lsm":
            values.append(np.random.default_rng(i).uniform(0.0, 1.0, s_lat.size).astype(np.float32))
        else:
            values.append(syn.synthetic_field(p, s_lat.size, 80 + i, 0.002 if i % 4 == 0 else 0.0))
    return ekd.from_source("list-of-dicts", [dict(values=v, latitudes=s_lat, longitudes=s_lon, param=p, levelist=lev) for v, (p, lev) in zip(values, specs)])


def test_structured_bicubic_regrid_fuses_with_its_followers(F):
    """`regrid(structured-bicubic) | uv_to_ddff | q_to_r | clip | apply_mask` is one launch
    (16 entries per row on the fused SpMM) and bitwise the filters run one after the other."""
    from anemoi_transform_b200.fusion import FusedRegrid
    from anemoi_transform_b200.source import FieldListSource

    s_lat, s_lon = syn.octahedral(48)
    data = _mixed_fields(s_lat, s_lon)
    filters = [
        F("regrid", in_grid="O48", out_grid="O24", method="structured-bicubic"),
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

    # a source that is not a structured grid, and one that is not global
    s_lat, s_lon = syn.octahedral(32)
    shuffle = np.random.default_rng(5).permutation(s_lat.size)
    values = [np.zeros(s_lat.size, np.float32)]
    for method in METHODS:
        with pytest.raises(NotImplementedError, match=method):
            F("regrid", in_grid=dict(latitudes=s_lat[shuffle], longitudes=s_lon[shuffle]), out_grid="O16", method=method).forward(_fieldlist(values, s_lat[shuffle], s_lon[shuffle]))
    b_lat, b_lon = syn.regular_latlon(2.0)
    band = np.abs(b_lat) <= 60.0
    with pytest.raises(ValueError, match="not global"):
        F("regrid", out_grid="O16", method="structured-bilinear").forward(_fieldlist([np.zeros(int(band.sum()), np.float32)], b_lat[band], b_lon[band]))

    # the C entry checks its arguments and answers with a status, not a launch
    rows = om.structured_rows(s_lat, s_lon)
    tables = [cuda.from_numpy(np.ascontiguousarray(a)).cuda() for a in rows]
    tgt = cuda.zeros(8, dtype=cuda.float64, device="cuda")
    data = cuda.full((128,), -7.0, dtype=cuda.float32, device="cuda")
    idx = cuda.full((128,), -7, dtype=cuda.int32, device="cuda")
    ptr = [ctypes.c_void_p(t.data_ptr()) for t in tables]
    n_rows, n_src = rows[0].size, s_lat.size
    good = dict(stencil=4, n_rows=n_rows, n_src=n_src, n_tgt=8, tables=ptr, tgt=ctypes.c_void_p(tgt.data_ptr()), data=ctypes.c_void_p(data.data_ptr()))
    cases = [
        (dict(stencil=3), "stencil"),
        (dict(stencil=2, n_rows=1), "rows"),
        (dict(n_rows=3), "rows"),
        (dict(n_src=1 << 31), "int32"),
        (dict(n_src=0), "int32"),
        (dict(n_tgt=(1 << 31) // 16), "int32"),
        (dict(n_tgt=-1), "int32"),
        (dict(tables=[ptr[0], None, ptr[2], ptr[3]]), "null"),
        (dict(tgt=None), "null"),
        (dict(data=None), "null"),
    ]
    lib = native_library
    cuda.cuda.synchronize()
    for change, message in cases:
        a = {**good, **change}
        rc = lib.at_structured_matrix(*a["tables"], a["n_rows"], a["n_src"], a["stencil"], a["tgt"], a["tgt"], a["n_tgt"], a["data"], ctypes.c_void_p(idx.data_ptr()), None)
        assert rc == _cabi.AT_ERR_INVALID, change
        assert message in lib.at_last_error().decode(), (change, lib.at_last_error())
    cuda.cuda.synchronize()
    assert (data == -7.0).all() and (idx == -7).all()  # nothing was launched
    # and the same arguments, put right, build the matrix
    assert lib.at_structured_matrix(*ptr, n_rows, n_src, 4, good["tgt"], good["tgt"], 8, good["data"], ctypes.c_void_p(idx.data_ptr()), None) == _cabi.AT_OK
    cuda.cuda.synchronize()
    want = om.structured_matrix(rows, np.zeros(8), np.zeros(8), 4)
    assert np.array_equal(idx.cpu().numpy(), want[1]) and np.array_equal(data.cpu().numpy().view(np.uint32), want[0].view(np.uint32))
