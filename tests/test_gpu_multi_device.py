"""The streamed regrid over several engines (AT_B200_DEVICES, `at_hostio_group_regrid`).

On one GPU, `AT_B200_DEVICES=d,d` gives that GPU two engines, which exercises the fan-out:
chunks dealt to engines, one shared staging pool, per-engine tickets.  The tests that need two
devices skip below two GPUs."""

import ctypes

import numpy as np
import pytest
from conftest import assert_same_values
from scipy.sparse import csr_array

from anemoi_transform_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

N_FIELDS = 50  # > 64 MB of 0.25° fields: several chunks of 4 per engine, the last one short


@pytest.fixture(scope="module")
def grids():
    s_lat, s_lon = syn.regular_latlon(0.25)
    t_lat, t_lon = syn.octahedral(32)
    return s_lat, s_lon, t_lat, t_lon


@pytest.fixture(scope="module")
def matrix64(grids, tmp_path_factory):
    """A float64 bilinear matrix 0.25° -> O32 as a MIR-style npz."""
    s_lat, s_lon, t_lat, t_lon = grids
    d, i, p, shape = syn.bilinear_matrix(0.25, t_lat, t_lon)
    d = d.astype(np.float64)
    path = str(tmp_path_factory.mktemp("mdev") / "m64.npz")
    syn.save_regrid_npz(path, d, i, p, shape, s_lat, s_lon, t_lat, t_lon)
    return path, csr_array((d, i, p), shape=shape)


def _values(n_src, n=N_FIELDS, seed=0):
    rng = np.random.default_rng(seed)
    vals = []
    for k in range(n):
        v = rng.standard_normal(n_src).astype(np.float32 if k % 3 else np.float64)
        if k % 7 == 0:
            v[rng.choice(n_src, 1000, replace=False)] = np.nan
        vals.append(v)
    return vals


def _fieldlist(values, lat, lon):
    from anemoi_transform_b200 import ekd

    return ekd.from_source("list-of-dicts", [dict(param="t", levelist=850, step=k, values=v, latitudes=lat, longitudes=lon) for k, v in enumerate(values)])


def _forward(monkeypatch, devices, filt, data):
    if devices is None:
        monkeypatch.delenv("AT_B200_DEVICES", raising=False)
    else:
        monkeypatch.setenv("AT_B200_DEVICES", devices)
    return [f.to_numpy() for f in filt.forward(data)]


def _twice(cuda):
    d = cuda.cuda.current_device()
    return f"{d},{d}"


def test_matrix_regrid_on_two_engines_equals_one_engine_and_scipy(cuda, monkeypatch, grids, matrix64):
    from anemoi_transform_b200.device import HostIOGroup
    from anemoi_transform_b200.filters import create_filter_by_name as F

    s_lat, s_lon, _, _ = grids
    path, m = matrix64
    values = _values(s_lat.size)
    data = _fieldlist(values, s_lat, s_lon)
    regrid = F("regrid", matrix=path)
    single = _forward(monkeypatch, None, regrid, data)
    group = _forward(monkeypatch, _twice(cuda), regrid, data)
    d = cuda.cuda.current_device()
    assert (d, d) in HostIOGroup._groups
    for k, v in enumerate(values):
        want = m @ v
        assert group[k].dtype == want.dtype == np.float64
        assert_same_values(group[k], single[k], f"group vs single, field {k}")
        assert_same_values(group[k], want, f"group vs scipy, field {k}")
    # a second call reuses the group, its slots and the matrix
    again = _forward(monkeypatch, _twice(cuda), regrid, data)
    for k in (0, N_FIELDS // 2, N_FIELDS - 1):
        assert_same_values(again[k], group[k], f"second call, field {k}")


def test_float32_matrix_with_page_locked_inputs(cuda, monkeypatch, grids):
    from anemoi_transform_b200.device import pinned_fields
    from anemoi_transform_b200.filters import create_filter_by_name as F

    s_lat, s_lon, t_lat, t_lon = grids
    d, i, p, shape = syn.bilinear_matrix(0.25, t_lat, t_lon)
    m = csr_array((d, i, p), shape=shape)
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:
        path = f"{tmp}/m32.npz"
        syn.save_regrid_npz(path, d, i, p, shape, s_lat, s_lon, t_lat, t_lon)
        regrid = F("regrid", matrix=path)
    src = _values(s_lat.size, n=N_FIELDS - 3, seed=1)
    values, _ = pinned_fields(len(src), s_lat.size, np.float32)
    assert values is not None
    for v, s in zip(values, src):
        v[:] = s
    data = _fieldlist(values, s_lat, s_lon)
    single = _forward(monkeypatch, None, regrid, data)
    group = _forward(monkeypatch, _twice(cuda), regrid, data)
    for k, v in enumerate(values):
        assert_same_values(group[k], single[k], f"pinned group vs single, field {k}")
        assert_same_values(group[k], m @ v, f"pinned group vs scipy, field {k}")


def test_nearest_and_mask_interpolators_on_two_engines(cuda, monkeypatch, grids, tmp_path):
    from anemoi_transform_b200.filters import create_filter_by_name as F

    s_lat, s_lon, t_lat, t_lon = grids
    values = _values(s_lat.size, seed=2)
    data = _fieldlist(values, s_lat, s_lon)
    nearest = F("regrid", method="nearest", in_grid=dict(latitudes=s_lat, longitudes=s_lon), out_grid=dict(latitudes=t_lat, longitudes=t_lon))
    single = _forward(monkeypatch, None, nearest, data)
    group = _forward(monkeypatch, _twice(cuda), nearest, data)
    idx = nearest.interpolator.nearest_grid_points.reshape(-1).cpu().numpy()
    for k, v in enumerate(values):
        assert_same_values(group[k], single[k], f"nearest group vs single, field {k}")
        assert_same_values(group[k], v[idx], f"nearest group vs numpy indexing, field {k}")

    mask = np.sort(np.random.default_rng(3).choice(s_lat.size, 200_000, replace=False))
    mpath = str(tmp_path / "mask.npz")
    np.savez(mpath, mask=mask)
    masked = F("regrid", mask=mpath)
    single = _forward(monkeypatch, None, masked, data)
    group = _forward(monkeypatch, _twice(cuda), masked, data)
    for k, v in enumerate(values):
        assert_same_values(group[k], single[k], f"mask group vs single, field {k}")
        assert_same_values(group[k], v[mask], f"mask group vs numpy indexing, field {k}")


def test_grib_packed_fieldlist_on_two_engines(cuda, monkeypatch, grids, matrix64):
    from grib_fields import GribMessageField
    from oracle import grib as ogrib

    from anemoi_transform_b200.filters import create_filter_by_name as F

    s_lat, s_lon, _, _ = grids
    path, m = matrix64
    rng = np.random.default_rng(4)
    n = 40
    fields = []
    for k in range(n):
        msg = (ogrib.encode_grib2 if k % 2 == 0 else ogrib.encode_grib1)(rng.normal(280.0, 10.0, s_lat.size), 16, 1)
        fields.append(GribMessageField(msg, s_lat.size, dict(param="t", levelist=850, step=k), latitudes=s_lat, longitudes=s_lon))
    regrid = F("regrid", matrix=path)
    single = _forward(monkeypatch, None, regrid, fields)
    group = _forward(monkeypatch, _twice(cuda), regrid, fields)
    assert all(f.decodes == 0 for f in fields), "the GRIB fields were decoded on the host"
    for k, f in enumerate(fields):
        want = m @ ogrib.decode(f.message(), n_points=s_lat.size)
        assert_same_values(group[k], single[k], f"grib group vs single, field {k}")
        assert_same_values(group[k], want, f"grib group vs scipy, field {k}")


def test_replicated_matrix_outlives_the_original(cuda):
    from ctypes import byref, c_void_p

    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.device import CsrMatrix, stream_ptr

    t_lat, t_lon = syn.octahedral(48)
    d, i, p, shape = syn.bilinear_matrix(2.0, t_lat, t_lon)
    for dtype in (np.float32, np.float64):
        csr = CsrMatrix(d.astype(dtype), i, p, shape)
        X = cuda.randn((shape[1], 8), device="cuda", dtype=cuda.float32)
        X[::17, 3] = float("nan")
        want = csr.apply(X)
        copy = c_void_p()
        _cabi.call("at_csr_replicate", csr.handle, cuda.cuda.current_device(), byref(copy))
        code = {cuda.float32: _cabi.AT_F32, cuda.float64: _cabi.AT_F64}

        def spmm(h):
            Y = cuda.empty_like(want)
            _cabi.call("at_spmm", h, c_void_p(X.data_ptr()), _cabi.AT_F32, X.stride(0), c_void_p(Y.data_ptr()), code[Y.dtype], Y.stride(0), X.shape[1], 0, stream_ptr())
            return Y.cpu().numpy()

        assert_same_values(spmm(copy), want.cpu().numpy(), f"replica {dtype.__name__}")
        csr.close()
        cuda.cuda.synchronize()
        assert_same_values(spmm(copy), want.cpu().numpy(), f"replica after close {dtype.__name__}")
        _cabi.call("at_csr_destroy", copy)


def test_group_rejects_bad_arguments(cuda):
    from ctypes import byref, c_int32, c_void_p

    from anemoi_transform_b200 import _cabi

    lib = _cabi.load()
    h = c_void_p()
    n = cuda.cuda.device_count()
    assert lib.at_hostio_group_create(2, (c_int32 * 2)(0, n), 0, byref(h)) == _cabi.AT_ERR_INVALID
    assert b"out of range" in lib.at_last_error() and h.value is None
    assert lib.at_hostio_group_create(0, (c_int32 * 1)(0), 0, byref(h)) == _cabi.AT_ERR_INVALID
    assert lib.at_hostio_group_wait(None, 0) == _cabi.AT_ERR_INVALID
    assert lib.at_csr_replicate(None, 0, byref(h)) == _cabi.AT_ERR_INVALID


# --------------------------------------------------------------- two or more GPUs ------
def _need_two(cuda):
    if cuda.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, {cuda.cuda.device_count()} visible: a matrix on another device and `all` need a second device")


def test_all_devices_equal_one_device(cuda, monkeypatch, grids, matrix64):
    _need_two(cuda)
    from anemoi_transform_b200.filters import create_filter_by_name as F

    s_lat, s_lon, _, _ = grids
    path, m = matrix64
    values = _values(s_lat.size, seed=5)
    data = _fieldlist(values, s_lat, s_lon)
    regrid = F("regrid", matrix=path)
    single = _forward(monkeypatch, None, regrid, data)
    group = _forward(monkeypatch, "all", regrid, data)
    for k, v in enumerate(values):
        assert_same_values(group[k], single[k], f"all vs one GPU, field {k}")
        assert_same_values(group[k], m @ v, f"all vs scipy, field {k}")


def test_matrix_on_another_device_is_refused(cuda):
    _need_two(cuda)
    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.device import CsrMatrix, HostIO, StreamedRegrid

    t_lat, t_lon = syn.octahedral(48)
    d, i, p, shape = syn.bilinear_matrix(2.0, t_lat, t_lon)
    with cuda.cuda.device(1):
        csr = CsrMatrix(d, i, p, shape)
    assert csr.device == 1
    with cuda.cuda.device(0):
        X = cuda.zeros((shape[1], 4), device="cuda:0")
        Y = cuda.zeros((shape[0], 4), device="cuda:0")
        lib = _cabi.load()
        rc = lib.at_spmm(csr.handle, ctypes.c_void_p(X.data_ptr()), _cabi.AT_F32, 4, ctypes.c_void_p(Y.data_ptr()), _cabi.AT_F32, 4, 4, 0, None)
        assert rc == _cabi.AT_ERR_INVALID and b"device 1" in lib.at_last_error()
        assert HostIO.get().device == 0
        with pytest.raises(ValueError, match="staged on device 1"):
            StreamedRegrid(_cabi.HOSTIO_SPMM, csr, None, shape[0], cuda.float32, [np.zeros(shape[1], np.float32)], False, True).join()
        # a batch on device 1 downloads through device 1's engine even with device 0 current
        with cuda.cuda.device(1):
            on1 = csr.apply(cuda.ones((shape[1], 4), device="cuda:1"))
        from anemoi_transform_b200.device import DeviceBatch

        batch = DeviceBatch(on1, 4)
        assert_same_values(batch.take_column(2), on1[:, 2].cpu().numpy(), "column of a device-1 batch")
