"""`at_spmm_missing` and `regrid(…, missing_values=…)` against oracle/spmm_missing.py, bit for
bit: every dtype pair and kernel (uniform 4 / 12 / 16 entries, variable rows, rows over the
1 024 staged entries, full and ragged column tiles, the scalar-column float64 kernel), the
recipes at full size on the resident and streamed routes, GRIB messages with bitmaps, a
two-engine fan-out, the unfused chain, and the gather regrids."""

import numpy as np
import pytest
from conftest import assert_same_values
from scipy.sparse import csr_array

from anemoi_transform_b200 import ekd
from anemoi_transform_b200 import synthetic as syn
from oracle import conservative_matrix as oc
from oracle import structured_matrix as om
from oracle.spmm_missing import ALL, HEAVIEST, PROPAGATE, csr_matvec_missing

pytestmark = pytest.mark.gpu

NAMES = {ALL: "missing-if-all-missing", HEAVIEST: "missing-if-heaviest-missing"}
DTYPES = [(np.float32, np.float32), (np.float64, np.float32), (np.float32, np.float64), (np.float64, np.float64)]


@pytest.fixture(scope="module")
def F(cuda):
    from anemoi_transform_b200.filters import create_filter_by_name

    return create_filter_by_name


def land_mask(lat, lon, seed=5, fraction=0.3):
    """About `fraction` of the points, in coherent blobs (coasts), seeded."""
    rng = np.random.default_rng(seed)
    la, lo = np.radians(lat), np.radians(lon)
    v = np.zeros(lat.size)
    for _ in range(12):
        c_la, c_lo = np.arcsin(rng.uniform(-1, 1)), rng.uniform(0, 2 * np.pi)
        v += np.exp(-((np.cos(la) * np.cos(c_la) * np.cos(lo - c_lo) + np.sin(la) * np.sin(c_la)) - 1) ** 2 * 8)
    return v > np.quantile(v, 1 - fraction)


def masked_values(lat, lon, n_fields, dtype, seed=0):
    """Point-major [n_src, n_fields]: a land mask (a second one in every fifth field), field 0 all
    valid, field 1 all NaN."""
    rng = np.random.default_rng(seed)
    base = (np.sin(np.radians(lat)) * 30 + 280).astype(np.float64)
    X = base[:, None] + rng.standard_normal((lat.size, n_fields))
    land, other = land_mask(lat, lon, 5), land_mask(lat, lon, 6)
    for f in range(2, n_fields):
        X[other if f % 5 == 0 else land, f] = np.nan
    X[:, 1] = np.nan
    return X.astype(dtype)


def _uniform12(n_rows, n_src, seed=3, land=None):
    """12 entries per row, weights in [0, 1) with explicit zeros.  With `land` (the mask most
    fields use), every 25th row ties its first and eighth entries at the row maximum, one of the
    two on land: the first tied entry is the heaviest, so `heaviest` gives NaN exactly when it is
    the missing one (a `>=` would pick the other)."""
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.integers(0, n_src, (n_rows, 12)), axis=1).astype(np.int32)
    w = rng.random((n_rows, 12)).astype(np.float32)
    w.reshape(-1)[::7] = 0.0
    if land is not None:
        wet, dry = np.flatnonzero(~land), np.flatnonzero(land)
        for r in range(0, n_rows, 25):
            first_dry = r % 50 == 0
            idx[r, 0] = rng.choice(dry if first_dry else wet)
            idx[r, 7] = rng.choice(wet if first_dry else dry)
            w[r, 0] = w[r, 7] = 1.5
    return w.ravel(), idx.ravel(), (12 * np.arange(n_rows + 1)).astype(np.int32), (n_rows, n_src)


def _csr(kind):
    """(data float32, indices, indptr, shape, source grid) of each kernel path."""
    if kind == "uniform4":
        s, t = syn.octahedral(96), syn.regular_latlon(1.0)
        return (*om.structured_matrix(om.structured_rows(*s), *t, 2), s)
    if kind == "uniform16":
        s, t = syn.octahedral(96), syn.regular_latlon(1.0)
        return (*om.structured_matrix(om.structured_rows(*s), *t, 4), s)
    if kind == "uniform12":
        s = syn.octahedral(96)
        return (*_uniform12(20000, s[0].size, land=land_mask(*s, 5)), s)
    if kind == "variable":
        s, t = syn.regular_latlon(1.0), syn.octahedral(96)
        m = oc.conservative_csr(*s, *t)
    else:  # rows over the 1 024 staged entries: the FALLBACK path
        s, t = syn.octahedral(320), syn.regular_latlon(10.0)
        m = oc.conservative_csr(*s, *t)
        assert np.diff(m.indptr).max() > 1024
    return m.data, m.indices, m.indptr, m.shape, s


@pytest.fixture(scope="module", params=["uniform4", "uniform12", "uniform16", "variable", "fallback"])
def matrix(request, cuda):
    return _csr(request.param), request.param


def _apply(cuda, csr, X, n_fields, missing):
    Xd = cuda.from_numpy(np.ascontiguousarray(X)).cuda()
    Y = csr.apply(Xd, n_fields=n_fields, missing=missing)
    cuda.cuda.synchronize()
    return Y.cpu().numpy()[:, :n_fields]


@pytest.mark.parametrize("wdt,xdt", DTYPES, ids=[f"{np.dtype(a).name}@{np.dtype(b).name}" for a, b in DTYPES])
def test_at_spmm_missing_is_bitwise_the_oracle(cuda, matrix, wdt, xdt):
    from anemoi_transform_b200.device import CsrMatrix

    (d, i, p, shape, (s_lat, s_lon)), kind = matrix
    d = d.astype(wdt)
    csr = CsrMatrix(d, i, p, shape)
    # fields: one float4 / 16-byte unit (packed rows), full tiles plus a ragged last tile packed
    # (300) and not packed (456); fewer on the large FALLBACK source
    counts = (3, 300, 456) if kind != "fallback" else (3, 140)
    X_all = masked_values(s_lat, s_lon, max(counts), xdt)
    want = {policy: csr_matvec_missing(p, i, d, X_all, policy) for policy in (ALL, HEAVIEST)}
    for n in counts:
        X = np.pad(X_all[:, :n], ((0, 0), (0, (-n) % 4)))  # the vectorised kernels want ld % 4 == 0
        for policy in (ALL, HEAVIEST):
            assert_same_values(_apply(cuda, csr, X, n, policy), want[policy][:, :n], f"{kind} {np.dtype(wdt).name}@{np.dtype(xdt).name} F={n} policy {policy}")
    if not (wdt == np.float32 and xdt == np.float32):  # ld not a multiple of 4: the scalar-column kernel
        n = 37
        X = np.pad(X_all[:, :n], ((0, 0), (0, 2)))
        for policy in (ALL, HEAVIEST):
            assert_same_values(_apply(cuda, csr, X, n, policy), want[policy][:, :n], f"{kind} generic F={n} policy {policy}")
    # NaN-free inputs: every policy is the plain SpMM
    nc = 140
    Xc = np.nan_to_num(X_all[:, :nc], nan=1.5)
    plain = _apply(cuda, csr, Xc, nc, PROPAGATE)
    assert_same_values(plain, csr_array((d, i, p), shape=shape) @ Xc, f"{kind} plain vs scipy")
    for policy in (ALL, HEAVIEST):
        assert_same_values(_apply(cuda, csr, Xc, nc, policy), plain, f"{kind} NaN-free policy {policy}")


def test_unknown_policy_and_variant_are_refused(cuda):
    from anemoi_transform_b200.device import CsrMatrix

    d, i, p, shape = _uniform12(64, 100)
    csr = CsrMatrix(d, i, p, shape)
    X = cuda.zeros((100, 4), device="cuda")
    with pytest.raises(ValueError, match="unknown policy 5"):
        csr.apply(X, missing=5)
    with pytest.raises(ValueError, match="variant"):
        csr.apply(X, missing=ALL, variant=1)


def _fieldlist(values, lat, lon):
    return ekd.from_source("list-of-dicts", [dict(values=v, latitudes=lat, longitudes=lon, param="sst", levelist=0, step=k) for k, v in enumerate(values)])


RECIPES = [
    ("o1280", "n320", "structured-bilinear"),
    ("o1280", "n320", "structured-conservative"),
    ("0.25deg", "o96", "structured-conservative"),
]


def _grid(name):
    if name.startswith("o"):
        return syn.octahedral(int(name[1:]))
    if name == "n320":
        return syn.n320_like()
    return syn.regular_latlon(float(name[:-3]))


@pytest.fixture(scope="module", params=RECIPES, ids=["-".join(r) for r in RECIPES])
def recipe(request, cuda):
    source, target, method = request.param
    s, t = _grid(source), _grid(target)
    m = oc.conservative_csr(*s, *t) if method == "structured-conservative" else om.structured_csr(*s, *t, 2)
    return s, t, method, m


@pytest.mark.parametrize("route", ["streamed", "resident"])
def test_recipes_at_full_size(F, recipe, route):
    from anemoi_transform_b200.device import results_stay_on_device

    (s_lat, s_lon), (t_lat, t_lon), method, m = recipe
    X = masked_values(s_lat, s_lon, 6, np.float32)
    values = [np.ascontiguousarray(X[:, k]) for k in range(X.shape[1])]
    for policy, name in NAMES.items():
        regrid = F("regrid", in_grid=dict(latitudes=s_lat, longitudes=s_lon), out_grid=dict(latitudes=t_lat, longitudes=t_lon), method=method, missing_values=name)
        if route == "streamed":
            out = regrid.forward(_fieldlist(values, s_lat, s_lon))
        else:
            with results_stay_on_device():
                out = regrid.forward(_fieldlist(values, s_lat, s_lon))
        want = csr_matvec_missing(m.indptr, m.indices, m.data, X, policy)
        n_recovered = 0
        for k, f in enumerate(out):
            got = f.to_numpy()
            assert_same_values(got, want[:, k], f"{method} {route} {name} field {k}")
            n_recovered += int(np.isnan(m @ values[k]).sum() - np.isnan(got).sum())
        assert n_recovered > 0


def test_grib_messages_with_bitmaps(F):
    from grib_fields import GribMessageField
    from oracle import grib as ogrib

    s_lat, s_lon = syn.octahedral(320)
    t_lat, t_lon = syn.regular_latlon(1.0)
    m = om.structured_csr(s_lat, s_lon, t_lat, t_lon, 2)
    rng = np.random.default_rng(8)
    fields = []
    for k in range(8):
        present = ~land_mask(s_lat, s_lon, 5 + (k % 3 == 0))
        if k == 0:
            present[:] = True
        v = rng.normal(290.0, 5.0, s_lat.size)[present]
        msg = (ogrib.encode_grib2 if k % 2 == 0 else ogrib.encode_grib1)(v, 16, 1, bitmap=present)
        fields.append(GribMessageField(msg, s_lat.size, dict(param="sst", levelist=0, step=k), latitudes=s_lat, longitudes=s_lon))
    X = np.stack([ogrib.decode(f.message(), n_points=s_lat.size) for f in fields], axis=1)
    for policy, name in NAMES.items():
        out = F("regrid", in_grid=dict(latitudes=s_lat, longitudes=s_lon), out_grid=dict(latitudes=t_lat, longitudes=t_lon), method="structured-bilinear", missing_values=name).forward(fields)
        want = csr_matvec_missing(m.indptr, m.indices, m.data, X, policy)
        for k, f in enumerate(out):
            assert_same_values(f.to_numpy(), want[:, k], f"grib edition {2 if k % 2 == 0 else 1} {name} field {k}")
    assert all(f.decodes == 0 for f in fields), "the GRIB fields were decoded on the host"


def test_two_engines_on_one_gpu_equal_one_engine(F, cuda, monkeypatch):
    s_lat, s_lon = syn.regular_latlon(0.25)
    t_lat, t_lon = syn.octahedral(96)
    m = oc.conservative_csr(s_lat, s_lon, t_lat, t_lon)
    X = masked_values(s_lat, s_lon, 30, np.float32, seed=2)
    values = [np.ascontiguousarray(X[:, k]) for k in range(X.shape[1])]
    d = cuda.cuda.current_device()
    for policy, name in NAMES.items():
        regrid = F("regrid", in_grid=dict(latitudes=s_lat, longitudes=s_lon), out_grid=dict(latitudes=t_lat, longitudes=t_lon), method="structured-conservative", missing_values=name)
        monkeypatch.delenv("AT_B200_DEVICES", raising=False)
        single = [f.to_numpy() for f in regrid.forward(_fieldlist(values, s_lat, s_lon))]
        monkeypatch.setenv("AT_B200_DEVICES", f"{d},{d}")
        group = [f.to_numpy() for f in regrid.forward(_fieldlist(values, s_lat, s_lon))]
        monkeypatch.delenv("AT_B200_DEVICES")
        want = csr_matvec_missing(m.indptr, m.indices, m.data, X, policy)
        for k in range(len(values)):
            assert_same_values(group[k], single[k], f"{name} group vs single, field {k}")
            assert_same_values(group[k], want[:, k], f"{name} group vs oracle, field {k}")


def test_a_missing_aware_regrid_runs_unfused_and_equals_the_chain(F):
    from anemoi_transform_b200.fusion import FusedRegrid
    from anemoi_transform_b200.source import FieldListSource

    s_lat, s_lon = syn.octahedral(48)
    land = land_mask(s_lat, s_lon)
    values = [syn.synthetic_field(p, s_lat.size, 30 + k) for k, p in enumerate(("q", "t"))]
    for v in values:
        v[land] = np.nan
    data = ekd.from_source("list-of-dicts", [dict(values=v, latitudes=s_lat, longitudes=s_lon, param=p, levelist=850) for v, p in zip(values, ("q", "t"))])
    for name in NAMES.values():
        filters = [F("regrid", in_grid="O48", out_grid=[2.5, 2.5], method="structured-bilinear", missing_values=name), F("q_to_r", return_inputs="none")]
        pipe = FieldListSource(dataset=data)
        for f in filters:
            pipe = pipe | f
        assert not any(isinstance(step, FusedRegrid) for step in pipe.execution_plan())
        got = pipe.forward(None)
        chain = data
        for f in filters:
            chain = f.forward(chain)
        assert [f.metadata("param") for f in got] == [f.metadata("param") for f in chain] == ["r"]
        for a, b in zip(got, chain):
            assert_same_values(a.to_numpy(flatten=True), b.to_numpy(flatten=True), name)
        assert not np.isnan(got[0].to_numpy()).all()


def test_gather_regrids_are_the_same_under_every_policy(F, tmp_path):
    s_lat, s_lon = syn.octahedral(48)
    t_lat, t_lon = syn.regular_latlon(5.0)
    X = masked_values(s_lat, s_lon, 5, np.float32)
    values = [np.ascontiguousarray(X[:, k]) for k in range(X.shape[1])]
    mask = np.arange(0, s_lat.size, 7)
    np.savez(tmp_path / "mask.npz", mask=mask)
    kinds = {
        "nearest": lambda name: F("regrid", in_grid=dict(latitudes=s_lat, longitudes=s_lon), out_grid=dict(latitudes=t_lat, longitudes=t_lon), method="nearest", missing_values=name),
        "mask": lambda name: F("regrid", mask=str(tmp_path / "mask.npz"), missing_values=name),
    }
    for kind, make in kinds.items():
        base = [f.to_numpy() for f in make(None).forward(_fieldlist(values, s_lat, s_lon))]
        if kind == "mask":
            for k, v in enumerate(values):
                assert_same_values(base[k], v[mask], f"mask field {k}")
        for name in NAMES.values():
            got = [f.to_numpy() for f in make(name).forward(_fieldlist(values, s_lat, s_lon))]
            for k in range(len(values)):
                assert_same_values(got[k], base[k], f"{kind} {name} field {k}")


def test_bad_missing_values_raise(F, tmp_path):
    s_lat, s_lon = syn.octahedral(16)
    t_lat, t_lon = syn.regular_latlon(10.0)
    d, i, p, shape = syn.bilinear_matrix(10.0, s_lat, s_lon)
    syn.save_regrid_npz(str(tmp_path / "m.npz"), d, i, p, shape, t_lat, t_lon, s_lat, s_lon)
    with pytest.raises(ValueError, match="missing_values='fraction'"):
        F("regrid", matrix=str(tmp_path / "m.npz"), missing_values="fraction")
    with pytest.raises(ValueError, match="missing_values='nonlinear'"):
        F("regrid", in_grid="O16", out_grid=[10.0, 10.0], method="structured-conservative", missing_values="nonlinear")
