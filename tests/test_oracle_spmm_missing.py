"""The missing-value SpMM oracle (oracle/spmm_missing.py), the C-ABI refusals of
`at_spmm_missing` and the missing-value ops of `at_hostio_regrid*`, and the
`missing_values=` argument of `regrid` (CPU only)."""

import ctypes

import numpy as np
import pytest

from anemoi_transform_b200 import synthetic as syn
from oracle import conservative_matrix as oc
from oracle import structured_matrix as om
from oracle.spmm import csr_matvec_sequential
from oracle.spmm_missing import ALL, HEAVIEST, PROPAGATE, csr_matvec_missing, heaviest_entries

POLICIES = (PROPAGATE, ALL, HEAVIEST)
DTYPES = [(np.float32, np.float32), (np.float64, np.float32), (np.float32, np.float64), (np.float64, np.float64)]


def _random_csr(rng, n_rows, n_cols, max_len, wdt, *, empty=0.1, zeros=0.1, negative=0.2, ties=0.2):
    """Random CSR with empty rows, explicit zeros, negative weights, duplicate columns and tied
    heaviest weights."""
    lengths = rng.integers(0, max_len + 1, n_rows)
    lengths[rng.random(n_rows) < empty] = 0
    indptr = np.concatenate(([0], np.cumsum(lengths))).astype(np.int32)
    nnz = int(indptr[-1])
    indices = rng.integers(0, n_cols, nnz).astype(np.int32)
    data = rng.random(nnz).astype(wdt)
    data[rng.random(nnz) < negative] *= -1
    data[rng.random(nnz) < zeros] = 0
    for r in np.nonzero((rng.random(n_rows) < ties) & (lengths >= 2))[0]:
        p0 = indptr[r]
        data[p0 + 1 : indptr[r + 1]] = np.minimum(data[p0 + 1 : indptr[r + 1]], data[p0])
        data[indptr[r + 1] - 1] = data[p0] = abs(data[p0]) + 1  # first and last entries tie
    return indptr, indices, data


def _loop_reference(indptr, indices, data, x, policy):
    """The contract restated per row and per field with numpy scalars."""
    dtype = np.result_type(data.dtype, x.dtype)
    t = dtype.type
    y = np.zeros(len(indptr) - 1, dtype=dtype)
    with np.errstate(invalid="ignore", over="ignore"):
        _loop_rows(indptr, indices, data, x, policy, t, y)
    return y


def _loop_rows(indptr, indices, data, x, policy, t, y):
    for r in range(len(indptr) - 1):
        p0, p1 = int(indptr[r]), int(indptr[r + 1])
        heaviest = p0
        for p in range(p0 + 1, p1):
            if data[p] > data[heaviest]:
                heaviest = p
        acc, ws, missing, heaviest_missing = t(0), t(0), False, False
        for p in range(p0, p1):
            w, v = t(data[p]), t(x[indices[p]])
            if policy != PROPAGATE and np.isnan(v):
                missing = True
                heaviest_missing |= p == heaviest
                continue
            acc = t(acc + t(w * v))
            ws = t(ws + w)
        if not missing:
            y[r] = acc
        elif (policy == HEAVIEST and heaviest_missing) or not ws > 0:
            y[r] = np.nan
        else:
            y[r] = t(acc / ws)


def _same(a, b, what=""):
    assert a.dtype == b.dtype, what
    assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}: NaN positions differ"
    ok = ~np.isnan(a)
    view = {4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
    assert np.array_equal(a[ok].view(view), b[ok].view(view)), f"{what}: values differ bitwise"


@pytest.mark.parametrize("wdt,xdt", DTYPES)
@pytest.mark.parametrize("policy", POLICIES)
def test_nan_free_inputs_are_the_plain_spmm(wdt, xdt, policy):
    rng = np.random.default_rng(1)
    indptr, indices, data = _random_csr(rng, 300, 200, 20, wdt)
    for seed in range(3):
        x = (np.random.default_rng(seed).standard_normal(200) * 10 ** seed).astype(xdt)
        x[:3] = [np.inf, -np.inf, 0.0]  # Inf is not missing
        _same(csr_matvec_missing(indptr, indices, data, x, policy), csr_matvec_sequential(indptr, indices, data, x), f"policy {policy}")


@pytest.mark.parametrize("wdt,xdt", DTYPES)
@pytest.mark.parametrize("policy", POLICIES)
def test_matches_the_per_row_loop_with_missing_values(wdt, xdt, policy):
    rng = np.random.default_rng(7)
    for trial in range(4):
        n_cols = 60
        indptr, indices, data = _random_csr(rng, 150, n_cols, 12, wdt)
        x = rng.standard_normal(n_cols).astype(xdt)
        x[rng.random(n_cols) < 0.3] = np.nan
        x[0] = np.inf
        # a row whose sources are all missing, and one whose heaviest entry is missing
        nan_cols = np.nonzero(np.isnan(x))[0]
        indices[indptr[5] : indptr[6]] = nan_cols[: indptr[6] - indptr[5]] if indptr[6] - indptr[5] <= nan_cols.size else indices[indptr[5] : indptr[6]]
        want = _loop_reference(indptr, indices, data, x, policy)
        _same(csr_matvec_missing(indptr, indices, data, x, policy), want, f"trial {trial} policy {policy}")


def test_a_batch_of_fields_is_each_field_on_its_own():
    rng = np.random.default_rng(3)
    indptr, indices, data = _random_csr(rng, 100, 80, 10, np.float32)
    X = rng.standard_normal((80, 7)).astype(np.float32)
    X[rng.random(X.shape) < 0.3] = np.nan
    X[:, 3] = np.nan
    X[:, 4] = 1.0
    for policy in POLICIES:
        Y = csr_matvec_missing(indptr, indices, data, X, policy)
        for f in range(X.shape[1]):
            _same(Y[:, f], csr_matvec_missing(indptr, indices, data, np.ascontiguousarray(X[:, f]), policy), f"policy {policy} field {f}")


def test_heaviest_is_the_first_of_tied_weights_and_none_for_an_empty_row():
    indptr = np.array([0, 3, 3, 6, 7])
    data = np.array([1.0, 2.0, 2.0, -1.0, -3.0, -1.0, 0.0], dtype=np.float32)
    assert heaviest_entries(indptr, data).tolist() == [1, -1, 3, 6]


def test_worked_examples():
    # a bilinear target on a missing source: the other entries are explicit zeros -> NaN
    indptr, indices = np.array([0, 4]), np.array([0, 1, 2, 3])
    data = np.array([1.0, 0.0, 0.0, 0.0], dtype=np.float32)
    x = np.array([np.nan, 1.0, 2.0, 3.0], dtype=np.float32)
    assert np.isnan(csr_matvec_missing(indptr, indices, data, x, ALL)[0])
    # bicubic-like weights whose valid part sums to <= 0 -> NaN; > 0 -> renormalised
    data = np.array([0.5, -0.25, 0.5, 0.25], dtype=np.float32)
    x = np.array([np.nan, 4.0, np.nan, 8.0], dtype=np.float32)
    assert np.isnan(csr_matvec_missing(indptr, indices, data, x, ALL)[0])
    x = np.array([1.0, np.nan, 3.0, 5.0], dtype=np.float32)
    assert csr_matvec_missing(indptr, indices, data, x, ALL)[0] == np.float32(0.5 + 1.5 + 1.25) / np.float32(1.25)
    # heaviest: entry 0 (first of the tied 0.5) missing -> NaN; entry 2 missing is not the heaviest
    x = np.array([np.nan, 1.0, 3.0, 5.0], dtype=np.float32)
    assert np.isnan(csr_matvec_missing(indptr, indices, data, x, HEAVIEST)[0])
    x = np.array([1.0, 1.0, np.nan, 5.0], dtype=np.float32)
    assert not np.isnan(csr_matvec_missing(indptr, indices, data, x, HEAVIEST)[0])
    with pytest.raises(ValueError, match="policy"):
        csr_matvec_missing(indptr, indices, data, x, 3)


def _land_mask(lat, lon, seed):
    """About 30 % of the points missing, in coherent blobs (coasts) rather than scattered."""
    rng = np.random.default_rng(seed)
    la, lo = np.radians(lat), np.radians(lon)
    v = np.zeros(lat.size)
    for k in range(12):
        c_la, c_lo = np.arcsin(rng.uniform(-1, 1)), rng.uniform(0, 2 * np.pi)
        v += np.exp(-((np.cos(la) * np.cos(c_la) * np.cos(lo - c_lo) + np.sin(la) * np.sin(c_la)) - 1) ** 2 * 8)
    return v > np.quantile(v, 0.7)


MATRICES = {
    "structured-bilinear O32 -> 2.5°": lambda: (syn.octahedral(32), om.structured_csr(*syn.octahedral(32), *syn.regular_latlon(2.5), 2)),
    "structured-conservative O48 -> 5°": lambda: (syn.octahedral(48), oc.conservative_csr(*syn.octahedral(48), *syn.regular_latlon(5.0))),
    "structured-conservative 2° -> O24": lambda: (syn.regular_latlon(2.0), oc.conservative_csr(*syn.regular_latlon(2.0), *syn.octahedral(24))),
}


@pytest.mark.parametrize("name", list(MATRICES))
def test_properties_on_non_negative_regrid_matrices(name):
    (lat, lon), m = MATRICES[name]()
    assert (m.data >= 0).all()
    indptr, indices, data = m.indptr, m.indices, m.data
    land = _land_mask(lat, lon, 5)
    x = (np.sin(np.radians(lat)) * 30 + np.cos(np.radians(2 * lon)) * 5 + 280).astype(np.float32)
    x[land] = np.nan
    lengths = np.diff(indptr)
    rows = np.repeat(np.arange(m.shape[0]), lengths)
    valid = ~np.isnan(x[indices])
    lo = np.full(m.shape[0], np.inf)
    hi = np.full(m.shape[0], -np.inf)
    np.minimum.at(lo, rows[valid], x[indices][valid])
    np.maximum.at(hi, rows[valid], x[indices][valid])

    y_all = csr_matvec_missing(indptr, indices, data, x, ALL)
    y_prop = csr_matvec_missing(indptr, indices, data, x, PROPAGATE)
    assert np.isnan(y_prop).sum() > np.isnan(y_all).sum(), "skipping missing sources recovers targets"
    ok = ~np.isnan(y_all)
    tol = 1e-6 * np.maximum(np.abs(lo[ok]), np.abs(hi[ok]))
    assert (y_all[ok] >= lo[ok] - tol).all() and (y_all[ok] <= hi[ok] + tol).all(), "result outside [min, max] of the valid sources"
    # NaN exactly where no valid source has a positive weight
    pos_valid = np.zeros(m.shape[0], dtype=bool)
    pos_valid[rows[valid & (data > 0)]] = True
    assert np.array_equal(ok, pos_valid)

    # a constant field with holes stays constant
    c = np.where(land, np.float32(np.nan), np.float32(273.15)).astype(np.float32)
    yc = csr_matvec_missing(indptr, indices, data, c, ALL)
    okc = ~np.isnan(yc)
    assert np.array_equal(okc, pos_valid)
    assert np.abs(yc[okc] / np.float32(273.15) - 1).max() <= 1e-6

    # heaviest: NaN wherever the row's heaviest source is missing, else what ALL gives
    y_h = csr_matvec_missing(indptr, indices, data, x, HEAVIEST)
    hp = heaviest_entries(indptr, data)
    heavy_missing = (hp >= 0) & np.isnan(x[indices[np.maximum(hp, 0)]])
    assert heavy_missing.any()
    assert np.isnan(y_h[heavy_missing]).all()
    _same(y_h[~heavy_missing], y_all[~heavy_missing], "heaviest present: as all-missing")


# ---- C-ABI refusals (no device needed: the checks come before any CUDA call) ----------
def test_unknown_policy_is_refused_with_a_message(native_library):
    from anemoi_transform_b200 import _cabi

    buf = (ctypes.c_float * 16)()
    rc = native_library.at_spmm_missing(None, ctypes.cast(buf, ctypes.c_void_p), _cabi.AT_F32, 4, ctypes.cast(buf, ctypes.c_void_p), _cabi.AT_F32, 4, 4, 7, None)
    assert rc == _cabi.AT_ERR_INVALID
    assert b"unknown policy 7" in native_library.at_last_error()
    # a known policy gets as far as at_spmm's own checks
    rc = native_library.at_spmm_missing(None, None, _cabi.AT_F32, 4, None, _cabi.AT_F32, 4, 4, _cabi.MISSING_ALL, None)
    assert rc == _cabi.AT_ERR_INVALID and b"null argument" in native_library.at_last_error()


@pytest.mark.parametrize("entry", ["at_hostio_regrid", "at_hostio_regrid_grib", "at_hostio_group_regrid"])
def test_unknown_hostio_op_is_refused_with_a_message(native_library, entry):
    from anemoi_transform_b200 import _cabi

    fn = getattr(native_library, entry)
    n_args = len(_cabi.PROTOTYPES[entry][1])
    for op, answer in ((9, b"unknown op 9"), (_cabi.HOSTIO_SPMM_MISSING_ALL, b"null argument"), (_cabi.HOSTIO_SPMM_MISSING_HEAVIEST, b"null argument")):
        args = [None] * n_args
        args[1] = op
        for k, t in enumerate(_cabi.PROTOTYPES[entry][1]):
            if t in (ctypes.c_int, ctypes.c_int32, ctypes.c_int64) and k != 1:
                args[k] = 0
        assert fn(*args) == _cabi.AT_ERR_INVALID
        assert answer in native_library.at_last_error(), (entry, op)


def test_header_declares_the_policies_and_ops():
    from conftest import REPO

    from anemoi_transform_b200 import _cabi

    header = (REPO / "include" / "at_b200.h").read_text()
    for name, value in (
        ("AT_MISSING_PROPAGATE", _cabi.MISSING_PROPAGATE),
        ("AT_MISSING_ALL", _cabi.MISSING_ALL),
        ("AT_MISSING_HEAVIEST", _cabi.MISSING_HEAVIEST),
        ("AT_HOSTIO_SPMM_MISSING_ALL", _cabi.HOSTIO_SPMM_MISSING_ALL),
        ("AT_HOSTIO_SPMM_MISSING_HEAVIEST", _cabi.HOSTIO_SPMM_MISSING_HEAVIEST),
    ):
        assert f"#define {name} {value}\n" in header, name


# ---- regrid(missing_values=…) ------------------------------------------------------
def test_bad_missing_values_raise_at_construction(tmp_path):
    from anemoi_transform_b200.filters.fields.regrid import RegridFilter

    np.savez(tmp_path / "mask.npz", mask=np.array([0, 2]))
    for kwargs in (
        dict(out_grid=[5.0, 5.0], method="structured-bilinear"),
        dict(in_grid=[10.0, 10.0], out_grid=[5.0, 5.0], method="nearest"),
        dict(mask=str(tmp_path / "mask.npz")),
        dict(matrix=str(tmp_path / "does-not-matter.npz")),
    ):
        for bad in ("missing", "nonlinear", "", 1):
            with pytest.raises(ValueError, match=rf"missing_values={bad!r}.*'propagate', 'missing-if-all-missing', 'missing-if-heaviest-missing'"):
                RegridFilter(**kwargs, missing_values=bad)


def test_gather_regrids_accept_every_policy(tmp_path):
    from anemoi_transform_b200.filters.fields.regrid import MISSING_VALUES, RegridFilter

    np.savez(tmp_path / "mask.npz", mask=np.array([0, 2]))
    for name in (None, *MISSING_VALUES):
        RegridFilter(mask=str(tmp_path / "mask.npz"), missing_values=name)
        RegridFilter(in_grid=[10.0, 10.0], out_grid=[5.0, 5.0], method="nearest", missing_values=name)


def test_a_regrid_that_skips_missing_values_is_not_fused():
    from anemoi_transform_b200.filters.fields.regrid import RegridFilter
    from anemoi_transform_b200.fusion import is_fusable_regrid

    assert is_fusable_regrid(RegridFilter(out_grid=[5.0, 5.0], method="structured-bilinear"))
    assert is_fusable_regrid(RegridFilter(out_grid=[5.0, 5.0], method="structured-bilinear", missing_values="propagate"))
    for name in ("missing-if-all-missing", "missing-if-heaviest-missing"):
        assert not is_fusable_regrid(RegridFilter(out_grid=[5.0, 5.0], method="structured-bilinear", missing_values=name))
        # one source per target: every policy gives the same result, the gathers stay fusable
        assert is_fusable_regrid(RegridFilter(in_grid=[10.0, 10.0], out_grid=[5.0, 5.0], method="nearest", missing_values=name))
