"""pointwise_kernel on awkward shapes, for every epilogue kind: the transcendental tiles stream their rows through a
shared-memory ring (cp.async, four rows in flight) with one row loop per kind — a row's result
must not depend on how many rows, column tiles or spare warps the launch has.

Every case is checked twice: against the numpy oracle (oracle/pointwise.py, the restatement of
the earthkit-meteo formulas the reference calls: uv_to_ddff.py:94-98, q_to_r.py:71-80,
dewpoint.py:62-74; rescale, lnsp_to_sp, impute_nans and cos_sin_* as numpy) within 1e-6 of the
field's range, every output column with its own pressure, and bitwise against the same kernel run one
row at a time (n_rows = 1: no ring wrap-around, no row sharing between warps).
"""

from __future__ import annotations

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _inputs(kind_name, n_rows, n_cols, dtype, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n_rows, n_cols))
    if kind_name in ("uv2ddff", "atan2"):
        x *= 8.0
    elif kind_name == "ddff2uv":
        x[:, 0::2] = np.abs(x[:, 0::2]) * 10
        x[:, 1::2] = (x[:, 1::2] * 100) % 360
    elif kind_name in ("qt2r", "qt2qtr"):
        x[:, 0::2] = np.abs(x[:, 0::2]) * 1e-3
        x[:, 1::2] = x[:, 1::2] * 15 + 270
    elif kind_name in ("rt2q", "rt2d", "rt2rtq", "rt2rtd"):
        x[:, 0::2] = np.clip(np.abs(x[:, 0::2]) * 40, 0.5, 100.0)
        x[:, 1::2] = x[:, 1::2] * 15 + 270
    elif kind_name in ("dt2r", "dt2dtr"):  # (td, t) with td <= t: r from a few % to 100 %
        x[:, 1::2] = x[:, 1::2] * 8 + 285
        x[:, 0::2] = x[:, 1::2] - np.abs(x[:, 0::2]) * 20
    elif kind_name in ("affine", "affine_inv"):  # temperatures: the result's rounding stays far inside 1e-6 of its range
        x = x * 40.0 + 270.0
    elif kind_name == "log":
        x = np.abs(x) + 0.05
    elif kind_name == "cossin":
        x *= 3.0
    elif kind_name == "impute_nan":
        x[rng.random(x.shape) < 0.2] = np.nan
    return x.astype(dtype)


def _oracle(kind_name, x, pressure, pa, pb):
    """Outputs of `kind_name` on x (float64), with `pressure` the pressure of each (q | r, t)
    pair's output column and pa / pb the segment's constants rounded to float32 as numpy rounds
    a Python float against a float32 array (NEP 50)."""
    from oracle import pointwise as pw

    a, b = x[:, 0::2], x[:, 1::2]

    def interleave(*cols):
        out = np.empty((x.shape[0], cols[0].shape[1] * len(cols)))
        for i, c in enumerate(cols):
            out[:, i :: len(cols)] = c
        return out

    if kind_name == "uv2ddff":
        return interleave(*pw.xy_to_polar(a, b))
    if kind_name == "ddff2uv":
        return interleave(*pw.polar_to_xy(a, b))
    if kind_name == "qt2r":
        return pw.relative_humidity_from_specific_humidity(b, a, pressure)
    if kind_name == "qt2qtr":
        return interleave(a, b, pw.relative_humidity_from_specific_humidity(b, a, pressure))
    if kind_name == "rt2q":
        return pw.specific_humidity_from_relative_humidity(b, a, pressure)
    if kind_name == "rt2rtq":
        return interleave(a, b, pw.specific_humidity_from_relative_humidity(b, a, pressure))
    if kind_name == "rt2d":
        return pw.dewpoint_from_relative_humidity(b, a)
    if kind_name == "rt2rtd":
        return interleave(a, b, pw.dewpoint_from_relative_humidity(b, a))
    if kind_name == "dt2r":
        return pw.relative_humidity_from_dewpoint(b, a)
    if kind_name == "dt2dtr":
        return interleave(a, b, pw.relative_humidity_from_dewpoint(b, a))
    if kind_name == "atan2":
        return np.arctan2(b, a)
    if kind_name == "affine":
        return x * pa + pb
    if kind_name == "affine_inv":
        return (x - pb) / pa
    if kind_name == "exp":
        return np.exp(x)
    if kind_name == "log":
        return np.log(x)
    if kind_name == "impute_nan":
        return np.where(np.isnan(x), pa, x)
    if kind_name == "cossin":
        return interleave(np.cos(x * pa), np.sin(x * pa))
    raise AssertionError(kind_name)


# name: (AT_EPI_* constant, inputs per group, outputs per group, pa, pb)
KINDS = {
    "uv2ddff": ("EPI_UV2DDFF", 2, 2, 1.0, 0.0),
    "ddff2uv": ("EPI_DDFF2UV", 2, 2, 1.0, 0.0),
    "qt2r": ("EPI_QT2R", 2, 1, 1.0, 0.0),
    "qt2qtr": ("EPI_QT2QTR", 2, 3, 1.0, 0.0),
    "rt2q": ("EPI_RT2Q", 2, 1, 1.0, 0.0),
    "rt2rtq": ("EPI_RT2RTQ", 2, 3, 1.0, 0.0),
    "rt2d": ("EPI_RT2D", 2, 1, 1.0, 0.0),
    "rt2rtd": ("EPI_RT2RTD", 2, 3, 1.0, 0.0),
    "dt2r": ("EPI_DT2R", 2, 1, 1.0, 0.0),
    "dt2dtr": ("EPI_DT2DTR", 2, 3, 1.0, 0.0),
    "atan2": ("EPI_ATAN2", 2, 1, 1.0, 0.0),
    "affine": ("EPI_AFFINE", 1, 1, 1.8, -459.67),  # rescale K -> F (rescale.py)
    "affine_inv": ("EPI_AFFINE_INV", 1, 1, 1.8, -459.67),
    "exp": ("EPI_EXP", 1, 1, 1.0, 0.0),
    "log": ("EPI_LOG", 1, 1, 1.0, 0.0),
    "impute_nan": ("EPI_IMPUTE_NAN", 1, 1, -1.5, 0.0),
    "cossin": ("EPI_COSSIN", 1, 2, 1.0, 0.0),
}
# the output column of each (q | r, t) pair whose pressure the kernel reads (epilogue_prepare)
P_COL = {"qt2r": (1, 0), "rt2q": (1, 0), "qt2qtr": (3, 2), "rt2rtq": (3, 2)}


@pytest.mark.parametrize("kind_name", sorted(KINDS))
@pytest.mark.parametrize("n_rows", [1, 2, 3, 5, 31, 32, 33, 97])
@pytest.mark.parametrize("n_cols", [8, 40, 136, 1032])
def test_rows_do_not_depend_on_the_launch_shape(cuda, kind_name, n_rows, n_cols):
    import torch

    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.device import Epilogue

    const, n_in, n_out, pa, pb = KINDS[kind_name]
    n_out_cols = n_cols // n_in * n_out
    # every output column its own pressure: a pair that read another column's would be off
    col_p = 50000.0 + 1000.0 * np.arange(n_out_cols)
    stride, off = P_COL.get(kind_name, (1, 0))
    pressure = col_p[off::stride].astype(np.float32).astype(np.float64)
    x = _inputs(kind_name, n_rows, n_cols, np.float32, seed=n_rows * 1000 + n_cols)
    epi = Epilogue([(getattr(_cabi, const), 0, n_cols, 0, pa, pb)], [(0.0, 0.0, p, 0) for p in col_p])
    X = torch.from_numpy(x).cuda()
    Y = torch.full((n_rows, (n_out_cols + 3) // 4 * 4), -7.0, device="cuda")
    got = epi.apply(X, out=Y).cpu().numpy()[:, :n_out_cols]

    with np.errstate(all="ignore"):
        want = _oracle(kind_name, x.astype(np.float64), pressure, float(np.float32(pa)), float(np.float32(pb)))
    span = float(np.nanmax(want) - np.nanmin(want)) or 1.0
    if kind_name in ("uv2ddff",):  # directions wrap at 360
        d = np.abs(got.astype(np.float64) - want)
        d[:, 1::2] = np.minimum(d[:, 1::2], 360.0 - d[:, 1::2])
        assert d[:, 0::2].max() <= 1e-6 * span and d[:, 1::2].max() <= 360e-6
    else:
        assert np.array_equal(np.isnan(got), np.isnan(want)), kind_name
        ok = ~np.isnan(want)
        assert np.abs(got[ok].astype(np.float64) - want[ok]).max() <= 1e-6 * span, kind_name

    # one row at a time: bitwise the same
    for r in sorted({0, n_rows // 2, n_rows - 1}):
        y1 = torch.empty((1, Y.shape[1]), device="cuda")
        one = epi.apply(X[r : r + 1].contiguous(), out=y1).cpu().numpy()[0, :n_out_cols]
        assert np.array_equal(one.view(np.uint32), got[r].view(np.uint32)), (kind_name, n_rows, n_cols, r)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_ring_with_row_gather_mask_and_clip(cuda, dtype):
    """The fused nearest-neighbour form: Y[r] = epilogue(X[gather[r]]) with a row mask and clip
    bounds, more rows than one CTA, a ragged last CTA and a ragged last column tile."""
    import torch

    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.device import Epilogue
    from oracle import pointwise as pw

    n_src, n_rows, n_cols = 211, 173, 264
    x = _inputs("uv2ddff", n_src, n_cols, dtype, seed=5)
    rng = np.random.default_rng(6)
    gather = rng.integers(0, n_src, n_rows)
    mask = (rng.random(n_rows) < 0.3).astype(np.uint8)
    CL, CH, MK = _cabi.COL_CLIP_LO, _cabi.COL_CLIP_HI, _cabi.COL_MASK
    cols = [(1.0, 9.0, 0.0, CL | CH | MK), (0.0, 0.0, 0.0, 0)] * (n_cols // 2)
    epi = Epilogue([(_cabi.EPI_UV2DDFF, 0, n_cols, 0, 1.0, 0.0)], cols)
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    X = torch.from_numpy(x).cuda()
    Y = torch.empty((n_rows, n_cols), device="cuda", dtype=tdt)
    got = epi.apply(X, out=Y, row_mask=torch.from_numpy(mask).cuda(), gather=torch.from_numpy(gather).cuda()).cpu().numpy()

    xs = x[gather].astype(np.float64)
    ws, wd = pw.xy_to_polar(xs[:, 0::2], xs[:, 1::2])
    ws = np.clip(ws, 1.0, 9.0)
    ws[mask != 0] = np.nan
    tol = 1e-6 if dtype == np.float32 else 1e-12
    assert np.array_equal(np.isnan(got[:, 0::2]), np.isnan(ws))
    ok = ~np.isnan(ws)
    assert np.abs(got[:, 0::2][ok] - ws[ok]).max() <= tol * 8.0
    d = np.abs(got[:, 1::2].astype(np.float64) - wd)
    assert np.minimum(d, 360.0 - d).max() <= 360 * tol


@pytest.mark.parametrize("n_cols", [4, 8, 40, 68, 136])
@pytest.mark.parametrize("n_rows", [1, 7, 32, 33, 200])
def test_copy_like_tiles_pack_rows_into_narrow_warps(cuda, n_rows, n_cols):
    """clip + mask (np.clip, values[mask] = nan — clipper.py:69, apply_mask.py:185) on column
    counts whose last tile is narrower than half a warp: exact."""
    import torch

    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.device import Epilogue

    rng = np.random.default_rng(n_rows * 100 + n_cols)
    x = rng.standard_normal((n_rows, n_cols)).astype(np.float32)
    x[rng.random(x.shape) < 0.01] = np.nan
    mask = (rng.random(n_rows) < 0.3).astype(np.uint8)
    CL, CH, MK = _cabi.COL_CLIP_LO, _cabi.COL_CLIP_HI, _cabi.COL_MASK
    cols = [(-0.5, 0.75, 0.0, CL | CH | (MK if c % 3 == 0 else 0)) for c in range(n_cols)]
    epi = Epilogue([(_cabi.EPI_PLAIN, 0, n_cols, 0, 1.0, 0.0)], cols)
    got = epi.apply(torch.from_numpy(x).cuda(), row_mask=torch.from_numpy(mask).cuda()).cpu().numpy()[:, :n_cols]
    want = np.clip(x, np.float32(-0.5), np.float32(0.75))
    want[np.ix_(mask != 0, np.arange(n_cols) % 3 == 0)] = np.nan
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.array_equal(got[ok].view(np.uint32), want[ok].view(np.uint32))


@pytest.mark.parametrize("nnz_per_row", [4, 12, 0])
@pytest.mark.parametrize("n_cols", [8, 40, 136, 264])
def test_fused_narrow_tiles_equal_the_unfused_chain(cuda, nnz_per_row, n_cols):
    """spmm_fused_kernel packs several target rows into a warp when a tile is narrower than half
    a warp (every lane walks its own row's CSR entries): bitwise the SpMM followed by the
    standalone epilogue, on uniform 4- and 12-nonzero rows and on ragged rows (0 = rows of 0..9
    entries, empty rows included)."""
    import torch
    from scipy.sparse import csr_array

    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.device import CsrMatrix, Epilogue

    rng = np.random.default_rng(nnz_per_row * 1000 + n_cols)
    n_tgt, n_src = 333, 517
    lengths = np.full(n_tgt, nnz_per_row) if nnz_per_row else rng.integers(0, 10, n_tgt)
    indptr = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
    indices = np.concatenate([np.sort(rng.choice(n_src, k, replace=False)) for k in lengths] + [np.empty(0, np.int64)]).astype(np.int32)
    data = rng.random(indices.size).astype(np.float32)
    x = (rng.standard_normal((n_src, n_cols)) * 8.0).astype(np.float32)
    mask = (rng.random(n_tgt) < 0.3).astype(np.uint8)
    CL, CH, MK = _cabi.COL_CLIP_LO, _cabi.COL_CLIP_HI, _cabi.COL_MASK
    half = n_cols // 8 * 4  # first half (u, v) -> (ws, wdir), second half clip + mask only
    segs = [(_cabi.EPI_UV2DDFF, 0, half, 0), (_cabi.EPI_PLAIN, half, n_cols - half, half)]
    cols = [(0.5, 30.0, 0.0, CL | CH | MK), (0.0, 0.0, 0.0, 0)] * (half // 2) + [(-4.0, 4.0, 0.0, CL | CH | MK)] * (n_cols - half)
    epi = Epilogue(segs, cols)
    csr = CsrMatrix(data, indices, indptr, (n_tgt, n_src))
    X = torch.from_numpy(x).cuda()
    M = torch.from_numpy(mask).cuda()
    fused = epi.apply_fused(csr, X, row_mask=M).cpu().numpy()[:, :n_cols]
    y = csr.apply(X, n_fields=n_cols)
    unfused = epi.apply(y, row_mask=M).cpu().numpy()[:, :n_cols]
    assert np.array_equal(np.isnan(fused), np.isnan(unfused))
    ok = ~np.isnan(fused)
    assert np.array_equal(fused[ok].view(np.uint32), unfused[ok].view(np.uint32))
    # and the SpMM half against scipy, bit for bit
    want = np.stack([csr_array((data, indices, indptr), shape=(n_tgt, n_src)) @ x[:, c] for c in (0, n_cols - 1)], axis=1)
    got = y.cpu().numpy()[:, [0, n_cols - 1]]
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
