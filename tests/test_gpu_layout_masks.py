"""The small layout and mask kernels every filter chain runs through, against numpy.

`at_gather_rows`, `at_gather_cols`, `at_compare_mask`, `at_sum_cols` and `at_range_flags`
(csrc/layout.cu), `at_compact_mask` and `at_cropping_mask` (csrc/masks.cu), called through
their `device.py` wrappers at the shapes that select each code path: the 16-byte and the
scalar row gathers, one and many column tiles, more than 32 output columns per warp, the
grid-stride row loop, more than one 1 024-block pass of the compaction scan, unaligned
byte views.  The reference is the numpy statement the filters restate, in the array's own
dtype as numpy evaluates it; results are compared bit for bit (NaN in the same places, the
sign of zero kept).
"""

from __future__ import annotations

import operator

import numpy as np
import pytest
from conftest import assert_same_values

from anemoi_transform_b200 import ekd

pytestmark = pytest.mark.gpu

DTYPES = [np.float32, np.float64]


@pytest.fixture(scope="module")
def dev(cuda):
    from anemoi_transform_b200 import device

    return device


@pytest.fixture(scope="module")
def F(cuda):
    from anemoi_transform_b200.filters import create_filter_by_name

    return create_filter_by_name


@pytest.fixture(scope="module")
def n_sms(cuda):
    return cuda.cuda.get_device_properties(0).multi_processor_count


def _round_up(n, m):
    return (n + m - 1) // m * m


def _specials(rng, shape, dtype):
    """Normal values with NaN, ±inf and −0.0 sprinkled in."""
    a = rng.normal(size=shape).astype(dtype)
    flat = a.reshape(-1)
    k = max(1, flat.size // 50)
    for v in (np.nan, -0.0, np.inf, -np.inf):
        flat[rng.integers(0, flat.size, k)] = v
    return a


def _poison(cuda, shape, dtype):
    """Free a NaN-filled block of the size the wrapper is about to allocate: the caching
    allocator hands it back, so anything the call leaves unwritten shows as NaN."""
    t = cuda.full(shape, float("nan"), dtype=dtype, device="cuda")
    del t


def _to_dev(cuda, a):
    return cuda.from_numpy(np.ascontiguousarray(a)).cuda()


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view({4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


# ---- at_gather_rows ------------------------------------------------------------------------
# path: how X and out are laid out, which selects the kernel
#   vec16      aligned rows, ld a multiple of 16 bytes: 16-byte chunks, padding columns copied
#   odd_ld     ld % per16 != 0: the scalar kernel (uint32_t / uint2)
#   x_offset   X a view starting one element into its rows: aligned ld, misaligned pointer
#   out_offset an explicit out starting one element into its rows
PATHS = ["vec16", "odd_ld", "x_offset", "out_offset"]


def _gather_source(rng, path, dtype, n_src, w):
    """(base host array, column offset of X in it) for an X of w columns."""
    per16 = 16 // np.dtype(dtype).itemsize
    if path == "odd_ld":
        ld, off = _round_up(w, per16) + 1, 0
    elif path == "x_offset":
        ld, off = _round_up(w + 1, 4), 1
    else:
        ld, off = _round_up(w, 4), 0
    return _specials(rng, (n_src, ld), dtype), off


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("fields", ["1", "3", "4", "5", "tile-1", "tile+1", "3120"])
def test_gather_rows(cuda, dev, dtype, path, fields):
    per16 = 16 // np.dtype(dtype).itemsize
    n_fields = {"tile-1": per16 * 128 - 1, "tile+1": per16 * 128 + 1}.get(fields) or int(fields)
    rng = np.random.default_rng(n_fields * 7 + PATHS.index(path))
    n_src, n_out, w = 300, 1001, n_fields + 2  # X wider than the n_fields gathered
    base, off = _gather_source(rng, path, dtype, n_src, w)
    idx = rng.integers(0, n_src, n_out)
    idx[:4] = [n_src - 1, 0, 0, n_src - 1]  # both ends, duplicates, unsorted
    xb = _to_dev(cuda, base)
    X = xb[:, off : off + w]
    d_idx = _to_dev(cuda, idx)
    want = base[idx, off : off + n_fields]
    if path == "out_offset":
        sentinel = dtype(7.25)
        ob = cuda.full((n_out, _round_up(w + 1, 4)), float(sentinel), dtype=xb.dtype, device="cuda")
        res = dev.gather_rows(X, d_idx, n_fields=n_fields, out=ob[:, 1 : 1 + w])
        got = ob.cpu().numpy()
        assert_same_values(got[:, 1 : 1 + n_fields], want, "gathered columns")
        rest = np.concatenate([got[:, :1], got[:, 1 + n_fields :]], axis=1)
        assert (rest == sentinel).all(), "scalar gather wrote outside the n_fields columns of out"
        assert res.data_ptr() == ob.data_ptr() + ob.element_size()
        return
    _poison(cuda, (n_out, _round_up(w, 4)), xb.dtype)
    got = dev.gather_rows(X, d_idx, n_fields=n_fields).cpu().numpy()
    assert got.shape == (n_out, _round_up(w, 4))
    assert_same_values(got[:, :n_fields], want, "gathered columns")
    pad = np.zeros((n_out, got.shape[1] - n_fields), dtype)
    if path == "vec16":
        # whole 16-byte chunks: columns up to the next chunk boundary are X's own storage there
        r = _round_up(n_fields, per16)
        pad[:, : r - n_fields] = base[idx, n_fields:r]
    assert np.array_equal(_bits(got[:, n_fields:]), _bits(pad)), f"padding columns of the {path} path"


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_gather_rows_bad_index_and_empty(cuda, dev, dtype, path):
    rng = np.random.default_rng(5)
    n_src, n_fields = 40, 5
    base, off = _gather_source(rng, path, dtype, n_src, n_fields)
    xb = _to_dev(cuda, base)
    X = xb[:, off : off + n_fields]

    def run(idx):
        d_idx = cuda.tensor(idx, dtype=cuda.int64, device="cuda")
        if path == "out_offset":
            ob = cuda.zeros((len(idx), 12), dtype=xb.dtype, device="cuda")
            return dev.gather_rows(X, d_idx, out=ob[:, 1 : 1 + n_fields])
        return dev.gather_rows(X, d_idx)

    for bad in (-1, n_src):
        with pytest.raises(IndexError):
            run([0, 3, bad, 1, 2, 5, 6, 7, 8])
    empty = run([])
    assert empty.shape[0] == 0
    assert_same_values(run([n_src - 1, 0]).cpu().numpy()[:, :n_fields], base[[n_src - 1, 0], off : off + n_fields])


# ---- at_gather_cols ------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("n_out", [1, 31, 32, 33, 100])
def test_gather_cols(cuda, dev, dtype, n_out):
    rng = np.random.default_rng(n_out)
    n_rows, nx, ldx = 1003, 70, 74
    base = _specials(rng, (n_rows, ldx), dtype)
    cols = list(rng.integers(0, nx, n_out))
    cols[: min(n_out, 6)] = [nx - 1, 0, 0, 5, 4, 3][: min(n_out, 6)]  # repeated and reversed
    if n_out > 40:
        cols[-30:] = list(range(nx - 1, nx - 31, -1))
    X = _to_dev(cuda, base)[:, :nx]
    _poison(cuda, (n_rows, _round_up(n_out, 4)), X.dtype)
    got = dev.gather_cols(X, cols).cpu().numpy()
    assert got.shape == (n_rows, _round_up(n_out, 4)) and got.shape[1] != ldx
    assert_same_values(got[:, :n_out], base[:, cols], "gathered columns")
    assert np.array_equal(_bits(got[:, n_out:]), _bits(np.zeros((n_rows, got.shape[1] - n_out), dtype)))
    # an explicit out with its own (odd) leading dimension
    ob = cuda.full((n_rows, n_out + 3), -5.0, dtype=X.dtype, device="cuda")
    dev.gather_cols(X, cols[::-1], out=ob[:, :n_out])
    got = ob.cpu().numpy()
    assert_same_values(got[:, :n_out], base[:, cols[::-1]], "explicit out")
    assert (got[:, n_out:] == -5.0).all()


# ---- at_compare_mask -----------------------------------------------------------------------
OPS = [operator.eq, operator.ne, operator.gt, operator.ge, operator.lt, operator.le, None]  # op codes 0..6; 6 = not NaN
THRESHOLDS = [0.5, 0.1, 1e40, -1e40, 1e-50, float("nan"), 0.0, -0.0]


def _numpy_compare(values, op, threshold):
    with np.errstate(over="ignore"):
        return ~np.isnan(values) if OPS[op] is None else OPS[op](values, threshold)


def _compare_values(rng, dtype, n, threshold):
    """n values of `dtype`: the threshold as the dtype holds it, one float32 ulp either side,
    NaN, ±inf, ±0.0, and normal values."""
    with np.errstate(over="ignore"):
        t32 = np.float32(threshold)
    pool = np.array([t32, np.nextafter(t32, np.float32(np.inf)), np.nextafter(t32, np.float32(-np.inf)), np.nan, np.inf, -np.inf, 0.0, -0.0], np.float32).astype(dtype)
    if dtype == np.float64:
        pool = np.concatenate([pool, [threshold]])
    v = rng.normal(size=n).astype(dtype)
    pick = rng.random(n) < 0.5
    v[pick] = pool[rng.integers(0, pool.size, int(pick.sum()))]
    v[: min(n, pool.size)] = pool[: min(n, pool.size)]
    return v


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("layout", ["unit", "column"])
@pytest.mark.parametrize("n", [1, 255, 256, 257, 1_000_003])
def test_compare_mask(cuda, dev, dtype, layout, n):
    rng = np.random.default_rng(n)
    for threshold in THRESHOLDS:
        v = _compare_values(rng, dtype, n, threshold)
        if layout == "column":
            # the column view remove_nans passes: batch.data[:, j]
            m = rng.normal(size=(n, 8)).astype(dtype)
            m[:, 3] = v
            d = _to_dev(cuda, m)[:, 3]
        else:
            d = _to_dev(cuda, v)
        for op in range(7):
            got = dev.compare_mask(d, op, threshold).cpu().numpy()
            assert got.dtype == np.uint8 and set(np.unique(got)) <= {0, 1}
            assert np.array_equal(got.astype(bool), _numpy_compare(v, op, threshold)), (op, threshold)


def _other_dtype_values(dtype):
    if dtype == np.float16:
        h = np.float16(0.1)
        return np.array([h, np.nextafter(h, np.float16(1)), np.nextafter(h, np.float16(0)), 0.5, 65504, -65504, np.inf, -np.inf, np.nan, 0.0, -0.0, 6e-8, -6e-8, 1.0], np.float16)
    if dtype == np.bool_:
        return np.array([True, False, True, True, False])
    info = np.iinfo(dtype)
    vals = [info.min, info.max, 0, 1, -1, 2, 127, -128, 255, 2**53, 2**53 + 1, -(2**53) - 1]
    return np.array([x for x in vals if info.min <= x <= info.max], dtype)


OTHER_THRESHOLDS = [0.1, 0.5, 1.0, 0.0, -0.0, float("nan"), 1e40, 1e-50, 65519.0, 65520.0, 127.5, -128.0, 255.0, float(2**53)]


@pytest.mark.parametrize("dtype", [np.float16, np.int8, np.uint8, np.int64, np.bool_], ids=lambda d: np.dtype(d).name)
def test_compare_mask_other_dtypes(cuda, dev, dtype):
    """numpy compares a float16 array with a Python float in float16 and an integer or bool
    array in float64 (NEP 50).  float16 values widen exactly, so rounding the threshold to
    float16 first makes the device's float64 comparison equal numpy's."""
    v = _other_dtype_values(dtype)
    d = _to_dev(cuda, v)
    for threshold in OTHER_THRESHOLDS:
        for op in range(7):
            got = dev.compare_mask(d, op, threshold).cpu().numpy().astype(bool)
            assert np.array_equal(got, _numpy_compare(v, op, threshold)), (op, threshold, v, got)


@pytest.mark.parametrize("spelling", ["==", "!=", ">", ">=", "<", "<="])
def test_apply_mask_from_float16_npy(F, tmp_path, spelling):
    """A float16 land-sea mask file goes into the comparison as np.load returns it."""
    mask = np.tile(_other_dtype_values(np.float16), 3)
    np.save(tmp_path / "lsm.npy", mask)
    x = np.arange(mask.size, dtype=np.float32) + 1
    fl = ekd.from_source("list-of-dicts", [dict(param="t", values=x, latitudes=np.zeros(x.size), longitudes=np.arange(x.size, dtype=np.float64))])
    op = {"==": operator.eq, "!=": operator.ne, ">": operator.gt, ">=": operator.ge, "<": operator.lt, "<=": operator.le}[spelling]
    for threshold in (0.1, 0.5, 65519.0, 1e-50, -0.0):
        with np.errstate(over="ignore"):
            hit = op(mask, threshold)
        want = x.copy()
        want[hit] = np.nan
        out = F("apply_mask", path=str(tmp_path / "lsm.npy"), threshold=threshold, threshold_operator=spelling).forward(fl)
        assert_same_values(out[0].to_numpy(flatten=True), want, f"{spelling} {threshold}")
        if spelling == "==":
            out = F("apply_mask", path=str(tmp_path / "lsm.npy"), mask_value=threshold).forward(fl)
            assert_same_values(out[0].to_numpy(flatten=True), want, f"mask_value {threshold}")


# ---- at_sum_cols ---------------------------------------------------------------------------
def _numpy_sum(terms):
    """The filter's statement: `s = c0.copy(); s += c1; …` (inf + -inf is NaN, quietly)."""
    s = terms[0].copy()
    with np.errstate(invalid="ignore"):
        for t in terms[1:]:
            s += t
    return s


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("n_groups", [1, 32, 33, 200])
@pytest.mark.parametrize("n_terms", [1, 2, 5])
def test_sum_cols(cuda, dev, dtype, n_groups, n_terms):
    rng = np.random.default_rng(n_groups * 10 + n_terms)
    n_rows, nx, ldx = 1003, 64, 67
    base = _specials(rng, (n_rows, ldx), dtype)
    base[:, 0] = -0.0
    base[:, 1] = np.where(np.arange(n_rows) % 2 == 0, 0.0, -0.0)
    cols = rng.integers(0, nx, n_groups * n_terms)  # reused, not contiguous
    if n_groups > 2:
        cols[-n_terms:] = 0  # a group of −0.0 terms only
        cols[-2 * n_terms : -n_terms] = [0] + [1] * (n_terms - 1)
    X = _to_dev(cuda, base)[:, :nx]
    _poison(cuda, (n_rows, _round_up(n_groups, 4)), X.dtype)
    got = dev.sum_cols(X, [int(c) for c in cols], n_groups, n_terms).cpu().numpy()
    want = np.stack([_numpy_sum([base[:, c] for c in cols[g * n_terms : (g + 1) * n_terms]]) for g in range(n_groups)], axis=1)
    assert_same_values(got[:, :n_groups], want, "group sums")
    assert np.array_equal(_bits(got[:, n_groups:]), _bits(np.zeros((n_rows, got.shape[1] - n_groups), dtype)))


def _sum_fields(specs):
    """(param, levelist, date, values) → a FieldList whose mars namespace holds levelist and date."""
    return ekd.from_source(
        "list-of-dicts",
        [dict(param=p, levelist=lev, date=date, values=v, latitudes=np.zeros(v.size), longitudes=np.arange(v.size, dtype=np.float64)) for p, lev, date, v in specs],
        mars=True,
    )


def _check_sums(result, want):
    got = [f for f in result if f.metadata("param") == "tp"]
    assert len(got) == len(want)
    for f, w in zip(got, want):
        assert_same_values(f.to_numpy(flatten=True), w, f"tp {w.dtype}")


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_sum_filter_many_levels(F, dtype):
    rng = np.random.default_rng(11)
    n, levels = 777, list(range(40))
    data = {(p, lev): _specials(rng, n, dtype) for p in ("lsp", "cp", "sf") for lev in levels}
    specs = [(p, lev, 20200101, data[p, lev]) for lev in levels for p in ("lsp", "cp", "sf")]
    specs.insert(4, ("t", 0, 20200101, _specials(rng, n, dtype)))
    out = F("sum", params=["lsp", "cp", "sf"], output="tp").forward(_sum_fields(specs))
    assert [f.metadata("param") for f in out][0] == "t"
    assert [int(f.metadata("levelist")) for f in out][1:] == levels
    _check_sums(out, [_numpy_sum([data[p, lev] for p in ("lsp", "cp", "sf")]) for lev in levels])
    # ignore_level: the terms of one sum sit on different levels (lsp at 2k, cp at 2k+1) of one date
    specs = [("lsp" if lev % 2 == 0 else "cp", lev, 20200101 + lev // 2, data["lsp" if lev % 2 == 0 else "cp", lev]) for lev in levels]
    out = F("sum", params=["lsp", "cp"], output="tp", ignore_level=True).forward(_sum_fields(specs))
    _check_sums(out, [_numpy_sum([data["lsp", lev], data["cp", lev + 1]]) for lev in levels[::2]])


def test_sum_filter_mixed_dtypes(F):
    """numpy's `s = c0.copy(); s += c1; …` keeps c0's dtype and rounds after every step, so a
    group that mixes float32 and float64 terms is neither summed nor returned in float64."""
    rng = np.random.default_rng(12)
    n = 1001
    lsp, cp, sf = rng.random(n).astype(np.float32), rng.random(n) * 1e-3, rng.random(n).astype(np.float32)
    cp[:5] = [1e-9, 3e-8, np.nan, -0.0, 2.0**-30]
    lsp[5:8] = [np.inf, -0.0, 0.0]
    cases = [
        (lsp, cp, sf),  # float32 lsp, float64 cp, float32 sf
        (cp, lsp, sf),
        (lsp, sf, lsp),
        (cp, cp, cp),
        (sf, lsp, sf),
    ]
    specs = [(p, 0, 20200101 + k, t) for k, terms in enumerate(cases) for p, t in zip(("lsp", "cp", "sf"), terms)]
    out = F("sum", params=["lsp", "cp", "sf"], output="tp").forward(_sum_fields(specs))
    want = [_numpy_sum(list(terms)) for terms in cases]
    assert [w.dtype for w in want] == [np.float32, np.float64, np.float32, np.float64, np.float32]
    assert [int(f.metadata("date")) for f in out] == [20200101 + k for k in range(len(cases))]
    _check_sums(out, want)


# ---- at_range_flags ------------------------------------------------------------------------
LO, HI = -2 * np.pi, 2 * np.pi  # the cos_sin_from_rad range check


def _numpy_flags(col):
    return int((col < LO).any()) | 2 * int((col > HI).any()) | 4 * int(np.isnan(col).any())


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("n_cols", [1, 32, 33, 70])
def test_range_flags(cuda, dev, n_sms, dtype, n_cols):
    """One warp per row chunk over at most 8·8·SMs warps: outliers in the first and the last
    row and on either side of row 8·8·SMs, where the grid-stride loop wraps."""
    rng = np.random.default_rng(n_cols)
    n_rows = 1_000_003 if n_cols <= 33 else 300_007
    ldx = n_cols + 8
    hi, lo = dtype(HI), dtype(LO)  # the bounds as the comparison in `dtype` sees them
    up, down = np.nextafter(hi, dtype(np.inf)), np.nextafter(lo, dtype(-np.inf))
    x = rng.uniform(-6.0, 6.0, size=(n_rows, ldx)).astype(dtype)
    wrap = 8 * 8 * n_sms
    for c in range(ldx):
        x[0, c], x[-1, c] = hi, lo  # exactly at the bounds: not outside
        case = c % 8
        if case == 1:
            x[0, c] = up
        elif case == 2:
            x[-1, c] = down
        elif case == 3:
            x[wrap - 1, c] = up
        elif case == 4:
            x[wrap, c] = down
        elif case == 5:
            x[rng.integers(0, n_rows), c] = np.nan
            x[rng.integers(0, n_rows), c] = up
        elif case == 6:
            x[wrap + 1, c] = np.nan
        elif case == 7:
            x[wrap - 2, c], x[rng.integers(0, n_rows), c] = up, down
    want = [_numpy_flags(x[:, c]) for c in range(ldx)]
    assert sorted(set(want)) == [0, 1, 2, 3, 4, 6]
    X = _to_dev(cuda, x)
    for first_col in range(ldx - n_cols + 1):
        got = dev.range_flags(X, first_col, n_cols, LO, HI)
        assert got == want[first_col : first_col + n_cols], first_col


# ---- at_compact_mask -----------------------------------------------------------------------
PASS_BYTES = 4096 * 1024  # bytes one pass of the 1 024-thread block scan covers


def _mark(rng, n, pattern):
    if pattern == "zeros":
        return np.zeros(n, np.uint8)
    if pattern == "nonzero":
        return rng.integers(1, 256, n).astype(np.uint8)  # every byte non-zero, not only 1
    m = np.where(rng.random(n) < 0.3, rng.integers(1, 256, n), 0).astype(np.uint8)
    if pattern == "block":
        m[:] = 0
        if n >= 3 * 4096:
            m[2 * 4096 : 3 * 4096] = 1  # one 4 096-byte block entirely non-zero
    if n:
        m[-1] = 0x80
    return m


@pytest.mark.parametrize("n", [0, 1, PASS_BYTES - 1, PASS_BYTES, PASS_BYTES + 1, 5_000_011])
@pytest.mark.parametrize("pattern", ["random", "zeros", "nonzero", "block"])
def test_compact_mask(cuda, dev, n, pattern):
    rng = np.random.default_rng(n % 1000)
    m = _mark(rng, n, pattern)
    got = dev.compact_mask(_to_dev(cuda, m)).cpu().numpy()
    assert got.dtype == np.int64
    assert np.array_equal(got, np.flatnonzero(m))


@pytest.mark.parametrize("n", [100, 4096 + 17, PASS_BYTES + 1, 5_000_011])
def test_compact_mask_unaligned_views(cuda, dev, n):
    """Views starting 1 … 15 bytes into an aligned buffer take the scalar loads of load_chunk16."""
    rng = np.random.default_rng(n)
    buf = _mark(rng, n + 16, "random")
    d = _to_dev(cuda, buf)
    for off in range(16):
        view = d[off : off + n]
        assert view.data_ptr() % 16 == off % 16
        got = dev.compact_mask(view).cpu().numpy()
        assert np.array_equal(got, np.flatnonzero(buf[off : off + n])), off


# ---- at_cropping_mask ----------------------------------------------------------------------
BOXES = [
    (60.0, -20.0, 30.0, 40.0),  # given in [-180, 180)
    (60.0, 340.0, 30.0, 400.0),  # the same box in [0, 360), east past 360
    (10.0, 170.0, -10.0, 190.0),  # across the dateline, east past 180
    (10.0, -190.0, -10.0, -170.0),  # across the dateline, west before -180
    (89.5, 0.0, -89.5, 359.75),
    (45.25, 100.125, 45.25, 100.125),  # a single point
]


def _edge_points(north, west, south, east):
    lats = [north, south, np.nextafter(north, np.inf), np.nextafter(south, -np.inf), (north + south) / 2]
    edges = [west, east, west + 360, east + 360, west - 360, east - 360]
    lons = []
    for e in edges:
        lons += [e, np.nextafter(e, np.inf), np.nextafter(e, -np.inf)]
    lons += [(west + east) / 2, (west + east) / 2 + 360, (west + east) / 2 - 360, 0.0, -0.0, 180.0, -180.0, 359.999]
    la, lo = np.meshgrid(np.array(lats), np.array(lons), indexing="ij")
    return la.reshape(-1), lo.reshape(-1)


@pytest.mark.parametrize("box", BOXES, ids=lambda b: "_".join(f"{v:g}" for v in b))
@pytest.mark.parametrize("convention", ["as_given", "pm180", "0to360"])
def test_cropping_mask(cuda, dev, box, convention):
    from oracle import spatial as osp

    rng = np.random.default_rng(3)
    la, lo = _edge_points(*box)
    rlat, rlon = rng.uniform(-90, 90, 5000), rng.uniform(-180, 180, 5000)
    lats, lons = np.concatenate([la, rlat]), np.concatenate([lo, rlon])
    if convention == "0to360":
        lons = np.mod(lons, 360.0)
    elif convention == "pm180":
        lons = np.mod(lons + 180.0, 360.0) - 180.0
    got = dev.cropping_mask_device(lats, lons, *box).cpu().numpy()
    want = osp.cropping_mask(lats, lons, *box)
    assert got.dtype == np.uint8 and set(np.unique(got)) <= {0, 1}
    assert np.array_equal(got.astype(bool), want)
    assert want.any()
