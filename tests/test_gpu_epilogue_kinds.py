"""Every epilogue kind (csrc/epilogue.cuh) value by value, and the same bits from every kernel
and kind family that runs it.

a. Exact kinds — PLAIN with clip and mask, AFFINE, AFFINE_INV, IMPUTE_NAN and the pass-through
   columns of QT2QTR / RT2RTQ / RT2RTD / DT2DTR — bitwise against numpy in the field's dtype.
   The library is built with -fmad=false, without -ftz and with IEEE division, so these are
   single IEEE operations or copies: anything short of bit equality is a bug.
b. Library-math kinds — EXP, LOG, COSSIN, ATAN2 (with and without the 360° wrap) — against a
   higher-precision evaluation at the same (dtype-rounded) arguments, within the CUDA Math API's
   documented maximum ulp errors (CUDA C++ Programming Guide, "Mathematical Functions"):
   expf 2, logf 1, sincosf 2, atan2f 3; exp 1, log 1, sincos 2, atan2 2 — and, for float32
   atan2 inside its range, the polynomial's stated 3.2e-7 rad (epilogue.cuh:84-85).
c. The float32 humidity and dewpoint fast paths (QT2R, RT2Q, RT2D, DT2R) against
   oracle/pointwise.py evaluated in float64 at the float32 inputs, on every es-table interval and
   on both sides of every switch between the fast path and the formula; bounds built from the
   stated ones (es from the table: 2e-7 relative, epilogue.cuh:200-203) and from the float32
   operations each path runs.  NaN / inf positions exactly the oracle's, except inside the
   explicitly computed band where the rounding of e can flip r_to_q's `p - e < 1e-4` test.
d. The same kinds in float64 (no fast path) against a long-double evaluation of the oracle,
   with the same derivations at float64's unit roundoff, and the wind kinds.
e. For every kind: at_pointwise in the kind's own family and in FAM_ALL, at_gather_pointwise,
   and at_spmm_fused on each fused instantiation (uniform 4 and 12 entries, ragged rows, a row
   longer than kSegCap) give bitwise the same columns as at_spmm followed by at_pointwise.
"""

from __future__ import annotations

import numpy as np
import pytest

from oracle import es_table as et
from oracle import pointwise as pw

pytestmark = pytest.mark.gpu

U32, U64 = 2.0**-24, 2.0**-53  # unit roundoff: one rounding is <= u relative, one ulp <= 2u relative

F32 = np.float32


def _nb(x, dtype=F32):
    """x and its two neighbours in dtype."""
    x = dtype(x)
    return [np.nextafter(x, dtype(-np.inf)), x, np.nextafter(x, dtype(np.inf))]


def _run(kind, x, cols, pa=1.0, pb=0.0, row_mask=None):
    import torch

    from anemoi_transform_b200 import _cabi
    from anemoi_transform_b200.device import Epilogue

    epi = Epilogue([(getattr(_cabi, kind), 0, x.shape[1], 0, pa, pb)], cols)
    m = None if row_mask is None else torch.from_numpy(row_mask).cuda()
    X = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return epi.apply(X, out=_sentinel(x.shape[0], len(cols), X.dtype), row_mask=m).cpu().numpy()[:, : len(cols)]


def _sentinel(n_rows, n_cols, dtype):
    """An output buffer holding -7.0 everywhere: a launch that skips a column cannot pass by
    finding the previous result in memory the allocator handed back."""
    import torch

    return torch.full((n_rows, -(-n_cols // 4) * 4), -7.0, dtype=dtype, device="cuda")


def _no_cols(n, p=0.0):
    return [(0.0, 0.0, p, 0)] * n


def _pack(*cols, width):
    """Interleave 1-D inputs into rows of `width` groups (zero padding at the end)."""
    n = cols[0].size
    rows = -(-n // width)
    out = np.zeros((rows * width, len(cols)), dtype=cols[0].dtype)
    for i, c in enumerate(cols):
        out[:n, i] = c
        out[n:, i] = c[-1]
    return out.reshape(rows, width * len(cols)), n


def _bits_equal(got, want):
    assert got.shape == want.shape and got.dtype == want.dtype
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w), f"NaN positions differ at {np.argwhere(nan_g != nan_w)[:5]}"
    view = {4: np.uint32, 8: np.uint64}[got.dtype.itemsize]
    bad = np.argwhere(got.view(view) != want.view(view))
    bad = [tuple(b) for b in bad if not nan_g[tuple(b)]]
    assert not bad, f"{len(bad)} values differ, first {bad[:3]}: {[(got[b], want[b]) for b in bad[:3]]}"


SPECIALS = {
    F32: [0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1.1754942e-38, 1.1754944e-38, -1.1754944e-38,
          3.4028235e38, -3.4028235e38, 1.0, -1.0, 0.1, 459.67, -459.67, 2e38, 1e-40, 6.5e-44],
    np.float64: [0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, -5e-324, 2.2250738585072014e-308, 2.225073858507201e-308,
                 1.7976931348623157e308, -1.7976931348623157e308, 1.0, -1.0, 0.1, 459.67, -459.67, 1e308, 1e-310],
}


def _special_field(dtype, n_rows, n_cols, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((n_rows, n_cols)) * 300).astype(dtype)
    sp = np.array(SPECIALS[dtype], dtype=dtype)
    flat = x.reshape(-1)
    flat[: sp.size * 3] = np.tile(sp, 3)
    idx = rng.integers(sp.size * 3, flat.size, flat.size // 7)
    flat[idx] = rng.choice(sp, idx.size)
    return x


# ---- a. exact kinds ------------------------------------------------------------------------------


@pytest.mark.parametrize("dtype", [F32, np.float64])
def test_exact_kinds_are_bitwise_numpy(cuda, dtype):
    from anemoi_transform_b200 import _cabi

    T = dtype
    x = _special_field(T, 64, 32, seed=1)
    CL, CH, MK = _cabi.COL_CLIP_LO, _cabi.COL_CLIP_HI, _cabi.COL_MASK
    with np.errstate(all="ignore"):
        # PLAIN: x < lo ? lo : x, then x > hi ? hi : x (NaN passes), then NaN on masked rows' mask columns
        cols, lo, hi, mk = [], np.full(32, -np.inf, T), np.full(32, np.inf, T), np.zeros(32, bool)
        for c in range(32):
            f = (CL if c % 4 in (0, 1) else 0) | (CH if c % 4 in (0, 2) else 0) | (MK if c % 3 == 0 else 0)
            cols.append((-1.5, 300.25, 0.0, f))
            lo[c] = T(-1.5) if f & CL else lo[c]
            hi[c] = T(300.25) if f & CH else hi[c]
            mk[c] = bool(f & MK)
        rmask = (np.arange(64) % 5 == 1).astype(np.uint8)
        want = np.where(x < lo, lo, x)
        want = np.where(want > hi, hi, want)
        want[np.ix_(rmask != 0, mk)] = np.nan
        _bits_equal(_run("EPI_PLAIN", x, cols, row_mask=rmask), want)

        # AFFINE x*pa + pb (mul, then add: never fused) and AFFINE_INV (x - pb) / pa, constants
        # rounded to T like numpy rounds a Python float against a T array (NEP 50); 3e38 * 3 and
        # 1e308 * 3 overflow
        for pa, pb in [(1.8, -459.67), (9.80665, 0.0), (3.0, 1e-45), (-0.5, 2.5), (1e-30, -0.0)]:
            _bits_equal(_run("EPI_AFFINE", x, _no_cols(32), pa, pb), x * T(pa) + T(pb))
            _bits_equal(_run("EPI_AFFINE_INV", x, _no_cols(32), pa, pb), (x - T(pb)) / T(pa))
        for v in (-1.5, 0.0, -0.0, 1e-45, np.inf):
            _bits_equal(_run("EPI_IMPUTE_NAN", x, _no_cols(32), v), np.where(np.isnan(x), T(v), x))

    # the pass-through columns of the (a, b) -> (a, b, f(a, b)) kinds are copies, specials included
    for kind in ("EPI_QT2QTR", "EPI_RT2RTQ", "EPI_RT2RTD", "EPI_DT2DTR"):
        got = _run(kind, x, _no_cols(48, 85000.0))
        _bits_equal(got[:, 0::3], x[:, 0::2])
        _bits_equal(got[:, 1::3], x[:, 1::2])


# ---- b. library-math kinds -----------------------------------------------------------------------

# CUDA Math API maximum errors in ulps (float32, float64)
ULPS = {"exp": (2, 1), "log": (1, 1), "sincos": (2, 2), "atan2": (3, 2)}


def _hi(T):
    """The evaluation type of the reference: float64 for float32 fields, long double for float64."""
    return np.float64 if T == F32 else np.longdouble


def _ulp(y, T):
    """One ulp of T at the (high-precision) value y; past the largest finite T, the ulp there."""
    a = np.minimum(np.abs(y), np.finfo(T).max).astype(T)
    return np.spacing(a).astype(_hi(T))


def _as_hi(got, T):
    """Kernel results in the reference's type, +-inf standing for the first value past T's range
    (so that a result that rounds to inf is compared like any other)."""
    g = got.astype(_hi(T))
    big = _hi(T)(2) ** (128 if T == F32 else 1024)
    return np.where(np.isinf(g), np.sign(g) * big, g)


def _check_ulps(got, want, T, n_ulp, what):
    """|got - want| <= n_ulp ulps of want, NaN in the same places; want past T's range counts as
    that first value past it."""
    assert np.array_equal(np.isnan(got), np.isnan(want)), (what, "NaN positions differ")
    ok = ~np.isnan(want)
    big = _hi(T)(2) ** (128 if T == F32 else 1024)
    w = np.clip(want[ok], -big, big)
    g = _as_hi(got[ok], T)
    err = np.abs(g - w)
    lim = n_ulp * _ulp(w, T)
    i = np.argmax(err / np.maximum(lim, np.finfo(_hi(T)).tiny))
    assert np.all(err <= lim), f"{what}: {np.sum(err > lim)} values beyond {n_ulp} ulp, worst got {g[i]!r} want {w[i]!r}"


@pytest.mark.parametrize("dtype", [F32, np.float64])
def test_exp_and_log_within_the_documented_ulps(cuda, dtype):
    """expf / exp: 2 / 1 ulp, logf / log: 1 / 1 ulp (CUDA Math API), over the overflow and
    underflow thresholds, zeros, negatives, infinities and subnormals."""
    T, H = dtype, _hi(dtype)
    fi = np.finfo(T)
    rng = np.random.default_rng(2)
    if T == F32:
        edges = [88.72283, 88.7, 88.8, -87.33655, -103.27893, -103.97208, -104.0, -88.0, 0.0, -0.0, 1e-7, -1e-7]
    else:
        edges = [709.782712893384, 709.78, 709.79, -708.3964185322641, -744.4400719213812, -745.1332191019412, -746.0, 0.0, -0.0, 1e-16]
    xe = np.concatenate([np.array([v for e in edges for v in _nb(e, T)], T), np.array(SPECIALS[T], T),
                         (rng.standard_normal(4000) * (30 if T == F32 else 250)).astype(T)])
    xe, n = _pack(xe, width=32)
    with np.errstate(all="ignore"):
        _check_ulps(_run("EPI_EXP", xe, _no_cols(32)).ravel()[:n], np.exp(xe.astype(H)).ravel()[:n], T, ULPS["exp"][T != F32], "exp")
        xl = np.concatenate([np.array([0.0, -0.0, -1.0, -fi.tiny, -np.inf, np.inf, np.nan, fi.smallest_subnormal, fi.tiny, fi.max, 1.0], T),
                             np.array([v for e in (1.0, 0.5, 2.0, fi.tiny) for v in _nb(e, T)], T),
                             (fi.smallest_subnormal * rng.integers(1, 2**20, 500)).astype(T),
                             np.exp(rng.uniform(-80, 80, 4000)).astype(T)])
        xl, n = _pack(xl, width=32)
        _check_ulps(_run("EPI_LOG", xl, _no_cols(32)).ravel()[:n], np.log(xl.astype(H)).ravel()[:n], T, ULPS["log"][T != F32], "log")


@pytest.mark.parametrize("dtype", [F32, np.float64])
@pytest.mark.parametrize("pa", [1.0, float(np.deg2rad(1.0))])
def test_cossin_within_the_documented_ulps(cuda, dtype, pa):
    """cos / sin of the T-rounded argument x*pa: sincosf / sincos 2 ulp each (CUDA Math API),
    up to arguments where the argument reduction takes its slow (Payne-Hanek) path."""
    T, H = dtype, _hi(dtype)
    rng = np.random.default_rng(3)
    x = np.concatenate([np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-30, -1e-45 if T == F32 else -5e-324], T),
                        (rng.standard_normal(3000) * 400).astype(T),
                        (10.0 ** rng.uniform(4, 38, 1000) * rng.choice([-1, 1], 1000)).astype(T),
                        np.array([105615.0, 105616.0, 1e5, 3.4e38 if T == F32 else 1.7e308], T)])
    x, n = _pack(x, width=16)
    got = _run("EPI_COSSIN", x, _no_cols(32), pa)
    with np.errstate(all="ignore"):
        arg = (x * T(pa)).astype(H)  # the kernel's argument: one rounding to T, exactly numpy's
        _check_ulps(got[:, 0::2].ravel()[:n], np.cos(arg).ravel()[:n], T, ULPS["sincos"][T != F32], "cos")
        _check_ulps(got[:, 1::2].ravel()[:n], np.sin(arg).ravel()[:n], T, ULPS["sincos"][T != F32], "sin")


@pytest.mark.parametrize("dtype", [F32, np.float64])
@pytest.mark.parametrize("wrap", [False, True])
def test_atan2_scaled_and_wrapped(cuda, dtype, wrap):
    """d = atan2(s, c) * pa, then (wrap) d >= 360 -> d - 360, d < 0 -> d + 360
    (cos_sin_mean_wave_direction.py:97-98).

    Bound, in the output's unit: the angle is off by E = max(3 ulp [atan2f] or 2 ulp [atan2],
    3.2e-7 rad [float32 polynomial, epilogue.cuh:84-85]) of the true angle; the product with the
    T-rounded pa scales that by |pa| and rounds once (0.5 ulp of d); the wrap's addition rounds
    once more (0.5 ulp of 360, d - 360 is exact by Sterbenz).  Wrapped results are compared
    modulo 360.  Signed zeros, 360 and -0.0 are checked exactly."""
    T, H = dtype, _hi(dtype)
    pa = float(np.rad2deg(1.0)) if wrap else 1.0
    rng = np.random.default_rng(4)
    sp = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 1e-45 if T == F32 else 5e-324, 1e30, -1e-30], T)
    c = np.concatenate([np.repeat(sp, sp.size), rng.standard_normal(5000).astype(T) * T(5), np.ones(64, T)])
    s = np.concatenate([np.tile(sp, sp.size), rng.standard_normal(5000).astype(T) * T(5), -np.geomspace(1e-12, 1e-7, 64).astype(T)])
    x, n = _pack(c, s, width=8)
    got = _run("EPI_ATAN2", x, _no_cols(8), pa, 1.0 if wrap else 0.0).ravel()[:n]
    ang = np.arctan2(s.astype(H), c.astype(H))
    pa_t = H(T(pa))
    want = ang * pa_t
    if wrap:
        want = np.where(want < 0, want + 360, want)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    g, w = got[ok].astype(H), want[ok]
    err = np.abs(g - w)
    if wrap:
        err = np.minimum(err, 360 - err)
    e_atan = ULPS["atan2"][T != F32] * _ulp(ang[ok], T)
    if T == F32:
        e_atan = np.maximum(e_atan, 3.2e-7)
    lim = abs(pa_t) * e_atan + 0.5 * _ulp(w, T) + (0.5 * float(np.spacing(T(360))) if wrap else 0)
    assert np.all(err <= lim), (np.max(err), np.sum(err > lim))
    # signed zeros exactly: atan2(+-0, x > 0) = +-0 (stays -0.0 under the wrap: -0.0 < 0 is false),
    # atan2(+-0, x < 0) = +-pi rounded to T, times pa_T
    zc = np.isin(c, [T(1.0), T(1e30)]) & (s == 0)
    assert np.array_equal(np.signbit(got[zc]), np.signbit(s[zc])) and np.all(got[zc] == 0)
    nc = (c == T(-1.0)) & (s == 0)
    pi_t = np.where(np.signbit(s[nc]), -T(np.pi), T(np.pi)) * T(pa)
    if wrap:
        pi_t = np.where(pi_t < 0, pi_t + T(360), pi_t)
    assert np.array_equal(got[nc], pi_t)
    if wrap:  # a direction a hair below 0 wraps to exactly 360, as in the reference
        tiny = got[c.size - 64 :]  # -5.7e-6 deg or closer to 0: below half an ulp of 360 in float32
        assert np.all(tiny == T(360)) if T == F32 else np.all(tiny < 360)


# ---- c / d. humidity and dewpoint ----------------------------------------------------------------

ES_TABLE = 2e-7  # es from the table vs the float64 formula, Horner included (epilogue.cuh:200-203)
T0_ERR = {F32: abs(float(F32(273.16)) - 273.16), np.float64: 0.0}  # the constant 273.16 as T


def _x_err(t, u, T, a, b):
    """Error of a Tetens exponent x = a (t - 273.16) / (t - b) evaluated in T: six roundings
    (t - t0, the constant a, a*(), t - b, the constant b, the division; each <= u relative, the
    last via div_normal or IEEE) plus 273.16 rounded to T, amplified by a / |t - b|."""
    x = a * (t - 273.16) / (t - b)
    return 7 * u * np.abs(x) + a * T0_ERR[T] / np.abs(t - b), x


def _es_rel(t, u, T, table):
    """Relative error of es(t): the table's 2e-7 where it is read, else the formula: the exponent's
    error (absolute in x is relative in exp(x)), exp's 2 / 1 ulp, *611.21 (2 roundings) and the
    mixed-phase blend (alpha: 3 roundings, the convex combination: 3)."""
    ew, _ = _x_err(t, u, T, 17.502, 32.19)
    ei, _ = _x_err(t, u, T, 22.587, -0.7)
    n_exp = 2 * (2 if T == F32 else 1)  # ulps of expf / exp, as multiples of u
    formula = np.maximum(ew, ei) + (n_exp + 2 + 6) * u
    return np.where(table, ES_TABLE, formula)


P_COLS = np.array([_nb(1.0)[0], 1.0, _nb(1.0)[2], 100.0, 5e4, 1e5, _nb(1e7)[0], 1e7], F32)  # both sides of 1 and 1e7 Pa


def _t_sweep():
    """Every table interval (4 Chebyshev points, ends, midpoint), the float32 neighbours of the
    table ends and both thresholds, and temperatures outside the table."""
    return np.concatenate([et.table_sample_points(), np.array([100.0, 150.0, 360.0, 400.0], F32)])


def _combos(first_typ, first_edges, t):
    """(first, t): the whole t sweep with typical values, a coarse sweep with the edge values."""
    tc = np.unique(np.concatenate([t[::8], np.array([v for e in (150.16, 250.16, 273.16, 350.15) for v in _nb(e)], F32)]))
    a = np.concatenate([np.repeat(np.array(first_typ, F32), t.size), np.repeat(np.array(first_edges, F32), tc.size)])
    b = np.concatenate([np.tile(t, len(first_typ)), np.tile(tc, len(first_edges))])
    return a, b


def _pressure_run(kind, a, b, T, pressures=P_COLS, a_per_col=None):
    """Rows of (a, t) pairs, pair j against pressures[j] (in the output column the kernel reads
    it from: the pair's own for 2-output kinds, its third for 6-output kinds); returns the
    outputs and the inputs."""
    n = a.size
    k = pressures.size
    x = np.empty((n, 2 * k), T)
    x[:, 0::2] = a[:, None] if a_per_col is None else a_per_col
    x[:, 1::2] = b[:, None]
    per = 3 if kind in ("EPI_QT2QTR", "EPI_RT2RTQ", "EPI_RT2RTD", "EPI_DT2DTR") else 1
    got = _run(kind, x, [(0.0, 0.0, float(p) if i == per - 1 else 0.0, 0) for p in pressures for i in range(per)])
    return got, x


def _fast_window(t, p, lo, hi, v, T):
    return (et.covers(t) & (v > lo) & (v < hi) & (p > 1.0) & (p < 1e7)) if T == F32 else np.zeros(np.broadcast(t, p, v).shape, bool)


def _check_rel(got, want, lim, what):
    assert np.array_equal(np.isnan(got), np.isnan(want)), (what, "NaN positions differ", np.argwhere(np.isnan(got) != np.isnan(want))[:5])
    assert np.array_equal(np.isinf(got), np.isinf(want)), (what, "inf positions differ")
    ok = np.isfinite(want)
    err = np.abs(got[ok].astype(np.float64) - want[ok])
    scale = lim[ok] * np.abs(want[ok])
    worst = np.argmax(err / np.maximum(scale, 1e-300))
    assert np.all(err <= scale), f"{what}: {np.sum(err > scale)} beyond the bound, worst rel {err[worst] / max(abs(want[ok][worst]), 1e-300):.3g} > {lim[ok][worst]:.3g}"
    print(f"{what}: max rel error {np.max(err / np.maximum(np.abs(want[ok]), 1e-300)):.3g}, max error/bound {np.max(err / np.maximum(scale, 1e-300)):.3g}")


@pytest.mark.parametrize("dtype", [F32, np.float64])
def test_q_to_r_fast_path_and_formula(cuda, dtype):
    """r = 100 p q / ((eps + c q) es(t)).  Relative bound: es's (2e-7 from the table, else the
    formula's, _es_rel) + 100*p, *q, *es and the division (div_normal or IEEE, <= 1 ulp = 2u):
    5 roundings, + eps + c*q (the constants eps and c, the product, the sum: 4 roundings)
    amplified by k = (eps + c|q|) / |eps + c q| (q down to -1 cancels)."""
    T, u = dtype, (U32 if dtype == F32 else U64)
    q, t = _combos([1e-3, 1.5e-2], [*_nb(-1.0), -0.5, 0.0, 1e-6, *_nb(1e3)], _t_sweep())
    got, x = _pressure_run("EPI_QT2R", q.astype(T), t.astype(T), T)
    H = _hi(T)
    q64, t64, p64 = q.astype(H)[:, None], t.astype(H)[:, None], P_COLS.astype(H)[None, :]
    with np.errstate(all="ignore"):
        want = pw.relative_humidity_from_specific_humidity(t64, q64, p64)
    eps, c = pw.epsilon, pw.epsilon * (1.0 / pw.epsilon - 1.0)
    k = (eps + c * np.abs(q64)) / np.abs(eps + c * q64)
    fast = _fast_window(t64, p64, -1.0, 1e3, q64, T)
    lim = _es_rel(t64, u, T, fast) + (5 * 2 + 4 * k) * u
    _check_rel(got, want, lim, f"qt2r {np.dtype(T).name}")
    if T == F32:
        assert fast.sum() > 0.3 * fast.size and (~fast).sum() > 0.2 * fast.size  # both paths ran


def test_float32_q_to_r_fast_path_is_bitwise_the_restated_table(cuda):
    """Inside the window the float32 q_to_r is IEEE float32 arithmetic around es_from_table:
    (100 p) q / ((eps + c q) es), div_normal giving the IEEE quotient (epilogue.cuh:172-177).
    With oracle/es_table.py (the host's fit, call for call, and the three FMAs rounded once)
    that is numpy's float32 evaluation bit for bit, at every interval's sample points and the
    thresholds' neighbours.  A table that is off by an ulp in some intervals — a wrong node
    origin, a coefficient off — can stay inside the 2e-7 bound; it fails here."""
    t = et.table_sample_points()
    t = t[et.covers(t)]
    q = np.repeat(np.array([1e-3, 1.5e-2, 0.3], F32), t.size)
    tt = np.tile(t, 3)
    p = np.array([100.0, 5e4, 1e5, _nb(1e7)[0]], F32)
    got, _ = _pressure_run("EPI_QT2R", q, tt, F32, p)
    es = et.es_from_table(tt)[:, None]
    num = (F32(100.0) * p[None, :]) * q[:, None]
    den = (F32(pw.epsilon) + F32(pw.epsilon * (1.0 / pw.epsilon - 1.0)) * q[:, None]) * es
    _bits_equal(got, num / den)


@pytest.mark.parametrize("dtype", [F32, np.float64])
def test_r_to_q_fast_path_formula_and_saturation(cuda, dtype):
    """q = eps e / (p + (eps - 1) e), e = r es(t) / 100, NaN where p - e < 1e-4.

    e: es's error + 2 roundings (r*es, /100 or *0.01f) + 0.01f's own (< u): rel_e = es + 3u.
    v = p - 0.378 e: rel_v <= g (rel_e + 2u) + u with g = 0.378|e| / |v| (< 1 wherever q is not
    NaN).  q: (1 + g) rel_e + 2g u + eps, eps*e, v and the division (<= 1 ulp): 5u more.

    NaN decision: the kernel compares its e, which is within rel_e |e| of the oracle's; where
    |p - e - 1e-4| <= rel_e |e| + u |p - e| + 3e-12 (1e-4f vs 1e-4) the comparison may flip.
    Inside the fast window a failed test falls back to the formula, so that band uses the
    formula's rel_e.  Outside the band NaN positions must be the oracle's exactly."""
    T, u = dtype, (U32 if dtype == F32 else U64)
    r, t = _combos([50.0, 95.0], [*_nb(-1e3), -50.0, 0.0, 1e-3, *_nb(1e3)], _t_sweep())
    # near saturation: per column r such that e = p - 1e-4 (+- a few 1e-7 relative)
    ts = np.array([255.0, 270.0, 273.16, 280.0, 290.0, 300.0, 320.0, 349.0], F32)
    ps = np.array([1000.0, 2000.0, 5000.0, 2e4, 4e4, 6e4, 8.5e4, 1e5], F32)
    kk = np.arange(-400, 401, 2) * 1e-7
    ts_rows = np.repeat(ts, kk.size)
    es_o = pw.saturation_vapour_pressure(ts_rows.astype(np.float64))
    r_sat = (100.0 * (ps.astype(np.float64)[None, :] - 1e-4) / es_o[:, None] * (1 + np.tile(kk, ts.size)[:, None])).astype(F32)
    for rr, tt, a_per_col in ((r, t, None), (np.zeros(ts_rows.size, F32), ts_rows, r_sat)):
        pcols = P_COLS if a_per_col is None else ps
        got, x = _pressure_run("EPI_RT2Q", rr.astype(T), tt.astype(T), T, pcols, None if a_per_col is None else a_per_col.astype(T))
        H = _hi(T)
        r64, t64, p64 = x[:, 0::2].astype(H), x[:, 1::2].astype(H), pcols.astype(H)[None, :]
        with np.errstate(all="ignore"):
            want = pw.specific_humidity_from_relative_humidity(t64, r64, p64)
            e = r64 * pw.saturation_vapour_pressure(t64) / 100.0
        fast = _fast_window(t64, p64, -1e3, 1e3, r64, T)
        rel_e_formula = _es_rel(t64, u, T, np.zeros_like(fast)) + 3 * u
        band = np.abs(p64 - e - 1e-4) <= rel_e_formula * np.abs(e) + u * np.abs(p64 - e) + 3e-12
        rel_e = np.where(fast & ~band, ES_TABLE, rel_e_formula - 3 * u) + 3 * u
        with np.errstate(all="ignore"):
            g = 0.378 * np.abs(e) / np.abs(p64 + (pw.epsilon - 1.0) * e)
        lim = (1 + g) * rel_e + 2 * g * u + 5 * 2 * u
        out = ~band
        assert np.array_equal(np.isnan(got[out]), np.isnan(want[out])), "NaN decision outside the rounding band"
        if a_per_col is not None:  # the sweep straddles the decision and the band is a sliver of it
            assert band.sum() < 0.2 * band.size and np.isnan(want).any() and (~np.isnan(want)).any()
            assert band.sum() > 0 or T != F32
        both = ~np.isnan(got) & ~np.isnan(want)
        _check_rel(np.where(both, got, np.nan), np.where(both, want, np.nan), lim, f"rt2q {np.dtype(T).name}")


def _td_bound(r, t, T, fast):
    """Absolute bound on td = (32.19 v - 4780.84632) / (v - 17.502) in kelvin.

    v on the fast path: lg2.approx(r*0.01f) * ln2 + xw(t): lg2.approx's error (absolute 2^-22 for
    arguments in (0.5, 2), relative 2^-22 elsewhere, epilogue.cuh:327-328) times ln 2, r*0.01f
    (2 roundings, 0.01f's own) and *ln2 (u |ln m| each), xw (_x_err), the sum (u |v|).  On the
    formula path: log(r es_w(t) / 100 / 611.21): es_w's error + 3 roundings, logf's 1 ulp of v.
    td then moves by |d td / d v| = 4217.36 / (v - 17.502)^2 per unit of v, and the last formula
    adds the constants 32.19f, 4780.846f (0.5 ulp of 4780) and 17.502f, the product, the two
    subtractions (u each of their results) and the division (1 ulp of td)."""
    u = U32 if T == F32 else U64
    with np.errstate(all="ignore"):
        m = r * 0.01
        ew, xw = _x_err(t, u, T, 17.502, 32.19)
        v = np.log(m) + xw
        lg2 = np.log(2) * 2.0**-22 * np.maximum(1.0, np.abs(np.log2(m)))
        dv_fast = lg2 + 3 * u * np.abs(np.log(m)) + ew + u * np.abs(v)
        dv_formula = ew + (2 * (2 if T == F32 else 1) + 2 + 3) * u + 2 * u * np.abs(v) + 2 * u * np.abs(np.log(m))
        dv = np.where(fast, dv_fast, dv_formula)
        den = v - 17.502
        num = 32.19 * v - 4780.84632
        td = num / den
        c_4780 = abs(float(T(4780.84632)) - 4780.84632) if T == F32 else 0.0
        c_17 = abs(float(T(17.502)) - 17.502) if T == F32 else 0.0
        d_num = 2 * u * np.abs(32.19 * v) + u * np.abs(num) + c_4780
        d_den = u * np.abs(den) + c_17
        return 4217.36 / den**2 * dv + d_num / np.abs(den) + np.abs(td) * d_den / np.abs(den) + 2 * u * np.abs(td)


@pytest.mark.parametrize("dtype", [F32, np.float64])
def test_dewpoint_from_r_fast_path_and_formula(cuda, dtype):
    """td from (r, t), r == 0 replaced by 1e-4 first (dewpoint.py:62-64, rt_to_d), against the
    oracle with the same replacement; absolute bound _td_bound per value."""
    T = dtype
    r, t = _combos([50.0, 99.0], [-1.0, -0.0, 0.0, 1e-4, 1e-3, 0.7, 1.0, *_nb(100.0), *_nb(1e4)], _t_sweep())
    x, n = _pack(r.astype(T), t.astype(T), width=16)
    got = _run("EPI_RT2D", x, _no_cols(16)).ravel()[:n]
    r_o = np.where(r == 0, _hi(T)(T(1e-4)), r.astype(_hi(T)))  # the filter's replacement, 1e-4 in the field's dtype
    t64 = t.astype(_hi(T))
    with np.errstate(all="ignore"):
        want = pw.dewpoint_from_relative_humidity(t64, r_o)
    fast = et.covers(t) & (r_o > 0) & (r_o < 1e4) if T == F32 else np.zeros(n, bool)
    lim = _td_bound(r_o, t64, T, fast)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(np.isinf(got), np.isinf(want))
    ok = np.isfinite(want)
    err = np.abs(got[ok].astype(np.float64) - want[ok])
    assert np.all(err <= lim[ok]), (np.sum(err > lim[ok]), float(np.max(err - lim[ok])))
    phys = (fast & (r_o >= 1) & (r_o <= 100) & (t >= 200) & (t <= 320))[ok]
    print(f"rt2d {np.dtype(T).name}: max |td error| {err.max():.3g} K (fast path {err[fast[ok]].max() if fast.any() else 0:.3g} K, "
          f"1-100 %, 200-320 K: {err[phys].max() if phys.any() else 0:.3g} K), max error/bound {np.max(err / lim[ok]):.3g}")
    assert np.all(np.isfinite(got[(r == 0) & np.isfinite(want)]))  # r == 0 is not log(0)


@pytest.mark.parametrize("dtype", [F32, np.float64])
def test_r_from_dewpoint_fast_path_and_formula(cuda, dtype):
    """r = 100 es_w(td) / es_w(t) (fast: 100 expf(xw(td) - xw(t))).  Relative bound: both
    exponents' errors (_x_err), the difference (u of it), exp's 2 / 1 ulp, *100, and on the
    formula path the two es_w (611.21: 2 roundings each) and the division: 16u in all."""
    T, u = dtype, (U32 if dtype == F32 else U64)
    tt = _t_sweep()
    few = np.array([*_nb(150.16), 200.0, 273.16, 300.0, *_nb(350.15), 360.0], F32)
    td = np.concatenate([np.repeat(tt, few.size), np.tile(few, tt.size)])
    t = np.concatenate([np.tile(few, tt.size), np.repeat(tt, few.size)])
    x, n = _pack(td.astype(T), t.astype(T), width=16)
    got = _run("EPI_DT2R", x, _no_cols(16)).ravel()[:n]
    td64, t64 = td.astype(_hi(T)), t.astype(_hi(T))
    with np.errstate(all="ignore"):
        want = pw.relative_humidity_from_dewpoint(t64, td64)
    e1, x1 = _x_err(td64, u, T, 17.502, 32.19)
    e2, x2 = _x_err(t64, u, T, 17.502, 32.19)
    lim = e1 + e2 + u * np.abs(x1 - x2) + 16 * u
    _check_rel(got, want, lim, f"dt2r {np.dtype(T).name}")


@pytest.mark.parametrize("kind", ["EPI_QT2R", "EPI_RT2Q", "EPI_RT2D", "EPI_DT2R", "EPI_QT2QTR", "EPI_RT2RTQ", "EPI_RT2RTD", "EPI_DT2DTR"])
def test_nan_and_inf_in_every_input_slot(cuda, kind):
    """NaN and +-inf in each input (and the pressure) give NaN / +-inf exactly where the
    float64 oracle does."""
    sp = np.array([np.nan, np.inf, -np.inf], F32)
    base = {"EPI_QT2R": (1e-3, 280.0), "EPI_RT2Q": (50.0, 280.0), "EPI_RT2D": (50.0, 280.0), "EPI_DT2R": (270.0, 280.0)}
    name = {"EPI_QT2QTR": "EPI_QT2R", "EPI_RT2RTQ": "EPI_RT2Q", "EPI_RT2RTD": "EPI_RT2D", "EPI_DT2DTR": "EPI_DT2R"}.get(kind, kind)
    a0, b0 = base[name]
    rows = [(s, b0) for s in sp] + [(a0, s) for s in sp] + [(s1, s2) for s1 in sp for s2 in sp] + [(a0, b0)]
    a = np.array([r[0] for r in rows], F32)
    b = np.array([r[1] for r in rows], F32)
    pcols = np.array([85000.0, np.nan, np.inf, -np.inf], F32)
    with np.errstate(all="ignore"):
        got, x = _pressure_run(kind, a, b, F32, pcols)
        a64, b64, p64 = x[:, 0::2].astype(np.float64), x[:, 1::2].astype(np.float64), pcols.astype(np.float64)[None, :]
        if name == "EPI_QT2R":
            want = pw.relative_humidity_from_specific_humidity(b64, a64, p64)
        elif name == "EPI_RT2Q":
            want = pw.specific_humidity_from_relative_humidity(b64, a64, p64)
        elif name == "EPI_RT2D":  # no pressure
            want = np.broadcast_to(pw.dewpoint_from_relative_humidity(b64[:, :1], a64[:, :1]), a64.shape)
        else:
            want = np.broadcast_to(pw.relative_humidity_from_dewpoint(b64[:, :1], a64[:, :1]), a64.shape)
    if kind != name:
        got = got[:, 2::3]
    assert np.array_equal(np.isnan(got), np.isnan(want)), np.argwhere(np.isnan(got) != np.isnan(want))[:5]
    assert np.array_equal(np.isposinf(got), np.isposinf(want)) and np.array_equal(np.isneginf(got), np.isneginf(want))


@pytest.mark.parametrize("kind", ["EPI_UV2DDFF", "EPI_DDFF2UV"])
def test_wind_kinds_in_float64(cuda, kind):
    """pointwise_kernel<double> against a long-double oracle.  UV2DDFF: speed hypot (2 ulp); direction (c - d) * deg with d = atan2 (2 ulp of d), c in
    {-pi/2, 3pi/2} as a double (u |c|), the subtraction (u |c - d|), deg as a double and the
    product (2u of the result).  DDFF2UV: a = (270 - wdir) * rad is off by u |270 - wdir| rad +
    2u |a|; u = ws cos(a) by 2 ulp (sincos) + |sin a| da + u, likewise v."""
    T, H, u = np.float64, np.longdouble, U64
    rng = np.random.default_rng(7)
    a = rng.standard_normal(20000) * 8
    b = rng.standard_normal(20000) * 8
    if kind == "EPI_DDFF2UV":
        a, b = np.abs(a) * 3, (b * 100) % 360
    x, n = _pack(a, b, width=16)
    got = _run(kind, x, _no_cols(32))
    g0, g1 = got[:, 0::2].ravel()[:n].astype(H), got[:, 1::2].ravel()[:n].astype(H)
    aH, bH = a.astype(H), b.astype(H)
    if kind == "EPI_UV2DDFF":
        ws, wd = pw.xy_to_polar(aH, bH)
        d = np.arctan2(bH, aH)
        c = np.where(d <= -np.pi / 2, np.pi / 2, 3 * np.pi / 2)
        lim_wd = pw.degree * (2 * _ulp(d, T) + u * c + u * np.abs(c - d)) + 2 * u * np.abs(wd)
        assert np.all(np.abs(g0 - ws) <= 2 * _ulp(ws, T))
        e = np.abs(g1 - wd)
        assert np.all(np.minimum(e, 360 - e) <= lim_wd), float(np.max(e / lim_wd))
    else:
        uu, vv = pw.polar_to_xy(aH, bH)
        ang = (270 - bH) * H(pw.radian)
        da = u * np.abs(270 - bH) * pw.radian + 2 * u * np.abs(ang)
        cs, sn = np.cos(ang), np.sin(ang)
        assert np.all(np.abs(g0 - uu) <= aH * (2 * _ulp(cs, T) + np.abs(sn) * da + 2 * u * np.abs(cs)))
        assert np.all(np.abs(g1 - vv) <= aH * (2 * _ulp(sn, T) + np.abs(cs) * da + 2 * u * np.abs(sn)))


# ---- e. the same bits from every kernel and family ------------------------------------------------

# kind: (outputs per 4 inputs, a kind of another family: with it the program runs FAM_ALL)
KINDS = {
    "EPI_PLAIN": (4, ("EPI_EXP", "EPI_COSSIN")), "EPI_UV2DDFF": (4, ("EPI_EXP",)), "EPI_DDFF2UV": (4, ("EPI_LOG",)),
    "EPI_QT2R": (2, ("EPI_COSSIN",)), "EPI_QT2QTR": (6, ("EPI_AFFINE",)), "EPI_RT2Q": (2, ("EPI_RT2D",)),
    "EPI_RT2RTQ": (6, ("EPI_IMPUTE_NAN",)),
    "EPI_AFFINE": (4, ("EPI_QT2R",)), "EPI_AFFINE_INV": (4, ("EPI_ATAN2",)), "EPI_EXP": (4, ("EPI_UV2DDFF",)),
    "EPI_LOG": (4, ("EPI_DT2R",)), "EPI_IMPUTE_NAN": (4, ("EPI_RT2Q",)),
    "EPI_COSSIN": (8, ("EPI_QT2QTR",)), "EPI_ATAN2": (2, ("EPI_EXP",)), "EPI_RT2D": (2, ("EPI_RT2Q",)),
    "EPI_RT2RTD": (6, ("EPI_LOG",)), "EPI_DT2R": (2, ("EPI_QT2R",)), "EPI_DT2DTR": (6, ("EPI_AFFINE_INV",)),
}


def _field_for(kind, shape, rng):
    """Values the kind is meant for, with both sides of the float32 fast-path switches."""
    x = rng.standard_normal(shape)
    a, b = x[:, 0::2], x[:, 1::2]
    t = rng.choice(_t_sweep(), a.shape)
    if kind in ("EPI_QT2R", "EPI_QT2QTR"):
        a[:] = np.abs(a) * 3e-3
        b[:] = t
    elif kind in ("EPI_RT2Q", "EPI_RT2RTQ", "EPI_RT2D", "EPI_RT2RTD"):
        a[:] = np.abs(a) * 50 * (rng.random(a.shape) < 0.9)  # some r == 0
        b[:] = t
    elif kind in ("EPI_DT2R", "EPI_DT2DTR"):
        b[:] = t
        a[:] = t - np.abs(a) * 15
    elif kind == "EPI_LOG":
        x = np.abs(x)
    elif kind in ("EPI_UV2DDFF", "EPI_ATAN2"):
        x *= 8
    elif kind == "EPI_DDFF2UV":
        b[:] = (b * 100) % 360
    elif kind == "EPI_AFFINE_INV" or kind == "EPI_AFFINE":
        x = x * 40 + 270
    x[rng.random(shape) < 0.01] = np.nan
    return x


def _program(kind, extra, n_in):
    """kind on input columns [0, n_in), the extra kinds after it; clip bounds on every third
    output column, the mask on every fourth, every column its own pressure."""
    from anemoi_transform_b200 import _cabi

    params = {"EPI_AFFINE": (1.8, -459.67), "EPI_AFFINE_INV": (1.8, -459.67), "EPI_IMPUTE_NAN": (-1.5, 0.0),
              "EPI_COSSIN": (float(np.deg2rad(1.0)), 0.0), "EPI_ATAN2": (float(np.rad2deg(1.0)), 1.0)}
    segs, out = [], 0
    for k in (kind, *extra):
        segs.append((getattr(_cabi, k), len(segs) * n_in, n_in, out, *params.get(k, (1.0, 0.0))))
        out += n_in // 4 * KINDS[k][0]
    CL, CH, MK = _cabi.COL_CLIP_LO, _cabi.COL_CLIP_HI, _cabi.COL_MASK
    cols = [(-1.0, 50.0, 50000.0 + 1000.0 * c, (CL | CH if c % 3 == 0 else 0) | (MK if c % 4 == 1 else 0)) for c in range(out)]
    return segs, cols, n_in // 4 * KINDS[kind][0]


def _matrices(rng, n_src):
    """One matrix per fused instantiation: uniform 4, uniform 12, ragged (0..9, empty rows), and
    ragged with one row of 1500 entries (> kSegCap: the FALLBACK staging).  Rows sum to 1, so the
    regridded values stay in the kinds' ranges."""
    from scipy.sparse import csr_array

    n_tgt = 300
    out = {}
    for name, lengths in (("uniform4", np.full(n_tgt, 4)), ("uniform12", np.full(n_tgt, 12)),
                          ("ragged", rng.integers(0, 10, n_tgt)), ("long_row", np.r_[rng.integers(1, 10, 37), 1500, rng.integers(1, 10, n_tgt - 38)])):
        indptr = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
        indices = np.concatenate([np.sort(rng.choice(n_src, k, replace=False)) for k in lengths]).astype(np.int32)
        data = np.concatenate([np.full(k, 1.0 / k) for k in lengths]).astype(np.float32)
        out[name] = csr_array((data, indices, indptr), shape=(n_tgt, n_src))
    return out


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_every_kernel_and_family_gives_the_same_bits(cuda, kind):
    import torch

    from anemoi_transform_b200.device import CsrMatrix, Epilogue

    rng = np.random.default_rng(sorted(KINDS).index(kind))
    n_in, n_rows = 32, 2000
    extra = KINDS[kind][1]
    alone, alone_cols, n_k = _program(kind, (), n_in)
    mixed, mixed_cols, _ = _program(kind, extra, n_in)
    width = n_in * (1 + len(extra))
    x = np.concatenate([_field_for(kind, (n_rows, n_in), rng)] + [_field_for(k, (n_rows, n_in), rng) for k in extra], axis=1)
    mask = torch.from_numpy((rng.random(n_rows) < 0.3).astype(np.uint8)).cuda()
    epi_a, epi_m = Epilogue(alone, alone_cols), Epilogue(mixed, mixed_cols)
    for T, tdt in ((np.float32, torch.float32), (np.float64, torch.float64)):
        X = torch.from_numpy(x.astype(T)).cuda()
        ref = epi_a.apply(X, out=_sentinel(n_rows, len(alone_cols), tdt), row_mask=mask).cpu().numpy()[:, :n_k]
        got = epi_m.apply(X, out=_sentinel(n_rows, len(mixed_cols), tdt), row_mask=mask).cpu().numpy()[:, :n_k]
        _bits_equal(got, ref)  # own family vs FAM_ALL
        gather = torch.from_numpy(rng.integers(0, n_rows, 300)).cuda()  # every index a valid row
        gm = torch.from_numpy((rng.random(300) < 0.3).astype(np.uint8)).cuda()
        want = epi_a.apply(X[gather].contiguous(), out=_sentinel(300, len(alone_cols), tdt), row_mask=gm).cpu().numpy()[:, :n_k]
        for epi, cols in ((epi_a, alone_cols), (epi_m, mixed_cols)):
            got = epi.apply(X, out=_sentinel(300, len(cols), tdt), row_mask=gm, gather=gather).cpu().numpy()[:, :n_k]
            _bits_equal(got, want)
    X = torch.from_numpy(x.astype(np.float32)).cuda()
    for name, m in _matrices(rng, n_rows).items():
        csr = CsrMatrix.from_scipy(m)
        tm = torch.from_numpy((rng.random(m.shape[0]) < 0.3).astype(np.uint8)).cuda()
        y = csr.apply(X, n_fields=width)
        want = epi_a.apply(y, out=_sentinel(m.shape[0], len(alone_cols), torch.float32), row_mask=tm).cpu().numpy()[:, :n_k]
        for label, epi, cols in (("own family", epi_a, alone_cols), ("FAM_ALL", epi_m, mixed_cols)):
            got = epi.apply_fused(csr, X, out=_sentinel(m.shape[0], len(cols), torch.float32), row_mask=tm).cpu().numpy()[:, :n_k]
            try:
                _bits_equal(got, want)
            except AssertionError as e:
                raise AssertionError(f"{kind} fused ({name}, {label}): {e}") from None
