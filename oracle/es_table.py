"""Oracle: numpy restatement of the float32 es(T) table of the humidity fast paths.

TEST INFRASTRUCTURE — see oracle/__init__.py.

Restates `fit_es_table` / `es_mixed_f64` (csrc/spmm.cu) and `es_from_table`
(csrc/epilogue.cuh): 400 cubics, one per 0.5 K from 150.16f K, each interpolating the float64
mixed-phase formula at four Chebyshev points of its interval, evaluated in float32 by three
FMAs.  The stated bound — relative error < 2e-7 against the float64 formula, Horner evaluation
included — is checked on this restatement in tests/test_oracle_pointwise.py, with no GPU.
"""

from __future__ import annotations

import math

import numpy as np

N, ZERO = 400, 200
T_TABLE = np.float32(250.16)  # node ZERO: the ice threshold as float32 (kEsTableT)
T_WATER = np.float32(273.16)  # node 246
T_LO, T_HI = np.float32(150.16), np.float32(350.15)  # es_table_covers: T_LO <= t < T_HI
# the fractions of the fit points; math.cos / math.exp are the C library's, like the host's std::
CHEB = np.array([0.5 * (1.0 - math.cos((2 * k + 1) * 3.14159265358979323846 / 8.0)) for k in range(4)])
_exp = np.vectorize(math.exp, otypes=[np.float64])


def es_mixed_f64(t):
    """The host's float64 formula, thresholds compared as float32 numbers (spmm.cu)."""
    t = np.asarray(t, dtype=np.float64)
    es_w = 611.21 * _exp(17.502 * (t - 273.16) / (t - 32.19))
    es_i = 611.21 * _exp(22.587 * (t - 273.16) / (t + 0.7))
    a = (t - 250.16) / 23.0
    return np.where(t <= float(T_TABLE), es_i, np.where(t >= float(T_WATER), es_w, a * a * es_w + (1.0 - a * a) * es_i))


def fit_es_table():
    """(N, 4) float32 coefficients (c0, c1, c2, c3) of c0 + c1 f + c2 f^2 + c3 f^3, f in [0, 1)."""
    nodes = float(T_TABLE) + 0.5 * (np.arange(N) - ZERO)
    dd = [es_mixed_f64(nodes + 0.5 * f) for f in CHEB]  # Newton divided differences
    for level in range(1, 4):
        for k in range(3, level - 1, -1):
            dd[k] = (dd[k] - dd[k - 1]) / (CHEB[k] - CHEB[k - level])
    c = [dd[3], 0.0, 0.0, 0.0]  # running polynomial, highest power first
    for deg, k in enumerate(range(2, -1, -1)):
        nc = [0.0] * 4
        for i in range(deg + 1):
            nc[i] = nc[i] + c[i]
            nc[i + 1] = nc[i + 1] - c[i] * CHEB[k]
        nc[deg + 1] = nc[deg + 1] + dd[k]
        c = nc
    return np.stack([c[3], c[2], c[1], c[0]], axis=1).astype(np.float32)


def _fma32(a, b, c):
    """float32 a*b + c rounded once: the product is exact in float64, the sum is rounded to odd
    in float64 (exact two-sum error, then the odd neighbour), and 53 >= 24 + 2 bits make the
    final rounding to float32 the correctly rounded one."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c = c.astype(np.float64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    even = (s.view(np.int64) & 1) == 0
    s = np.where((err != 0) & even, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def es_from_table(t, table=None):
    """float32 es(t) as the kernels evaluate it; t float32 with T_LO <= t < T_HI."""
    table = fit_es_table() if table is None else table
    t = np.asarray(t, dtype=np.float32)
    x = (t - T_TABLE) * np.float32(2.0)  # exact (Sterbenz), like the index and the fraction
    fl = np.floor(x)
    f = x - fl
    c = table[fl.astype(np.int64) + ZERO]
    return _fma32(_fma32(_fma32(c[:, 3], f, c[:, 2]), f, c[:, 1]), f, c[:, 0])


def table_sample_points():
    """float32 t in every interval: its 4 Chebyshev points, both ends, the midpoint, and the
    float32 neighbours of the table ends and of both thresholds (the ones just outside the
    table included)."""
    nodes = float(T_TABLE) + 0.5 * (np.arange(N) - ZERO)
    fr = np.concatenate([CHEB, [0.0, 0.5, 1.0]])
    t = (nodes[:, None] + 0.5 * fr[None, :]).astype(np.float32).ravel()
    edges = [T_LO, T_HI, T_TABLE, T_WATER]
    near = [np.nextafter(e, np.float32(d)) for e in edges for d in (-np.inf, np.inf)]
    return np.unique(np.concatenate([t, np.array(edges + near, dtype=np.float32)]))


def covers(t):
    """es_table_covers: the float32 fast paths read the table for these t."""
    return (t >= T_LO) & (t < T_HI)
