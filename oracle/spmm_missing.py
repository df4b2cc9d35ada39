"""Oracle: the regrid matrix application with missing values (`at_spmm_missing`).

TEST INFRASTRUCTURE — see oracle/__init__.py.

A source value is missing when it is NaN (Inf is not).  For each target row and field, Σ′ sums
over the row's entries whose x is not NaN, sequentially in storage order from +0, in
numpy's result_type of weights and fields, multiply and add rounded separately (as
`oracle.spmm.csr_matvec_sequential`, which is scipy's csr_matvec):

    PROPAGATE  y = Σ w·x                       (scipy: a NaN reaches every row that references it)
    ALL        no entry missing: y = Σ w·x (no division);
               otherwise y = Σ′ w·x / Σ′ w, NaN when every entry is missing or Σ′ w is not > 0
    HEAVIEST   as ALL, and NaN whenever the row's heaviest entry is missing (the largest
               weight, the first in storage order on ties; it does not depend on the field)

The policy names of the package (`missing_values=`) are MIR's `nonlinear` options; these
semantics are the package's own and are not checked against MIR.  PINNED in
tests/test_oracle_spmm_missing.py: bitwise `csr_matvec_sequential` on NaN-free inputs, bitwise a
per-row loop over numpy scalars, and the properties of the scheme on the structured and
conservative matrices.
"""

from __future__ import annotations

import numpy as np

PROPAGATE, ALL, HEAVIEST = 0, 1, 2


def heaviest_entries(indptr, data) -> np.ndarray:
    """Storage position of each row's heaviest entry: its first entry, replaced in storage order
    by every later entry whose weight is strictly larger; -1 for an empty row."""
    indptr = np.asarray(indptr).astype(np.int64)
    n = indptr.shape[0] - 1
    lengths = np.diff(indptr)
    best = np.where(lengths > 0, indptr[:-1], -1)
    if n == 0 or not lengths.any():
        return best
    wmax = np.zeros(n, dtype=data.dtype)
    rows = np.nonzero(lengths > 0)[0]
    wmax[rows] = data[indptr[rows]]
    for j in range(1, int(lengths.max())):
        rows = np.nonzero(lengths > j)[0]
        p = indptr[rows] + j
        better = data[p] > wmax[rows]
        best[rows[better]] = p[better]
        wmax[rows[better]] = data[p[better]]
    return best


def csr_matvec_missing(indptr, indices, data, x, policy: int) -> np.ndarray:
    """y = A · x under a missing-value policy; x is one field [n_src] or a point-major batch
    [n_src, F].  Vectorised over rows by position-in-row."""
    if policy not in (PROPAGATE, ALL, HEAVIEST):
        raise ValueError(f"unknown policy {policy}")
    indptr = np.asarray(indptr).astype(np.int64)
    indices = np.asarray(indices)
    dtype = np.result_type(data.dtype, x.dtype)
    a = data.astype(dtype, copy=False)
    xv = x.astype(dtype, copy=False)
    n = indptr.shape[0] - 1
    lengths = np.diff(indptr)
    shape = (n,) + xv.shape[1:]
    y = np.zeros(shape, dtype=dtype)
    ws = np.zeros(shape, dtype=dtype)
    miss = np.zeros(shape, dtype=bool)
    heavy = np.zeros(shape, dtype=bool)
    hp = heaviest_entries(indptr, data) if policy == HEAVIEST else None
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        for j in range(int(lengths.max()) if n else 0):
            rows = np.nonzero(lengths > j)[0]
            p = indptr[rows] + j
            w = a[p] if xv.ndim == 1 else a[p][:, None]
            xs = xv[indices[p]]
            if policy == PROPAGATE:
                y[rows] = y[rows] + w * xs
                continue
            nan = np.isnan(xs)
            y[rows] = np.where(nan, y[rows], y[rows] + w * xs)
            ws[rows] = np.where(nan, ws[rows], ws[rows] + w)
            miss[rows] |= nan
            if hp is not None:
                at_heaviest = p == hp[rows]
                heavy[rows] |= nan & (at_heaviest if xv.ndim == 1 else at_heaviest[:, None])
        if policy == PROPAGATE:
            return y
        ratio = y / ws
    return np.where(miss, np.where(heavy | ~(ws > 0), dtype.type(np.nan), ratio), y)
