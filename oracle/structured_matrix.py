"""Oracle: structured-grid interpolation matrices.

TEST INFRASTRUCTURE — see oracle/__init__.py.

The `method="structured-bilinear" | "structured-bicubic"` recipes build their matrix on the
device (`at_structured_matrix`) from a global structured grid: rows of constant latitude, row r
holding n_r points at lon0_r + i·(360/n_r) (octahedral / classic reduced Gaussian, full
Gaussian, regular lat-lon).  Neither MIR nor atlas is available offline and parity with their
weights is unpinned (as for oracle/matrix.py); this module restates the scheme in numpy —
`structured_matrix` is what the device builder is checked against, bit for bit — and is pinned
by its defining properties in tests/test_oracle_structured_matrix.py: rows sum to 1, a target
on a source point takes that point's value, the error on a smooth field falls with resolution,
targets poleward of the outermost rows are continuous.
"""

from __future__ import annotations

import numpy as np
from scipy.sparse import csr_array


def structured_rows(lat: np.ndarray, lon: np.ndarray):
    """(row_lat, row_lon0, row_first, row_count) of a structured grid given as its point lists,
    rows north → south (row_first indexes the points as stored), or None when the points are
    not such a grid.  Plain loop over the rows: the package's `structured_grid_rows` is the
    vectorised version of the same rules."""
    lat, lon = np.asarray(lat, dtype=np.float64).reshape(-1), np.asarray(lon, dtype=np.float64).reshape(-1)
    if lat.size < 2 or lon.size != lat.size:
        return None
    rows = []
    start = 0
    for k in range(1, lat.size + 1):
        if k == lat.size or lat[k] != lat[start]:
            n = k - start
            dlon = 360.0 / n
            if np.abs(lon[start:k] - (lon[start] + dlon * np.arange(n))).max() > 1e-6 * dlon:
                return None
            rows.append((lat[start], lon[start], start, n))
            start = k
    if len(rows) < 2:
        return None
    row_lat = np.array([r[0] for r in rows])
    d = np.diff(row_lat)
    if not ((d < 0).all() or (d > 0).all()):
        return None
    if d[0] > 0:  # stored south → north: the table runs north → south all the same
        rows = rows[::-1]
    return (np.array([r[0] for r in rows]), np.array([r[1] for r in rows]),
            np.array([r[2] for r in rows], dtype=np.int64), np.array([r[3] for r in rows], dtype=np.int64))  # fmt: skip


def check_global(rows) -> None:
    """ValueError unless the outermost row at each end lies within one row spacing of its pole."""
    row_lat = rows[0]
    for a, b in ((row_lat[0], row_lat[1]), (row_lat[-1], row_lat[-2])):
        if 90.0 - abs(a) > abs(a - b):
            raise ValueError(f"the source grid is not global: its outermost row at {a}° lies more than one row spacing from the pole")


def _lon_weights(t: np.ndarray, stencil: int) -> list[np.ndarray]:
    """Weights of the points i (bilinear: i, i+1; bicubic: i-1 … i+2) at offset t from point i."""
    if stencil == 2:
        return [1.0 - t, t]
    tp1, tm1, tm2 = t + 1.0, t - 1.0, t - 2.0
    return [t * tm1 * tm2 / -6.0, tp1 * tm1 * tm2 / 2.0, tp1 * t * tm2 / -2.0, tp1 * t * tm1 / 6.0]


def _lat_weights(y: list[np.ndarray], phi: np.ndarray) -> list[np.ndarray]:
    """Lagrange weights of the stencil rows at latitudes y (2: linear, 4: cubic)."""
    if len(y) == 2:
        t = (y[0] - phi) / (y[0] - y[1])
        return [1.0 - t, t]
    w = []
    for k in range(4):
        o = [m for m in range(4) if m != k]
        w.append((phi - y[o[0]]) / (y[k] - y[o[0]]) * ((phi - y[o[1]]) / (y[k] - y[o[1]])) * ((phi - y[o[2]]) / (y[k] - y[o[2]])))
    return w


def structured_matrix(rows, tgt_lat, tgt_lon, stencil: int, weights_dtype=np.float32):
    """Structured bilinear (stencil 2: 2 rows × 2 points) or bicubic (stencil 4: 4 rows × 4 points,
    cubic Lagrange in longitude on each row, then in latitude on the rows' latitudes) weights
    → (data float32[S²n], indices int32[S²n], indptr int32[n+1], shape).

    j is the last row (north → south) with latitude ≥ the target's, -1 north of every row; the
    stencil takes rows j, j+1 (bilinear) or j-1 … j+2 (bicubic).  Rows beyond an outermost row
    are that end's rows seen across the pole: latitude ±180 - φ_k, longitudes shifted by 180°,
    row k's columns; an outermost row on the pole itself is the mirror's centre and is not
    repeated.  float64, weights rounded to float32 last (`weights_dtype=np.float64` keeps them);
    each target row stable-sorted by column, explicit zeros and duplicate columns kept.  Rows
    of the table are clamped to the grid, so the caller rejects targets outside [-90, 90]."""
    if stencil not in (2, 4):
        raise ValueError(f"stencil must be 2 or 4, not {stencil}")
    row_lat, row_lon0, row_first, row_count = rows
    R = row_lat.size
    if R < stencil:
        raise ValueError(f"a {stencil}-row stencil needs at least {stencil} rows, the grid has {R}")
    tgt_lat, tgt_lon = np.asarray(tgt_lat, dtype=np.float64).reshape(-1), np.asarray(tgt_lon, dtype=np.float64).reshape(-1)
    n = tgt_lat.size
    n_src = int(row_count.sum())
    # j = (number of rows with φ_k >= φ) - 1
    j = np.searchsorted(-row_lat, -tgt_lat, side="right").astype(np.int64) - 1
    north_pole, south_pole = int(row_lat[0] == 90.0), int(row_lat[R - 1] == -90.0)
    y, lon0, first, count = [], [], [], []
    for s in range(stencil):
        v = j + (s - (stencil // 2 - 1))  # virtual row index
        k = np.where(v < 0, -v - 1 + north_pole, np.where(v >= R, 2 * R - 1 - v - south_pole, v)).clip(0, R - 1)
        lat_k, lon_k = row_lat[k], row_lon0[k]
        y.append(np.where(v < 0, 180.0 - lat_k, np.where(v >= R, -180.0 - lat_k, lat_k)))
        lon0.append(np.where((v < 0) | (v >= R), lon_k + 180.0, lon_k))
        first.append(row_first[k])
        count.append(row_count[k])
    wlat = _lat_weights(y, tgt_lat)
    cols, w = [], []
    for s in range(stencil):
        nr = count[s]
        x = np.mod(tgt_lon - lon0[s], 360.0) / (360.0 / nr)
        i = np.floor(x)
        wlon = _lon_weights(x - i, stencil)
        i = i.astype(np.int64) % nr
        for p in range(stencil):
            o = p - (stencil // 2 - 1)
            cols.append(first[s] + (i + o + nr) % nr)
            w.append(wlat[s] * wlon[p])
    cols, w = np.stack(cols, axis=1), np.stack(w, axis=1)
    order = np.argsort(cols, axis=1, kind="stable")
    cols = np.take_along_axis(cols, order, axis=1)
    w = np.take_along_axis(w, order, axis=1)
    nnz = stencil * stencil
    indptr = (nnz * np.arange(n + 1)).astype(np.int32)
    return w.astype(weights_dtype).ravel(), cols.astype(np.int32).ravel(), indptr, (n, n_src)


def structured_csr(src_lat, src_lon, tgt_lat, tgt_lon, stencil: int) -> csr_array:
    rows = structured_rows(src_lat, src_lon)
    if rows is None:
        raise ValueError("source grid is not a structured grid (rows of constant latitude, equally spaced longitudes)")
    check_global(rows)
    d, i, p, shape = structured_matrix(rows, tgt_lat, tgt_lon, stencil)
    return csr_array((d, i, p), shape=shape)
