"""Oracle: first-order conservative matrices between structured grids.

TEST INFRASTRUCTURE — see oracle/__init__.py.

The `method="structured-conservative"` recipe builds its matrix on the device
(`at_conservative_matrix_count` / `_fill`) between two global structured grids.  Neither MIR's
grid-box-average nor atlas is available offline and parity with their weights is unpinned; this
module restates the scheme in numpy — `conservative_matrix` is what the device builder is
checked against, bit for bit — and is pinned in tests/test_oracle_conservative_matrix.py by a
brute force over every pair of boxes and by the scheme's defining properties: rows sum to 1,
a grid onto itself is the identity, nested grids take their sub-boxes' area shares, and the
area integral of a field is kept.

Boxes.  Row k of a grid (rows north → south) spans the latitudes between the midpoints of its
neighbouring rows, ±90° at the ends, kept as z = sin(latitude) (`box_tables`); its point i
covers [lon0_k + (i - ½)Δ_k, lon0_k + (i + ½)Δ_k), Δ_k = 360/n_k.  A target box's weight on a
source box is (dz / dz_T) · (piece / wc): the band overlap over the target's band, times the
longitude overlap over the target's width, both measured in source-cell units on the source
row (x = the target's start, wc = n_k / n_T its width).
"""

from __future__ import annotations

import numpy as np
from scipy.sparse import csr_array

from .structured_matrix import check_global, structured_rows


def box_tables(rows) -> tuple[np.ndarray, np.ndarray]:
    """(z_north, z_south) of each row's band, rows north → south, z = sin(latitude)."""
    row_lat = rows[0]
    edges = [90.0] + [(row_lat[k - 1] + row_lat[k]) / 2.0 for k in range(1, row_lat.size)] + [-90.0]
    z = np.sin(np.deg2rad(np.array(edges, dtype=np.float64)))
    return z[:-1], z[1:]


def conservative_matrix(src_rows, tgt_rows, weights_dtype=np.float32):
    """First-order conservative weights from the grid of `src_rows` to the grid of `tgt_rows`
    (both as `structured_rows` returns them) → (data, indices int32, indptr int32, shape), the
    rows in the target's storage order, columns ascending and unique in every row.

    float64 without contraction, weights rounded to `weights_dtype` last.  An overlap is
    dropped when dz <= 0 or when its piece is shorter than 1e-9 of a source cell.  On a source
    row the target interval touches at most n_k + 1 cells; when it touches n_k + 1, the first
    and the last are the same point and their pieces are summed into one entry."""
    zn_s, zs_s = box_tables(src_rows)
    zn_t, zs_t = box_tables(tgt_rows)
    _, lon0_s, first_s, count_s = src_rows
    _, lon0_t, first_t, count_t = tgt_rows
    n_src, n_tgt = int(count_s.sum()), int(count_t.sum())
    src_order = range(first_s.size) if first_s[0] < first_s[-1] else range(first_s.size - 1, -1, -1)
    rows_out, cols_out, w_out = [], [], []
    for r in range(first_t.size):
        n_t = int(count_t[r])
        d_t = 360.0 / n_t
        i = np.arange(n_t, dtype=np.int64)
        start = lon0_t[r] + (i - 0.5) * d_t
        dz_t = zn_t[r] - zs_t[r]
        for k in src_order:
            dz = min(zn_t[r], zn_s[k]) - max(zs_t[r], zs_s[k])
            if not dz > 0.0:
                continue
            n = int(count_s[k])
            d_s = 360.0 / n
            x = np.mod(start - (lon0_s[k] - d_s / 2.0), 360.0) / d_s
            x = np.where(x >= n, x - n, x)  # a remainder rounded up to 360 is cell 0
            wc = n / n_t
            end = x + wc
            a = dz / dz_t
            i0 = np.floor(x).astype(np.int64)
            last = np.ceil(end).astype(np.int64) - 1
            merge = last - i0 == n
            first_piece = None
            for o in range(int((last - i0).max()) + 1):
                c = i0 + o
                p = np.minimum(end, c + 1.0) - np.maximum(x, c.astype(np.float64))
                if o == 0:
                    first_piece = p
                if o == n:
                    p = np.where(merge, p + first_piece, p)
                keep = (c <= last) & (p >= 1e-9)
                if o == 0:
                    keep &= ~merge
                rows_out.append(first_t[r] + i[keep])
                cols_out.append(first_s[k] + np.where(c >= n, c - n, c)[keep])
                w_out.append(a * (p[keep] / wc))
    rows_all = np.concatenate(rows_out) if rows_out else np.zeros(0, np.int64)
    cols_all = np.concatenate(cols_out) if cols_out else np.zeros(0, np.int64)
    w_all = np.concatenate(w_out) if w_out else np.zeros(0)
    order = np.lexsort((cols_all, rows_all))
    rows_all, cols_all, w_all = rows_all[order], cols_all[order], w_all[order]
    if rows_all.size and ((np.diff(rows_all) == 0) & (np.diff(cols_all) == 0)).any():
        raise AssertionError("a column appears twice in a row")
    indptr = np.concatenate(([0], np.cumsum(np.bincount(rows_all, minlength=n_tgt)))).astype(np.int32)
    return w_all.astype(weights_dtype), cols_all.astype(np.int32), indptr, (n_tgt, n_src)


def conservative_csr(src_lat, src_lon, tgt_lat, tgt_lon) -> csr_array:
    grids = []
    for lat, lon in ((src_lat, src_lon), (tgt_lat, tgt_lon)):
        rows = structured_rows(lat, lon)
        if rows is None:
            raise ValueError("grid is not a structured grid (rows of constant latitude, equally spaced longitudes)")
        check_global(rows)
        grids.append(rows)
    d, i, p, shape = conservative_matrix(*grids)
    return csr_array((d, i, p), shape=shape)
