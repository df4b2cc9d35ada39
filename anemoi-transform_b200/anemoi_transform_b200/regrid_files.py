"""The two on-disk artefacts the `regrid` filter consumes — reference
`commands/make-regrid-file.py:142-160` (matrix npz) and `:225-242` (global-on-LAM mask npz).

The file formats and the mask computation live here.  Building an interpolation matrix is
MIR's job in the reference (`earthkit.regrid.utils.mir.mir_make_matrix` + the external `mir`
binary, neither available offline); any scipy sparse matrix can be written with
`save_regrid_matrix`, and four builders run locally on the device:

    make_bilinear_matrix    4-point bilinear weights from a regular, longitude-periodic lat-lon
                            source grid (`at_bilinear_matrix`; bitwise the numpy restatement
                            oracle/matrix.py) — what `regrid(in_grid=…, out_grid=…,
                            method="linear")` uses in place of earthkit-regrid's inventory
    make_structured_matrix  structured bilinear (2 rows × 2 points) or bicubic (4 rows × 4
                            points) weights from any global structured grid — octahedral and
                            classic reduced Gaussian, full Gaussian, regular lat-lon
                            (`at_structured_matrix`; bitwise oracle/structured_matrix.py) — what
                            `method="structured-bilinear" | "structured-bicubic"` uses
    make_conservative_matrix
                            first-order conservative (area-weighted grid-box average) weights
                            between two global structured grids (`at_conservative_matrix_count`
                            / `_fill`; bitwise oracle/conservative_matrix.py) — what
                            `method="structured-conservative"` uses
    make_healpix_conservative_matrix
                            first-order conservative weights with the true HEALPix pixels,
                            between a HEALPix grid and a HEALPix or global structured grid
                            (`at_healpix_conservative_count` / `_fill`; bitwise
                            oracle/healpix_conservative.py) — what `method="healpix-conservative"` uses
    make_knn_matrix         nearest neighbour (k = 1) or inverse-distance weights of the k
                            nearest sources, on the device kNN

None is MIR's scheme (nor atlas's) for reduced Gaussian sources, so fields regridded with them
are comparable with a scipy matrix of the same construction, not with a MIR matrix.
"""

from __future__ import annotations

from typing import Any

import numpy as np


def save_regrid_matrix(output: str, sparse_array: Any, lat1, lon1, lat2, lon2) -> None:
    """Write a CSR matrix with the schema `RegridFilter(matrix=…)` / `MIRMatrix` reads
    (make-regrid-file.py:150-160)."""
    m = sparse_array.tocsr() if hasattr(sparse_array, "tocsr") else sparse_array
    np.savez(
        output,
        matrix_data=m.data,
        matrix_indices=m.indices,
        matrix_indptr=m.indptr,
        matrix_shape=m.shape,
        in_latitudes=lat1,
        in_longitudes=lon1,
        out_latitudes=lat2,
        out_longitudes=lon2,
    )


def make_global_on_lam_mask(lam_lat, lam_lon, global_lat, global_lon, output: str, **kwargs: Any) -> np.ndarray:
    """`anemoi-transform make-regrid-file global-on-lam-mask`: the sorted indices of the global
    points within `distance_km` of a LAM point, computed on the device, written as `mask`
    (what `RegridFilter(mask=…)` / `MaskedRegrid` loads)."""
    from .spatial import global_on_lam_mask

    mask = global_on_lam_mask(lam_lat, lam_lon, global_lat, global_lon, **kwargs)
    np.savez(output, mask=mask)
    return mask


def make_knn_matrix(lat1, lon1, lat2, lon2, output: str | None = None, k: int = 4, power: float = 1.0):
    """A [n_target, n_source] CSR matrix from the k nearest source points of every target
    (device kNN on the unit sphere): weight ∝ 1 / distance**power, rows normalised to 1, columns
    sorted within a row; a target that coincides with a source takes that source alone.
    k = 1 is nearest-neighbour regridding as a matrix.  Written with the regrid-file schema when
    `output` is given.  → (data float32, indices int32, indptr int32, shape)."""
    from .device import KnnIndex
    from .spatial import latlon_to_xyz

    lat1, lon1, lat2, lon2 = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (lat1, lon1, lat2, lon2))
    n_src, n_tgt = lat1.size, lat2.size
    if not 1 <= k <= n_src:
        raise ValueError(f"k={k} must be between 1 and the number of source points ({n_src})")
    index = KnnIndex(latlon_to_xyz(lat1, lon1))
    try:
        idx, dist, _ = index.query(latlon_to_xyz(lat2, lon2), k=k)
        idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    finally:
        index.close()
    exact = dist[:, 0] == 0.0
    with np.errstate(divide="ignore"):
        w = 1.0 / dist**power
    w[exact] = 0.0
    w[exact, 0] = 1.0
    w /= w.sum(axis=1, keepdims=True)
    order = np.argsort(idx, axis=1, kind="stable")
    indices = np.take_along_axis(idx, order, axis=1).astype(np.int32).ravel()
    data = np.take_along_axis(w, order, axis=1).astype(np.float32).ravel()
    indptr = (k * np.arange(n_tgt + 1)).astype(np.int32)
    shape = (n_tgt, n_src)
    if output is not None:
        np.savez(output, matrix_data=data, matrix_indices=indices, matrix_indptr=indptr, matrix_shape=np.asarray(shape),
                 in_latitudes=lat1, in_longitudes=lon1, out_latitudes=lat2, out_longitudes=lon2)  # fmt: skip
    return data, indices, indptr, shape


def regular_grid_parameters(lat, lon):
    """(lat0, dlat, n_lat, lon0, dlon, n_lon) when (lat, lon) are the point lists of a row-major
    regular lat-lon grid that wraps in longitude, else None."""
    lat, lon = np.asarray(lat, dtype=np.float64).reshape(-1), np.asarray(lon, dtype=np.float64).reshape(-1)
    n = lat.size
    if n < 4 or lon.size != n:
        return None
    change = np.flatnonzero(lat != lat[0])
    n_lon = int(change[0]) if change.size else 0
    if n_lon < 2 or n % n_lon or n // n_lon < 2:
        return None
    n_lat = n // n_lon
    rows, cols = lat.reshape(n_lat, n_lon), lon.reshape(n_lat, n_lon)
    if not (rows == rows[:, :1]).all() or not (cols == cols[:1, :]).all():
        return None
    lat0, lon0 = float(rows[0, 0]), float(cols[0, 0])
    dlat, dlon = float(rows[1, 0] - rows[0, 0]), float(cols[0, 1] - cols[0, 0])
    if dlat == 0.0 or dlon <= 0.0:
        return None
    regular = (
        np.abs(rows[:, 0] - (lat0 + dlat * np.arange(n_lat))).max() <= 1e-6 * abs(dlat)
        and np.abs(cols[0] - (lon0 + dlon * np.arange(n_lon))).max() <= 1e-6 * dlon
        and abs(n_lon * dlon - 360.0) <= 1e-6 * dlon
    )
    return (lat0, dlat, n_lat, lon0, dlon, n_lon) if regular else None


def make_bilinear_matrix(lat1, lon1, lat2, lon2, output: str | None = None):
    """A [n_target, n_source] CSR matrix of 4-point bilinear weights from a regular,
    longitude-periodic lat-lon source grid, built on the device.  Four entries per row, sorted
    by column, explicit zeros kept (they propagate NaN like scipy).  Written with the
    regrid-file schema when `output` is given.  → (data float32, indices int32, indptr int32, shape)."""
    from ctypes import c_void_p

    from ._cabi import call
    from .device import require_cuda, stream_ptr, to_device_f64

    torch = require_cuda()
    prm = regular_grid_parameters(lat1, lon1)
    if prm is None:
        raise NotImplementedError(
            "linear interpolation is built locally for regular, longitude-periodic lat-lon source grids only; "
            "pass `matrix=` (make-regrid-file) for other sources, method='structured-bilinear' or "
            "'structured-bicubic' for global structured grids (reduced Gaussian, octahedral), or method='nearest'"
        )
    lat2, lon2 = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (lat2, lon2))
    n_tgt = int(lat2.size)
    lo, hi = sorted((prm[0], prm[0] + prm[1] * (prm[2] - 1)))
    if n_tgt and (lat2.min() < lo - 1e-9 or lat2.max() > hi + 1e-9):
        raise ValueError(f"target latitudes [{lat2.min()}, {lat2.max()}] leave the source grid's [{lo}, {hi}]")
    tlat, tlon = to_device_f64(lat2), to_device_f64(lon2)
    data = torch.empty((4 * n_tgt,), dtype=torch.float32, device="cuda")
    indices = torch.empty((4 * n_tgt,), dtype=torch.int32, device="cuda")
    call("at_bilinear_matrix", *prm[:3], *prm[3:], c_void_p(tlat.data_ptr()), c_void_p(tlon.data_ptr()), n_tgt, c_void_p(data.data_ptr()), c_void_p(indices.data_ptr()), stream_ptr())
    data, indices = data.cpu().numpy(), indices.cpu().numpy()
    indptr = (4 * np.arange(n_tgt + 1)).astype(np.int32)
    shape = (n_tgt, prm[2] * prm[5])
    if output is not None:
        np.savez(output, matrix_data=data, matrix_indices=indices, matrix_indptr=indptr, matrix_shape=np.asarray(shape),
                 in_latitudes=np.asarray(lat1), in_longitudes=np.asarray(lon1), out_latitudes=lat2, out_longitudes=lon2)  # fmt: skip
    return data, indices, indptr, shape


STRUCTURED_STENCILS = {"structured-bilinear": 2, "structured-bicubic": 4}


def structured_grid_rows(lat, lon):
    """The rows of a structured grid given as its point lists → (row_lat float64, row_lon0
    float64, row_first int64, row_count int64), rows north → south whatever the storage order
    (row_first indexes the points as stored), or None when the points are not such a grid.

    Rows are runs of consecutive points with equal latitude; row latitudes must be strictly
    monotone (north → south or south → north) and row r's n_r points lie at
    lon0_r + i·(360/n_r), i = 0 … n_r - 1, to 1e-6 of the spacing.  Whether the grid reaches the
    poles is `make_structured_matrix`'s concern."""
    lat, lon = np.asarray(lat, dtype=np.float64).reshape(-1), np.asarray(lon, dtype=np.float64).reshape(-1)
    n = lat.size
    if n < 2 or lon.size != n:
        return None
    first = np.flatnonzero(np.concatenate(([True], lat[1:] != lat[:-1])))
    if first.size < 2:
        return None
    row_lat = lat[first]
    d = np.diff(row_lat)
    if not ((d < 0).all() or (d > 0).all()):  # also catches NaN latitudes
        return None
    count = np.diff(np.append(first, n))
    dlon = 360.0 / count
    row = np.repeat(np.arange(first.size), count)
    local = np.arange(n) - first[row]
    off = np.abs(lon - (lon[first][row] + dlon[row] * local))
    if not (off <= 1e-6 * dlon[row]).all():
        return None
    rows = (row_lat, lon[first], first.astype(np.int64), count.astype(np.int64))
    return tuple(a[::-1].copy() for a in rows) if d[0] > 0 else rows


def _require_global(row_lat, method: str, which: str) -> None:
    """ValueError unless the outermost row at each end lies within one row spacing of its pole."""
    for a, b in ((row_lat[0], row_lat[1]), (row_lat[-1], row_lat[-2])):
        if 90.0 - abs(a) > abs(a - b):
            raise ValueError(f"{method}: the {which} grid is not global: its outermost row at {a}° lies more than one row spacing from the pole")


def make_structured_matrix(lat1, lon1, lat2, lon2, method: str, output: str | None = None):
    """A [n_target, n_source] CSR matrix of structured-grid interpolation weights, built on the
    device.  `method="structured-bilinear"`: 2 rows × 2 points, linear in longitude on each row,
    then in latitude (4 entries per target).  `"structured-bicubic"`: 4 rows × 4 points, cubic
    Lagrange in longitude on each row, then in latitude on the rows' latitudes (16 entries;
    weights go negative).  The source is any global structured grid (`structured_grid_rows`);
    targets poleward of its outermost rows take the rows across the pole.  Entries sorted by
    column, explicit zeros kept (they propagate NaN like scipy).  Written with the regrid-file
    schema when `output` is given.  → (data float32, indices int32, indptr int32, shape).

    NotImplementedError when the source is not a structured grid, ValueError when it is not
    global (an outermost row further than one row spacing from its pole) or a target latitude
    is outside [-90, 90]."""
    from ctypes import c_void_p

    from ._cabi import call
    from .device import require_cuda, stream_ptr, to_device_f64

    if method not in STRUCTURED_STENCILS:
        raise ValueError(f"method {method!r} is not one of {tuple(STRUCTURED_STENCILS)}")
    stencil = STRUCTURED_STENCILS[method]
    hp = healpix_grid_of(lat1, lon1)
    if hp is not None and hp[1] == "nested":  # built in ring order, then the columns mapped
        from .synthetic import healpix

        data, indices, indptr, shape = make_structured_matrix(*healpix(hp[0], "ring"), lat2, lon2, method)
        data, indices = _nested_columns(hp[0], data, indices, indptr)
        if output is not None:
            np.savez(output, matrix_data=data, matrix_indices=indices, matrix_indptr=indptr, matrix_shape=np.asarray(shape),
                     in_latitudes=np.asarray(lat1), in_longitudes=np.asarray(lon1), out_latitudes=np.asarray(lat2), out_longitudes=np.asarray(lon2))  # fmt: skip
        return data, indices, indptr, shape
    rows = structured_grid_rows(lat1, lon1)
    if rows is None:
        raise NotImplementedError(
            f"{method} is built locally for global structured source grids only (rows of constant, strictly monotone "
            "latitude, each with equally spaced longitudes over 360°); pass `matrix=` (make-regrid-file) for other sources"
        )
    row_lat, row_lon0, row_first, row_count = rows
    if row_lat.size < stencil:
        raise NotImplementedError(f"{method} needs a source grid of at least {stencil} rows, this one has {row_lat.size}")
    _require_global(row_lat, method, "source")
    lat2, lon2 = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (lat2, lon2))
    n_tgt, n_src = int(lat2.size), int(np.size(lat1))
    if n_tgt and not (np.abs(lat2) <= 90.0).all():
        raise ValueError(f"{method}: target latitudes must lie in [-90, 90] (got [{lat2.min()}, {lat2.max()}])")
    if n_tgt and not np.isfinite(lon2).all():
        raise ValueError(f"{method}: target longitudes must be finite")
    torch = require_cuda()
    tables = [to_device_f64(row_lat), to_device_f64(row_lon0)] + [torch.from_numpy(a).cuda() for a in (row_first, row_count)]
    tlat, tlon = to_device_f64(lat2), to_device_f64(lon2)
    nnz = stencil * stencil
    data = torch.empty((nnz * n_tgt,), dtype=torch.float32, device="cuda")
    indices = torch.empty((nnz * n_tgt,), dtype=torch.int32, device="cuda")
    call("at_structured_matrix", *(c_void_p(t.data_ptr()) for t in tables), row_lat.size, n_src, stencil, c_void_p(tlat.data_ptr()), c_void_p(tlon.data_ptr()), n_tgt, c_void_p(data.data_ptr()), c_void_p(indices.data_ptr()), stream_ptr())
    data, indices = data.cpu().numpy(), indices.cpu().numpy()
    indptr = (nnz * np.arange(n_tgt + 1)).astype(np.int32)
    shape = (n_tgt, n_src)
    if output is not None:
        np.savez(output, matrix_data=data, matrix_indices=indices, matrix_indptr=indptr, matrix_shape=np.asarray(shape),
                 in_latitudes=np.asarray(lat1), in_longitudes=np.asarray(lon1), out_latitudes=lat2, out_longitudes=lon2)  # fmt: skip
    return data, indices, indptr, shape


def box_z_edges(row_lat):
    """The latitude edges of a structured grid's boxes as z = sin(latitude), rows north → south:
    row k spans [z[k + 1], z[k]], edges halfway between row latitudes and ±90° at the ends.
    The device builder only compares and subtracts these, so an edge two grids share is the
    same double on both."""
    row_lat = np.asarray(row_lat, dtype=np.float64)
    edges = np.concatenate(([90.0], (row_lat[:-1] + row_lat[1:]) / 2.0, [-90.0]))
    return np.sin(np.deg2rad(edges))


def _box_rows(lat, lon, method: str, which: str):
    """(zn, zs, lon0, first, count) of a global structured grid's boxes, rows north → south;
    NotImplementedError when the grid is not structured, ValueError when it is not global."""
    rows = structured_grid_rows(lat, lon)
    if rows is None:
        raise NotImplementedError(
            f"{method} is built locally between global structured grids only (rows of constant, strictly monotone "
            f"latitude, each with equally spaced longitudes over 360°); the {which} grid is not one: pass `matrix=` "
            "(make-regrid-file) for other grids"
        )
    if not (np.abs(rows[0]) <= 90.0).all():
        raise ValueError(f"{method}: the {which} grid has rows outside [-90, 90] (got [{rows[0].min()}, {rows[0].max()}])")
    _require_global(rows[0], method, which)
    z = box_z_edges(rows[0])
    return (z[:-1], z[1:], *rows[1:])


def make_conservative_matrix(lat1, lon1, lat2, lon2, output: str | None = None):
    """A [n_target, n_source] CSR matrix of first-order conservative (area-weighted grid-box
    average) weights between two global structured grids, built on the device.  Both grids are
    cut into boxes: a latitude band between the midpoints of neighbouring rows (±90° at the
    ends; a row on the pole is a cap cut into wedges) times the longitude interval half a
    spacing either side of each point.  Target t's weight on source s is the area of their
    overlap over the area of t, so rows sum to 1 and the area integral of a field is kept.
    Entries sorted by column, unique; overlaps shorter than 1e-9 of a source cell are dropped.
    A HEALPix grid given as points gets these latitude-band boxes too, not its pixels: use
    `make_healpix_conservative_matrix` for the true pixels.
    Written with the regrid-file schema when `output` is given.
    → (data float32, indices int32, indptr int32, shape).

    NotImplementedError when either grid is not a structured grid, ValueError when either is not
    global (an outermost row further than one row spacing from its pole, or a row outside
    [-90, 90]) or when the matrix has more entries than int32 offsets can hold."""
    from ctypes import c_void_p

    from ._cabi import call
    from .device import require_cuda, stream_ptr, to_device_f64

    method = "structured-conservative"
    grids = {which: _box_rows(lat, lon, method, which) for which, (lat, lon) in (("source", (lat1, lon1)), ("target", (lat2, lon2)))}
    tgt = grids["target"]
    if tgt[3][0] > tgt[3][-1]:  # stored south → north: the device wants the target's rows in storage order
        tgt = tuple(a[::-1].copy() for a in tgt)
    n_src, n_tgt = int(np.size(lat1)), int(np.size(lat2))
    torch = require_cuda()

    def upload(t):
        return [to_device_f64(a) for a in t[:3]] + [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in t[3:]]

    src_d, tgt_d = upload(grids["source"]), upload(tgt)
    grid_args = (*(c_void_p(t.data_ptr()) for t in src_d), len(src_d[0]), n_src, *(c_void_p(t.data_ptr()) for t in tgt_d), len(tgt_d[0]), n_tgt)
    counts = torch.empty((n_tgt,), dtype=torch.int32, device="cuda")
    call("at_conservative_matrix_count", *grid_args, c_void_p(counts.data_ptr()), stream_ptr())
    indptr64 = torch.zeros((n_tgt + 1,), dtype=torch.int64, device="cuda")
    indptr64[1:] = torch.cumsum(counts, 0, dtype=torch.int64)
    nnz = int(indptr64[-1])
    if nnz > np.iinfo(np.int32).max:
        raise ValueError(f"{method}: the matrix has {nnz} entries, more than int32 offsets can hold")
    indptr = indptr64.to(torch.int32)
    data = torch.empty((nnz,), dtype=torch.float32, device="cuda")
    indices = torch.empty((nnz,), dtype=torch.int32, device="cuda")
    call("at_conservative_matrix_fill", *grid_args, c_void_p(indptr.data_ptr()), nnz, c_void_p(data.data_ptr()), c_void_p(indices.data_ptr()), stream_ptr())
    data, indices, indptr = data.cpu().numpy(), indices.cpu().numpy(), indptr.cpu().numpy()
    shape = (n_tgt, n_src)
    if output is not None:
        np.savez(output, matrix_data=data, matrix_indices=indices, matrix_indptr=indptr, matrix_shape=np.asarray(shape),
                 in_latitudes=np.asarray(lat1), in_longitudes=np.asarray(lon1), out_latitudes=np.asarray(lat2), out_longitudes=np.asarray(lon2))  # fmt: skip
    return data, indices, indptr, shape


def healpix_grid_of(lat, lon):
    """(nside, "ring" | "nested") when (lat, lon) are the pixel centres of a HEALPix grid in that
    order — 12·nside² points equal to `synthetic.healpix` to 1e-6 of the pixel spacing,
    longitudes compared mod 360 — else None."""
    from .synthetic import check_healpix, healpix

    lat, lon = np.asarray(lat, dtype=np.float64).reshape(-1), np.asarray(lon, dtype=np.float64).reshape(-1)
    n = lat.size
    nside = int(round(np.sqrt(n / 12.0)))
    if n == 0 or lon.size != n or 12 * nside * nside != n:
        return None
    try:
        check_healpix(nside)
    except ValueError:
        return None
    tol = 1e-6 * np.rad2deg(np.sqrt(4.0 * np.pi / n))
    for ordering in ("ring", "nested"):
        if ordering == "nested" and nside & (nside - 1):
            break
        hlat, hlon = healpix(nside, ordering)
        if np.abs(lat - hlat).max() <= tol and np.abs((lon - hlon + 180.0) % 360.0 - 180.0).max() <= tol:
            return nside, ordering
    return None


def _nested_columns(nside: int, data, indices, indptr):
    """A matrix built on the ring-ordered grid → the same on the nested grid: columns mapped
    ring → nested on the device (`at_healpix_reorder`), then each row sorted by column (stable)."""
    from ctypes import c_void_p

    from ._cabi import call
    from .device import require_cuda, stream_ptr

    torch = require_cuda()
    idx = torch.from_numpy(np.ascontiguousarray(indices, dtype=np.int32)).cuda()
    call("at_healpix_reorder", nside, 1, c_void_p(idx.data_ptr()), idx.numel(), c_void_p(idx.data_ptr()), stream_ptr())
    counts = torch.from_numpy(np.diff(np.asarray(indptr, dtype=np.int64))).cuda()
    row = torch.repeat_interleave(torch.arange(counts.numel(), device="cuda"), counts)
    order = torch.sort(row * (12 * nside * nside) + idx.to(torch.int64), stable=True).indices
    vals = torch.from_numpy(np.ascontiguousarray(data)).cuda()
    return vals[order].cpu().numpy(), idx[order].cpu().numpy()


def make_healpix_conservative_matrix(lat1, lon1, lat2, lon2, output: str | None = None):
    """A [n_target, n_source] CSR matrix of first-order conservative weights with the true
    HEALPix pixels, built on the device.  At least one grid is HEALPix (`healpix_grid_of`, ring
    or nested, any nside); the other is HEALPix or a global structured grid, whose boxes are
    those of `make_conservative_matrix`.  Target t's weight on source s is the area of their
    overlap over the area of t, computed exactly as polygon areas in the equal-area plane of the
    HEALPix projection, so rows sum to 1 and the area integral of a field is kept.  Entries
    sorted by column, unique; overlaps under 1e-9 of the smaller cell are dropped.  Written
    with the regrid-file schema when `output` is given.
    → (data float32, indices int32, indptr int32, shape).

    ValueError when neither grid is HEALPix (use "structured-conservative"), when the other grid
    is not global, or when the matrix has more entries than int32 offsets can hold;
    NotImplementedError when the other grid is not a structured grid."""
    from ctypes import c_void_p

    from ._cabi import call
    from .device import require_cuda, stream_ptr, to_device_f64

    method = "healpix-conservative"
    sides = {}
    for which, (lat, lon) in (("source", (lat1, lon1)), ("target", (lat2, lon2))):
        sides[which] = healpix_grid_of(lat, lon)
    if sides["source"] is None and sides["target"] is None:
        raise ValueError(f"{method}: neither grid is a HEALPix grid; use method='structured-conservative' between structured grids")
    n_src, n_tgt = int(np.size(lat1)), int(np.size(lat2))
    rows = {}
    for which, (lat, lon) in (("source", (lat1, lon1)), ("target", (lat2, lon2))):
        if sides[which] is None:
            r = _box_rows(lat, lon, method, which)
            if which == "target" and r[3][0] > r[3][-1]:  # the device wants the target's rows in storage order
                r = tuple(a[::-1].copy() for a in r)
            rows[which] = r
    torch = require_cuda()
    keep = []

    def side_args(which, n_points):
        hp = sides[which]
        if hp is not None:
            return (hp[0], 1 if hp[1] == "nested" else 0, *[c_void_p(0)] * 5, 0, n_points)
        dev = [to_device_f64(a) for a in rows[which][:3]] + [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in rows[which][3:]]
        keep.extend(dev)
        return (0, 0, *(c_void_p(t.data_ptr()) for t in dev), len(rows[which][0]), n_points)

    grid_args = (*side_args("source", n_src), *side_args("target", n_tgt))
    counts = torch.empty((n_tgt,), dtype=torch.int32, device="cuda")
    call("at_healpix_conservative_count", *grid_args, c_void_p(counts.data_ptr()), stream_ptr())
    indptr64 = torch.zeros((n_tgt + 1,), dtype=torch.int64, device="cuda")
    indptr64[1:] = torch.cumsum(counts, 0, dtype=torch.int64)
    nnz = int(indptr64[-1])
    if nnz > np.iinfo(np.int32).max:
        raise ValueError(f"{method}: the matrix has {nnz} entries, more than int32 offsets can hold")
    indptr = indptr64.to(torch.int32)
    data = torch.empty((nnz,), dtype=torch.float32, device="cuda")
    indices = torch.empty((nnz,), dtype=torch.int32, device="cuda")
    call("at_healpix_conservative_fill", *grid_args, c_void_p(indptr.data_ptr()), nnz, c_void_p(data.data_ptr()), c_void_p(indices.data_ptr()), stream_ptr())
    data, indices, indptr = data.cpu().numpy(), indices.cpu().numpy(), indptr.cpu().numpy()
    if sides["source"] is not None and sides["source"][1] == "nested":
        data, indices = _nested_columns(sides["source"][0], data, indices, indptr)
    shape = (n_tgt, n_src)
    if output is not None:
        np.savez(output, matrix_data=data, matrix_indices=indices, matrix_indptr=indptr, matrix_shape=np.asarray(shape),
                 in_latitudes=np.asarray(lat1), in_longitudes=np.asarray(lon1), out_latitudes=np.asarray(lat2), out_longitudes=np.asarray(lon2))  # fmt: skip
    return data, indices, indptr, shape
