"""Synthetic grids, interpolation matrices and fields of the shapes BASELINE.json names.

There is no network in the build / bench environment, so the grids the reference would
download (`grids/named.py:27-70`) and the matrices MIR would compute
(`commands/make-regrid-file.py:142-160`) are generated locally.  The .npz schema written by
`save_regrid_npz` is exactly the one `make-regrid-file.py:150-160` writes and
`MIRMatrix.__init__` (`filters/fields/regrid.py:281-290`) reads.

numpy only — nothing here touches the GPU.
"""

from __future__ import annotations

import numpy as np


# ------------------------------------------------------------------------------ grids ---
def regular_latlon(step: float) -> tuple[np.ndarray, np.ndarray]:
    """Regular lat-lon grid incl. poles: lat 90→-90, lon 0→360-step, row-major N→S."""
    nlat = int(round(180.0 / step)) + 1
    nlon = int(round(360.0 / step))
    lat = 90.0 - step * np.arange(nlat, dtype=np.float64)
    lon = step * np.arange(nlon, dtype=np.float64)
    lats = np.repeat(lat, nlon)
    lons = np.tile(lon, nlat)
    return lats, lons


def gaussian_latitudes(n: int) -> np.ndarray:
    """The 2n Gaussian latitudes (degrees), north to south."""
    x, _ = np.polynomial.legendre.leggauss(2 * n)
    return np.rad2deg(np.arcsin(x))[::-1].copy()


def _reduced_grid(lat: np.ndarray, pl: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    lats = np.repeat(lat, pl)
    lons = np.concatenate([np.arange(p, dtype=np.float64) * (360.0 / p) for p in pl])
    return lats, lons


def octahedral(n: int) -> tuple[np.ndarray, np.ndarray]:
    """Octahedral reduced Gaussian grid O{n}: pl = 4i + 16 (i = 1..n) per hemisphere."""
    lat = gaussian_latitudes(n)
    half = 4 * np.arange(1, n + 1) + 16
    pl = np.concatenate([half, half[::-1]])
    return _reduced_grid(lat, pl)


def n320_like() -> tuple[np.ndarray, np.ndarray]:
    """A 640-ring reduced Gaussian grid with N320's point count (542,080).

    The real N320 `pl` table is not available offline; this one follows 1280·cos(lat),
    capped at 1280, and is adjusted ring by ring (from the equator polewards) to the exact
    total, so sizes, density and access pattern match N320.
    """
    n = 320
    target_half = 542_080 // 2
    lat = gaussian_latitudes(n)
    coslat = np.cos(np.deg2rad(lat[:n]))  # northern hemisphere, pole → equator
    lo, hi = 0.5, 2.0
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        pl = np.clip(np.round(mid * 1280.0 * coslat), 18, 1280)
        if pl.sum() < target_half:
            lo = mid
        else:
            hi = mid
    pl = np.clip(np.round(lo * 1280.0 * coslat), 18, 1280).astype(np.int64)
    deficit = int(target_half - pl.sum())
    i = n - 1
    while deficit != 0:
        step = 1 if deficit > 0 else -1
        if 18 <= pl[i] + step <= 1280:
            pl[i] += step
            deficit -= step
        i = i - 1 if i > 0 else n - 1
    pl = np.concatenate([pl, pl[::-1]])
    assert pl.sum() == 542_080
    return _reduced_grid(lat, pl)


def rotated_lam(n_lat: int, n_lon: int, spacing_deg: float, centre_lat: float = 60.0, centre_lon: float = 10.0):
    """A regular grid in rotated-pole coordinates centred on (centre_lat, centre_lon)."""
    rlat = (np.arange(n_lat, dtype=np.float64) - (n_lat - 1) / 2.0) * spacing_deg
    rlon = (np.arange(n_lon, dtype=np.float64) - (n_lon - 1) / 2.0) * spacing_deg
    rlat2, rlon2 = np.meshgrid(rlat, rlon, indexing="ij")
    phi, lam = np.deg2rad(rlat2.ravel()), np.deg2rad(rlon2.ravel())
    x, y, z = np.cos(phi) * np.cos(lam), np.cos(phi) * np.sin(lam), np.sin(phi)
    a = np.deg2rad(centre_lat)
    x2 = np.cos(a) * x - np.sin(a) * z
    z2 = np.sin(a) * x + np.cos(a) * z
    b = np.deg2rad(centre_lon)
    x3 = np.cos(b) * x2 - np.sin(b) * y
    y3 = np.sin(b) * x2 + np.cos(b) * y
    lats = np.rad2deg(np.arcsin(np.clip(z2, -1.0, 1.0)))
    lons = np.rad2deg(np.arctan2(y3, x3)) % 360.0
    return lats, lons


HEALPIX_MAX_PIXELS = 2**31 - 1
_JRLL = np.array([2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4], dtype=np.int64)
_JPLL = np.array([1, 3, 5, 7, 0, 2, 4, 6, 1, 3, 5, 7], dtype=np.int64)


def check_healpix(nside: int, ordering: str = "ring") -> int:
    """nside as an int; ValueError for an unknown ordering, a nested non-power-of-two nside or
    more than 2**31 - 1 pixels."""
    if ordering not in ("ring", "nested"):
        raise ValueError(f"HEALPix ordering {ordering!r} is not 'ring' or 'nested'")
    n = int(nside)
    if n < 1 or 12 * n * n > HEALPIX_MAX_PIXELS:
        raise ValueError(f"HEALPix nside {nside} is not in 1 .. 13376 (12·nside² pixels must fit int32)")
    if ordering == "nested" and n & (n - 1):
        raise ValueError(f"nested HEALPix order needs a power-of-two nside, not {nside}")
    return n


def _isqrt(v: np.ndarray) -> np.ndarray:
    r = np.floor(np.sqrt(v.astype(np.float64))).astype(np.int64)
    r -= r * r > v
    r += (r + 1) * (r + 1) <= v
    return r


def healpix_ring_of(nside: int, pix: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Ring-order pixels → (ring i in 1 .. 4·nside - 1, position p in the ring), int64."""
    n, pix = int(nside), np.asarray(pix, dtype=np.int64)
    ncap, npix = 2 * n * (n - 1), 12 * n * n
    i, p = np.empty_like(pix), np.empty_like(pix)
    north, south = pix < ncap, pix >= npix - ncap
    eq = ~north & ~south
    i[north] = (1 + _isqrt(1 + 2 * pix[north])) >> 1
    p[north] = pix[north] - 2 * i[north] * (i[north] - 1)
    q = pix[eq] - ncap
    i[eq], p[eq] = q // (4 * n) + n, q % (4 * n)
    q = npix - pix[south]
    ir = (1 + _isqrt(2 * q - 1)) >> 1
    i[south], p[south] = 4 * n - ir, 4 * ir - (q - 2 * ir * (ir - 1))
    return i, p


def _spread(v: np.ndarray) -> np.ndarray:
    out = np.zeros_like(v)
    for b in range(31):
        out |= ((v >> b) & 1) << (2 * b)
    return out


def _compress(v: np.ndarray) -> np.ndarray:
    out = np.zeros_like(v)
    for b in range(31):
        out |= ((v >> (2 * b)) & 1) << b
    return out


def healpix_nest2ring(nside: int, pix) -> np.ndarray:
    """Nested-order pixel indices → ring order (power-of-two nside), int64."""
    n, pix = int(nside), np.asarray(pix, dtype=np.int64)
    face, ipf = pix // (n * n), pix % (n * n)
    ix, iy = _compress(ipf), _compress(ipf >> 1)
    jr = _JRLL[face] * n - ix - iy - 1
    north, south = jr < n, jr > 3 * n
    nr = np.where(north, jr, np.where(south, 4 * n - jr, n))
    start = np.where(north, 2 * jr * (jr - 1), np.where(south, 12 * n * n - 2 * nr * (nr + 1), 2 * n * (n - 1) + (jr - n) * 4 * n))
    kshift = np.where(north | south, 0, (jr - n) & 1)
    jp = (_JPLL[face] * nr + ix - iy + 1 + kshift) // 2
    jp = np.where(jp > 4 * nr, jp - 4 * nr, jp)
    jp = np.where(jp < 1, jp + 4 * nr, jp)
    return start + jp - 1


def healpix_ring2nest(nside: int, pix) -> np.ndarray:
    """Ring-order pixel indices → nested order (power-of-two nside), int64."""
    n = int(nside)
    i, p = healpix_ring_of(n, pix)
    iphi = p + 1
    north, south = i < n, i > 3 * n
    nr = np.where(north, i, np.where(south, 4 * n - i, n))
    tmp = i - n
    ifm = (iphi - ((tmp + 1) >> 1) + n - 1) // n
    ifp = (iphi - ((2 * n + 1 - tmp) >> 1) + n - 1) // n
    face_eq = np.where(ifp == ifm, ifp | 4, np.where(ifp < ifm, ifp, ifm + 8))
    face = np.where(north, (iphi - 1) // np.maximum(nr, 1), np.where(south, (iphi - 1) // np.maximum(nr, 1) + 8, face_eq))
    kshift = np.where(north | south, 0, (i + n) & 1)
    irt = i - (2 + (face >> 2)) * n + 1
    ipt = 2 * iphi - _JPLL[face] * nr - kshift - 1
    ipt = np.where(ipt >= 2 * n, ipt - 8 * n, ipt)
    ix, iy = (ipt - irt) >> 1, (-ipt - irt) >> 1
    return face * n * n + _spread(ix) + (_spread(iy) << 1)


def healpix(nside: int, ordering: str = "ring") -> tuple[np.ndarray, np.ndarray]:
    """HEALPix pixel centres (latitudes, longitudes in [0, 360), degrees, float64) at `nside`,
    Górski et al. 2005 (ApJ 622, 759) eqs. 4-9.  Ring order runs north → south over
    4·nside - 1 rings, the first pixel of ring 1 at 45° and that of an equatorial ring at 0° or
    half a pixel east of it, as the HEALPix library numbers them; nested order is face·nside² + the bit
    interleave of (ix, iy) within the base face (nside a power of two)."""
    n = check_healpix(nside, ordering)
    i, p = healpix_ring_of(n, np.arange(12 * n * n, dtype=np.int64))
    cap = (i < n) | (i > 3 * n)
    ir = np.where(i < n, i, 4 * n - i)
    z = np.where(cap, 1.0 - ir.astype(np.float64) ** 2 / (3.0 * n * n), 4.0 / 3.0 - 2.0 * i / (3.0 * n))
    z = np.where(i > 3 * n, -z, z)
    s = (i - n + 1) & 1
    lon = np.where(cap, (p + 0.5) * 90.0 / np.maximum(ir, 1), (p + s / 2.0) * 90.0 / n)
    lat = np.rad2deg(np.arcsin(z))
    if ordering == "nested":
        ring = healpix_nest2ring(n, np.arange(12 * n * n, dtype=np.int64))
        lat, lon = lat[ring], lon[ring]
    return lat, lon


# --------------------------------------------------------------------------- matrices ---
def bilinear_matrix(step: float, tgt_lat: np.ndarray, tgt_lon: np.ndarray):
    """4-point bilinear CSR matrix from the `regular_latlon(step)` grid to the target points.

    Returns (data float32[4n], indices int32[4n], indptr int32[n+1], shape).  Every row has
    four stored entries sorted by column; weights that are exactly zero (a target on a source
    line) are kept as explicit zeros, as they propagate NaN like scipy's csr_matvec does.
    """
    nlat = int(round(180.0 / step)) + 1
    nlon = int(round(360.0 / step))
    n = tgt_lat.shape[0]
    fy = (90.0 - tgt_lat) / step
    j = np.clip(np.floor(fy).astype(np.int64), 0, nlat - 2)
    wy = fy - j
    fx = (tgt_lon % 360.0) / step
    i0 = np.floor(fx).astype(np.int64)
    wx = fx - i0
    i0 %= nlon
    i1 = (i0 + 1) % nlon
    cols = np.stack([j * nlon + i0, j * nlon + i1, (j + 1) * nlon + i0, (j + 1) * nlon + i1], axis=1)
    w = np.stack([(1 - wy) * (1 - wx), (1 - wy) * wx, wy * (1 - wx), wy * wx], axis=1)
    order = np.argsort(cols, axis=1, kind="stable")
    cols = np.take_along_axis(cols, order, axis=1)
    w = np.take_along_axis(w, order, axis=1)
    indptr = (4 * np.arange(n + 1)).astype(np.int32)
    return w.astype(np.float32).ravel(), cols.astype(np.int32).ravel(), indptr, (n, nlat * nlon)


def knn_matrix(idx: np.ndarray, dist: np.ndarray, n_src: int):
    """k-nearest inverse-distance matrix from neighbour indices / distances [n, k]."""
    n, k = idx.shape
    w = 1.0 / np.maximum(dist, 1e-12)
    w /= w.sum(axis=1, keepdims=True)
    order = np.argsort(idx, axis=1, kind="stable")
    cols = np.take_along_axis(idx, order, axis=1)
    w = np.take_along_axis(w, order, axis=1)
    indptr = (k * np.arange(n + 1)).astype(np.int32)
    return w.astype(np.float32).ravel(), cols.astype(np.int32).ravel(), indptr, (n, n_src)


def save_regrid_npz(path, data, indices, indptr, shape, in_lat, in_lon, out_lat, out_lon) -> None:
    """Write the regrid file schema of make-regrid-file.py:150-160."""
    np.savez(
        path,
        matrix_data=data,
        matrix_indices=indices,
        matrix_indptr=indptr,
        matrix_shape=np.asarray(shape),
        in_latitudes=in_lat,
        in_longitudes=in_lon,
        out_latitudes=out_lat,
        out_longitudes=out_lon,
    )


# ----------------------------------------------------------------------------- fields ---
PRESSURE_LEVELS = (50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000)


def synthetic_field(param: str, n_points: int, seed: int, nan_fraction: float = 0.0) -> np.ndarray:
    """One seeded float32 field with the value range of `param`."""
    rng = np.random.default_rng(seed)
    if param == "t":
        v = rng.normal(280.0, 15.0, n_points)
    elif param in ("u", "v"):
        v = rng.normal(0.0, 8.0, n_points)
    elif param == "q":
        v = rng.uniform(1e-5, 2e-2, n_points)
    elif param == "lsm":
        v = (rng.uniform(0.0, 1.0, n_points) > 0.7).astype(np.float64)
    else:
        v = rng.normal(0.0, 1.0, n_points)
    v = v.astype(np.float32)
    if nan_fraction > 0:
        v[rng.uniform(size=n_points) < nan_fraction] = np.nan
    return v


def field_specs(n_vars: int = 10, levels=PRESSURE_LEVELS, n_steps: int = 24):
    """(param, level, step) for the 10 vars × 13 levels × 24 steps = 3120-field workload."""
    params = ["t", "u", "v", "q", "z", "w", "r", "d", "vo", "o3"][:n_vars]
    return [(p, lev, s) for s in range(n_steps) for lev in levels for p in params]
