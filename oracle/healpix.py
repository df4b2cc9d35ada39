"""Oracle: HEALPix grids and the plane of the HEALPix projection.

TEST INFRASTRUCTURE — see oracle/__init__.py.

healpy is not available offline (oracle/refstubs/healpy only lets the reference's tabular
module import); the package generates HEALPix grids itself (`synthetic.healpix`).  This module
restates, in numpy and plain Python:

- `centres`: pixel centres in ring order from Górski et al. 2005 (ApJ 622, 759) eqs. 4-9;
- `ang2pix_ring` / `ang2pix_nest`: the pixel holding a point, from the same paper's
  construction (the two families of edge lines in the equatorial zone, the distance to the
  pole in the caps) — independent of the index arithmetic of `nest2ring` / `ring2nest`, which
  the tests check against it;
- `nest2ring` / `ring2nest`: index conversion through the base face and (ix, iy);
- the plane geometry of Calabretta & Roukema 2007 (MNRAS 381, 865), scaled by 4/π: X =
  longitude / 45° (periodic with 8), Y in [-2, 2].  Pixel p of ring i at nside n is the
  diamond with centre (xnum / n, (2n - i) / n) and half-diagonal 1 / n; a structured box is
  cut at Y = ±1 and at the cap facet meridians into convex pieces.  The device builder's
  geometry (csrc/matrix.cu) is restated operation for operation in `diamond`, `box_pieces`
  and `clip_area`.
"""

from __future__ import annotations

import math

import numpy as np

JRLL = (2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4)
JPLL = (1, 3, 5, 7, 0, 2, 4, 6, 1, 3, 5, 7)


# ------------------------------------------------------------------------- indices ---
def ring_of(n: int, r: int) -> tuple[int, int]:
    """Ring pixel r → (ring i in 1 .. 4n - 1, position p in the ring)."""
    ncap, npix = 2 * n * (n - 1), 12 * n * n
    if r < ncap:
        i = (1 + math.isqrt(1 + 2 * r)) >> 1
        return i, r - 2 * i * (i - 1)
    if r < npix - ncap:
        q = r - ncap
        return q // (4 * n) + n, q % (4 * n)
    q = npix - r
    ir = (1 + math.isqrt(2 * q - 1)) >> 1
    return 4 * n - ir, 4 * ir - (q - 2 * ir * (ir - 1))


def ring_size(n: int, i: int) -> int:
    return i if i < n else (4 * n - i if i > 3 * n else n)


def ring_start(n: int, i: int) -> int:
    if i < n:
        return 2 * i * (i - 1)
    if i <= 3 * n:
        return 2 * n * (n - 1) + (i - n) * 4 * n
    ir = 4 * n - i
    return 12 * n * n - 2 * ir * (ir + 1)


def centres(n: int) -> tuple[np.ndarray, np.ndarray]:
    """(z, φ in radians) of the 12 n² pixels in ring order, Górski eqs. 4-9."""
    z, phi = [], []
    for i in range(1, 4 * n):
        if i < n or i > 3 * n:
            ir = i if i < n else 4 * n - i
            zz = 1.0 - ir * ir / (3.0 * n * n)
            z += [zz if i < n else -zz] * (4 * ir)
            phi += [(j + 0.5) * math.pi / (2 * ir) for j in range(4 * ir)]
        else:
            s = (i - n + 1) % 2  # 1: the ring is shifted by half a pixel
            z += [4.0 / 3.0 - 2.0 * i / (3.0 * n)] * (4 * n)
            phi += [(j + s / 2.0) * math.pi / (2 * n) for j in range(4 * n)]
    return np.array(z), np.array(phi)


def _xyf(n: int, pix: np.ndarray):
    face, ipf = pix // (n * n), pix % (n * n)
    ix, iy = np.zeros_like(pix), np.zeros_like(pix)
    for b in range(31):
        ix |= ((ipf >> (2 * b)) & 1) << b
        iy |= ((ipf >> (2 * b + 1)) & 1) << b
    return face, ix, iy


def _nest(n: int, face, ix, iy):
    out = face * n * n
    for b in range(31):
        out = out | (((ix >> b) & 1) << (2 * b)) | (((iy >> b) & 1) << (2 * b + 1))
    return out


def nest2ring(n: int, pix) -> np.ndarray:
    pix = np.asarray(pix, dtype=np.int64)
    face, ix, iy = _xyf(n, pix)
    jr = np.asarray(JRLL)[face] * n - ix - iy - 1
    out = np.empty_like(pix)
    for k in range(pix.size):
        r = int(jr[k])
        if r < n:
            nr, start, kshift = r, 2 * r * (r - 1), 0
        elif r > 3 * n:
            nr = 4 * n - r
            start, kshift = 12 * n * n - 2 * nr * (nr + 1), 0
        else:
            nr, start, kshift = n, 2 * n * (n - 1) + (r - n) * 4 * n, (r - n) & 1
        jp = (JPLL[int(face[k])] * nr + int(ix[k]) - int(iy[k]) + 1 + kshift) // 2
        if jp > 4 * nr:
            jp -= 4 * nr
        if jp < 1:
            jp += 4 * nr
        out[k] = start + jp - 1
    return out


def ring2nest(n: int, pix) -> np.ndarray:
    """The inverse of `nest2ring`, as a permutation inverse."""
    pix = np.asarray(pix, dtype=np.int64)
    inv = np.empty(12 * n * n, dtype=np.int64)
    inv[nest2ring(n, np.arange(12 * n * n))] = np.arange(12 * n * n)
    return inv[pix]


def ang2pix_ring(n: int, z, phi) -> np.ndarray:
    """Górski's ang2pix in ring order: the edge-line indices jp, jm give the ring and the
    position in the equatorial zone; in the caps, the scaled distance to the pole."""
    z, tt = np.asarray(z, dtype=np.float64), np.mod(np.asarray(phi, dtype=np.float64), 2 * np.pi) / (np.pi / 2)
    out = np.empty(z.shape, dtype=np.int64)
    eq = np.abs(z) <= 2.0 / 3.0
    t1, t2 = n * (0.5 + tt[eq]), n * z[eq] * 0.75
    jp, jm = np.floor(t1 - t2).astype(np.int64), np.floor(t1 + t2).astype(np.int64)
    ir = n + 1 + jp - jm
    kshift = 1 - (ir & 1)
    ip = np.mod((jp + jm - n + kshift + 1) // 2, 4 * n)
    out[eq] = 2 * n * (n - 1) + (ir - 1) * 4 * n + ip
    cap = ~eq
    tp = tt[cap] - np.floor(tt[cap])
    tmp = n * np.sqrt(3.0 * (1.0 - np.abs(z[cap])))
    jp, jm = np.floor(tp * tmp).astype(np.int64), np.floor((1.0 - tp) * tmp).astype(np.int64)
    ir = jp + jm + 1
    ip = np.mod(np.floor(tt[cap] * ir).astype(np.int64), 4 * ir)
    out[cap] = np.where(z[cap] > 0, 2 * ir * (ir - 1) + ip, 12 * n * n - 2 * ir * (ir + 1) + ip)
    return out


def ang2pix_nest(n: int, z, phi) -> np.ndarray:
    """Górski's ang2pix in nested order: the base face and (ix, iy) from the edge lines."""
    z, tt = np.asarray(z, dtype=np.float64), np.mod(np.asarray(phi, dtype=np.float64), 2 * np.pi) / (np.pi / 2)
    face, ix, iy = (np.empty(z.shape, dtype=np.int64) for _ in range(3))
    eq = np.abs(z) <= 2.0 / 3.0
    t1, t2 = n * (0.5 + tt[eq]), n * (z[eq] * 0.75)
    jp, jm = np.floor(t1 - t2).astype(np.int64), np.floor(t1 + t2).astype(np.int64)
    ifp, ifm = jp // n, jm // n
    face[eq] = np.where(ifp == ifm, ifp | 4, np.where(ifp < ifm, ifp, ifm + 8))
    ix[eq], iy[eq] = jm % n, n - (jp % n) - 1
    cap = ~eq
    ntt = np.minimum(np.floor(tt[cap]).astype(np.int64), 3)
    tp = tt[cap] - ntt
    tmp = n * np.sqrt(3.0 * (1.0 - np.abs(z[cap])))
    jp = np.minimum(np.floor(tp * tmp).astype(np.int64), n - 1)
    jm = np.minimum(np.floor((1.0 - tp) * tmp).astype(np.int64), n - 1)
    north = z[cap] >= 0
    face[cap] = np.where(north, ntt, ntt + 8)
    ix[cap] = np.where(north, n - jm - 1, jp)
    iy[cap] = np.where(north, n - jp - 1, jm)
    return _nest(n, face, ix, iy)


# --------------------------------------------------------------------------- plane ---
def xnum(n: int, i: int, pp: int) -> int:
    """X numerator (X = xnum / n) of pixel p' of ring i, p' unwrapped."""
    if i < n or i > 3 * n:
        ir = i if i < n else 4 * n - i
        k = pp // ir
        return (2 * k + 1) * n + 2 * (pp - k * ir) + 1 - ir
    return 2 * pp + ((i - n + 1) & 1)


def y_of_z(z: float) -> float:
    a = abs(z)
    if a <= 2.0 / 3.0:
        return 1.5 * z
    y = 2.0 - math.sqrt(3.0 * (1.0 - a))
    return -y if z < 0.0 else y


def z_of_y(y: float) -> float:
    a = abs(y)
    if a <= 1.0:
        return y / 1.5
    s = 2.0 - a
    z = 1.0 - s * s / 3.0
    return -z if y < 0.0 else z


def diamond(n: int, i: int, pp: int, ox: float, oy: float):
    """Pixel (i, p') at nside n as a counter-clockwise vertex list relative to (ox, oy)."""
    nd = float(n)
    x = float(xnum(n, i, pp)) / nd - ox
    y = float(2 * n - i) / nd - oy
    h = 1.0 / nd
    return [(x, y - h), (x + h, y), (x, y + h), (x - h, y)]


def box_pieces(ya: float, yb: float, fa: float, fb: float, ox: float, oy: float):
    """Convex pieces (counter-clockwise, relative to (ox, oy)) of the box Y in [ya, yb], Φ in
    [fa, fb]: the equatorial rectangle, then the north and south cap pieces facet by facet."""
    out = []
    y0, y1 = (ya if ya > -1.0 else -1.0), (yb if yb < 1.0 else 1.0)
    if y1 > y0:
        out.append([(fa - ox, y0 - oy), (fb - ox, y0 - oy), (fb - ox, y1 - oy), (fa - ox, y1 - oy)])
    for cap in (0, 1):
        c0 = (ya if ya > 1.0 else 1.0) if cap == 0 else ya
        c1 = yb if cap == 0 else (yb if yb < -1.0 else -1.0)
        if not c1 > c0:
            continue
        s0, s1 = 2.0 - abs(c0), 2.0 - abs(c1)
        k = math.floor(fa / 2.0)
        while 2.0 * float(k) < fb:
            e0 = 2.0 * float(k)
            g0, g1 = (fa if fa > e0 else e0), (fb if fb < e0 + 2.0 else e0 + 2.0)
            k += 1
            if not g1 > g0:
                continue
            xc = e0 + 1.0
            t = [(xc + (g0 - xc) * s0 - ox, c0 - oy)]
            if s0 != 0.0:
                t.append((xc + (g1 - xc) * s0 - ox, c0 - oy))
            t.append((xc + (g1 - xc) * s1 - ox, c1 - oy))
            if s1 != 0.0:
                t.append((xc + (g0 - xc) * s1 - ox, c1 - oy))
            out.append(t)
    return out


def clip_area(a, b) -> float:
    """Area of the intersection of convex counter-clockwise polygons a and b: a clipped by
    each edge of b (Sutherland-Hodgman), then the shoelace formula."""
    p = list(a)
    for e in range(len(b)):
        if not p:
            break
        ex, ey = b[e]
        fx, fy = b[(e + 1) % len(b)]
        dx, dy = fx - ex, fy - ey
        q = []
        m = len(p)
        for v in range(m):
            px, py = p[v]
            wx, wy = p[(v + 1) % m]
            sp = dx * (py - ey) - dy * (px - ex)
            sq = dx * (wy - ey) - dy * (wx - ex)
            if sp >= 0.0 and len(q) < 12:
                q.append((px, py))
            if ((sp > 0.0 and sq < 0.0) or (sp < 0.0 and sq > 0.0)) and len(q) < 12:
                t = sp / (sp - sq)
                q.append((px + (wx - px) * t, py + (wy - py) * t))
        p = q
    s = 0.0
    for v in range(len(p)):
        px, py = p[v]
        wx, wy = p[(v + 1) % len(p)]
        s = s + (px * wy - wx * py)
    return 0.5 * s


def shoelace(poly) -> float:
    s = 0.0
    for v in range(len(poly)):
        s = s + (poly[v][0] * poly[(v + 1) % len(poly)][1] - poly[(v + 1) % len(poly)][0] * poly[v][1])
    return 0.5 * s
