"""Oracle: pixel-exact conservative matrices between HEALPix and structured grids.

TEST INFRASTRUCTURE — see oracle/__init__.py.

The `method="healpix-conservative"` recipe builds its matrix on the device
(`at_healpix_conservative_count` / `_fill`).  Neither MIR's nor atlas's HEALPix weights can be
obtained offline, so parity with them is unpinned.  This module restates the device builder in
plain Python floats with the device's float64 operation order — `row` is what the device is
checked against, bit for bit — and tests/test_oracle_healpix.py pins it by its defining
properties (rows sum to 1, the area integral is kept in both directions, nested HEALPix grids
take exactly their sub-pixels) and by a Monte-Carlo estimate of the overlaps that classifies
random points with `oracle.healpix.ang2pix_ring` and a box search, independent of the plane.

A grid is ("healpix", nside, ordering) or ("boxes", zn, zs, lon0, first, count) with the rows
of `oracle.conservative_matrix.box_tables` (north → south for a source, storage order for a
target).  Weight of source s in target t = area(s ∩ t) / area(t) in the plane of
oracle/healpix.py: area(t) = 2 / n² for a pixel and 12 dz / count for a box.
"""

from __future__ import annotations

import math

import numpy as np

from . import healpix as hp
from .conservative_matrix import box_tables
from .structured_matrix import check_global, structured_rows


def healpix_grid(nside: int, ordering: str = "ring"):
    return ("healpix", int(nside), ordering)


def box_grid(lat, lon, target: bool):
    rows = structured_rows(lat, lon)
    if rows is None:
        raise ValueError("grid is not a structured grid")
    check_global(rows)
    zn, zs = box_tables(rows)
    t = (zn, zs, rows[1], rows[2], rows[3])
    if target and t[3][0] > t[3][-1]:
        t = tuple(a[::-1].copy() for a in t)
    return ("boxes", *t)


def npoints(grid) -> int:
    return 12 * grid[1] ** 2 if grid[0] == "healpix" else int(np.sum(grid[5]))


def _np_mod(a: float, b: float) -> float:
    return float(np.mod(a, b))


def _runs(pa: int, pb: int, count: int):
    """(c, p') pairs of the unwrapped range [pa, pb], columns ascending (wrapped run first)."""
    if pb < pa:
        return
    length, a = pb - pa + 1, pa % count

    def one(c):
        pp = pa + (c - a) % count
        while pp <= pb:
            yield c, pp
            pp += count

    if length >= count:
        for c in range(count):
            yield from one(c)
        return
    for c in range(0, a + length - count):
        yield from one(c)
    for c in range(a, min(count, a + length)):
        yield from one(c)


def row(src, tgt, t: int):
    """Target t's entries → [(column, float64 weight)], in the device's emission order
    (ring-order columns for a HEALPix source, whatever its ordering)."""
    out = []
    if tgt[0] == "healpix":
        tn = tgt[1]
        r = int(hp.nest2ring(tn, [t])[0]) if tgt[2] == "nested" else t
        ti, tp = hp.ring_of(tn, r)
        nd = float(tn)
        ox = float(hp.xnum(tn, ti, tp)) / nd
        oy = float(2 * tn - ti) / nd
        ya, yb = oy - 1.0 / nd, oy + 1.0 / nd
        area_t = 2.0 / (nd * nd)
        pieces = [hp.diamond(tn, ti, tp, ox, oy)]
    else:
        zn, zs, lon0, first, count = tgt[1:]
        r = int(np.searchsorted(first, t, side="right")) - 1
        cnt = float(count[r])
        d = 360.0 / cnt
        start = float(lon0[r]) + (float(t - first[r]) - 0.5) * d
        fa, fb = start / 45.0, (start + d) / 45.0
        ya, yb = hp.y_of_z(float(zs[r])), hp.y_of_z(float(zn[r]))
        ox, oy = 0.5 * (fa + fb), 0.5 * (ya + yb)
        area_t = 12.0 * (float(zn[r]) - float(zs[r])) / cnt
        pieces = hp.box_pieces(ya, yb, fa, fb, ox, oy)

    if src[0] == "healpix":
        n = src[1]
        nd = float(n)
        h = 1.0 / nd
        area_s = 2.0 / (nd * nd)
        keep = 1e-9 * (area_s if area_s < area_t else area_t)
        i0 = max(1, math.floor((2.0 - yb) * nd))
        i1 = min(4 * n - 1, math.ceil((2.0 - ya) * nd))
        for i in range(i0, i1 + 1):
            yc = float(2 * n - i) / nd
            xlo = xhi = 0.0
            anyp = False
            for q in pieces:
                ys = [v[1] for v in q]
                xs = [v[0] for v in q]
                qlo, qhi, plo, phi = min(ys), max(ys), min(xs), max(xs)
                if not (qlo + oy < yc + h and qhi + oy > yc - h):
                    continue
                plo, phi = plo + ox, phi + ox
                xlo = plo if (not anyp or plo < xlo) else xlo
                xhi = phi if (not anyp or phi > xhi) else xhi
                anyp = True
            if not anyp:
                continue
            ir = hp.ring_size(n, i)
            if i < n or i > 3 * n:
                ka, kb = math.floor(xlo / 2.0), math.floor(xhi / 2.0)
                ja = math.floor(((xlo - 2.0 * float(ka) - 1.0) * nd + float(ir) - 2.0) / 2.0)
                jb = math.ceil(((xhi - 2.0 * float(kb) - 1.0) * nd + float(ir)) / 2.0)
                ja = min(max(ja, 0), ir)
                jb = min(max(jb, -1), ir - 1)
                pa, pb, cnt_i = ka * ir + ja, kb * ir + jb, 4 * ir
            else:
                s = float((i - n + 1) & 1)
                pa = math.floor((xlo * nd - 1.0 - s) / 2.0)
                pb = math.ceil((xhi * nd + 1.0 - s) / 2.0)
                cnt_i = 4 * n
            base = hp.ring_start(n, i)
            col, acc = -1, 0.0
            for c, pp in _runs(pa, pb, cnt_i):
                if c != col:
                    if col >= 0 and acc >= keep:
                        out.append((base + col, acc / area_t))
                    col, acc = c, 0.0
                dia = hp.diamond(n, i, pp, ox, oy)
                for q in pieces:
                    acc = acc + hp.clip_area(dia, q)
            if col >= 0 and acc >= keep:
                out.append((base + col, acc / area_t))
        return out

    # structured source, HEALPix target
    nd = float(tgt[1])
    h = 1.0 / nd
    xf = 2.0 * math.floor(ox / 2.0) + 1.0
    plo = phi = 0.0
    for v in range(4):
        vx = ox + (h if v == 1 else (-h if v == 3 else 0.0))
        vy = oy + (-h if v == 0 else (h if v == 2 else 0.0))
        if abs(vy) <= 1.0:
            lo_v = hi_v = vx
        else:
            s = 2.0 - abs(vy)
            if s == 0.0:
                lo_v, hi_v = xf - 1.0, xf + 1.0
            else:
                lo_v = hi_v = xf + (vx - xf) / s
        plo = lo_v if (v == 0 or lo_v < plo) else plo
        phi = hi_v if (v == 0 or hi_v > phi) else phi
    zn, zs, lon0, first, count = src[1:]
    zlo, zhi = hp.z_of_y(ya), hp.z_of_y(yb)
    k0 = int(np.sum(zs >= zhi))  # edges descend
    k1 = int(np.sum(zn > zlo)) - 1
    order = range(k0, k1 + 1) if first[0] < first[-1] else range(k1, k0 - 1, -1)
    start, width = plo * 45.0, (phi - plo) * 45.0
    dia = pieces[0]
    for k in order:
        n = int(count[k])
        cnt = float(n)
        d = 360.0 / cnt
        x = _np_mod(start - (float(lon0[k]) - d / 2.0), 360.0) / d
        if x >= cnt:
            x = x - cnt
        shift = start - x * d
        ca = math.floor(x)
        cb = math.ceil(x + width / d) - 1
        by0, by1 = hp.y_of_z(float(zs[k])), hp.y_of_z(float(zn[k]))
        area_s = 12.0 * (float(zn[k]) - float(zs[k])) / cnt
        keep = 1e-9 * (area_s if area_s < area_t else area_t)
        col, acc = -1, 0.0
        for c, cc in _runs(ca, cb, n):
            if c != col:
                if col >= 0 and acc >= keep:
                    out.append((int(first[k]) + col, acc / area_t))
                col, acc = c, 0.0
            ga = (shift + float(cc) * d) / 45.0
            gb = (shift + float(cc + 1) * d) / 45.0
            for b in hp.box_pieces(by0, by1, ga, gb, ox, oy):
                acc = acc + hp.clip_area(b, dia)
        if col >= 0 and acc >= keep:
            out.append((int(first[k]) + col, acc / area_t))
    return out


def matrix(src, tgt, rows=None, weights_dtype=np.float32):
    """The matrix (or only the target rows `rows`, in that order) → (data, indices int32,
    indptr int32, shape): columns of a nested source mapped and each row sorted by column."""
    n_tgt = npoints(tgt)
    rows = range(n_tgt) if rows is None else rows
    nested = src[0] == "healpix" and src[2] == "nested"
    inv = hp.ring2nest(src[1], np.arange(12 * src[1] ** 2)) if nested else None
    cols, ws, indptr = [], [], [0]
    for t in rows:
        e = row(src, tgt, int(t))
        c = np.array([x[0] for x in e], dtype=np.int64)
        w = np.array([x[1] for x in e], dtype=np.float64)
        if nested:
            c = inv[c]
            o = np.argsort(c, kind="stable")
            c, w = c[o], w[o]
        cols.append(c)
        ws.append(w)
        indptr.append(indptr[-1] + c.size)
    data = np.concatenate(ws) if ws else np.zeros(0)
    return data.astype(weights_dtype), np.concatenate(cols).astype(np.int32), np.array(indptr, dtype=np.int32), (n_tgt, npoints(src))
