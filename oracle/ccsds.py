"""Oracle: CCSDS 121.0-B adaptive entropy coding (AEC) as GRIB2 template 5.42 uses it — numpy.

TEST INFRASTRUCTURE — see oracle/__init__.py.

GRIB2 data representation template 5.42 (`packingType=grid_ccsds`) stores the same unsigned
integers X as simple packing (template 5.0), coded as one AEC bitstream in section 7.  ECMWF
writes it with libaec.  Neither libaec nor ecCodes is installed here, so this module restates
the coding from the standard (CCSDS 121.0-B, Lossless Data Compression) with libaec's
conventions for the option-ID lengths, the reference sample and the padding:

* A stream is blocks of J samples; `rsi` blocks form a reference sample interval (RSI).
* Option ID: 3 bits for n <= 8, 4 for n <= 16, 5 otherwise.  All zeros: low entropy, one more
  bit selects zero-block (0) or second extension (1).  1 .. 2^len - 2: split-sample with
  k = ID - 1.  All ones: no compression.
* With AEC_DATA_PREPROCESS the first block of every RSI carries a reference sample (n bits,
  right after the full option ID), and the other samples are the unit-delay predictor's
  mapped differences δ (`postprocess` inverts the mapping).
* Zero-block: one fundamental-sequence (FS) code m, z = m + 1; z == 5 ("remainder of segment")
  runs to the end of the RSI or of the current 64-block segment, whichever comes first; z > 5
  means z - 1 blocks.
* Second extension: J/2 FS codes, pair (a, b) coded as m = (a+b)(a+b+1)/2 + b; the first pair of
  a reference block carries only b.
* AEC_PAD_RSI: after each RSI the stream continues at the next octet.
* Flags 2 (AEC_DATA_3BYTE) and 4 (AEC_DATA_MSB) describe libaec's in-memory sample layout and
  do not change the stream.

PARITY UNPINNED: libaec cannot be run here.  Two bitstreams derived by hand from the standard
(tests/test_oracle_ccsds.py) tie this restatement to it; the encoder and the decoder are then
checked against each other over the parameter grid.
"""

from __future__ import annotations

import numpy as np

AEC_DATA_SIGNED = 1
AEC_DATA_3BYTE = 2
AEC_DATA_MSB = 4
AEC_DATA_PREPROCESS = 8
AEC_RESTRICTED = 16
AEC_PAD_RSI = 32

ROS = 5  # zero-block code z meaning "remainder of segment"
SEGMENT = 64  # blocks of a segment


def id_length(n: int) -> int:
    return 5 if n > 16 else 4 if n > 8 else 3


def check_parameters(n: int, J: int, rsi: int, flags: int) -> None:
    if flags & AEC_DATA_SIGNED:
        raise NotImplementedError("signed AEC samples")
    if flags & AEC_RESTRICTED and n <= 4:
        raise NotImplementedError("restricted AEC option set")
    if J not in (8, 16, 32, 64):
        raise NotImplementedError(f"AEC block size {J}")
    if not 1 <= rsi <= 4096:
        raise NotImplementedError(f"AEC reference sample interval {rsi}")
    if not 0 <= n <= 32:
        raise NotImplementedError(f"{n} bits per sample")


# ------------------------------------------------------------------ predictor mapping -----
def preprocess(x: np.ndarray, n: int, J: int, rsi: int) -> np.ndarray:
    """X → δ: the unit-delay predictor's mapped differences; the first sample of every RSI
    (the reference) is left as 0 in δ."""
    x = x.astype(np.int64)
    xmax = (1 << n) - 1
    d = np.zeros_like(x)
    if x.size > 1:
        prev, cur = x[:-1], x[1:]
        theta = np.minimum(prev, xmax - prev)
        delta = cur - prev
        d[1:] = np.where((delta >= 0) & (delta <= theta), 2 * delta, np.where((delta < 0) & (-delta <= theta), 2 * (-delta) - 1, theta + np.abs(delta)))
    d[:: rsi * J] = 0
    return d


def postprocess_one(delta: int, prev: int, xmax: int) -> int:
    theta = min(prev, xmax - prev)
    if delta <= 2 * theta:
        return prev + delta // 2 if delta % 2 == 0 else prev - (delta + 1) // 2
    return delta if prev <= xmax - prev else xmax - delta


# ------------------------------------------------------------------ decoder ---------------
class _Bits:
    def __init__(self, stream: bytes):
        self.bits = np.unpackbits(np.frombuffer(bytes(stream), dtype=np.uint8))
        self.ones = np.flatnonzero(self.bits)
        self.pos = 0

    def read(self, w: int) -> int:
        if w == 0:
            return 0
        if self.pos + w > self.bits.size:
            raise ValueError("AEC stream ends early")
        v = 0
        for b in self.bits[self.pos : self.pos + w]:
            v = (v << 1) | int(b)
        self.pos += w
        return v

    def read_many(self, count: int, w: int) -> np.ndarray:
        if w == 0 or count == 0:
            return np.zeros(count, dtype=np.int64)
        end = self.pos + count * w
        if end > self.bits.size:
            raise ValueError("AEC stream ends early")
        b = self.bits[self.pos : end].reshape(count, w).astype(np.int64)
        self.pos = end
        return (b << np.arange(w - 1, -1, -1, dtype=np.int64)).sum(axis=1)

    def fs(self, count: int) -> np.ndarray:
        """`count` fundamental-sequence codes: m zeros then a one."""
        if count == 0:
            return np.zeros(0, dtype=np.int64)
        i = int(np.searchsorted(self.ones, self.pos))
        if i + count > self.ones.size:
            raise ValueError("AEC stream ends inside a fundamental sequence")
        ends = self.ones[i : i + count].astype(np.int64)
        starts = np.concatenate(([self.pos], ends[:-1] + 1))
        self.pos = int(ends[-1]) + 1
        return ends - starts


def aec_decode(stream: bytes, n: int, J: int, rsi: int, flags: int, n_values: int) -> np.ndarray:
    """The n_values unsigned samples X (uint64) of one AEC stream."""
    check_parameters(n, J, rsi, flags)
    out = np.zeros(n_values, dtype=np.uint64)
    if n == 0 or n_values == 0:
        return out
    pre = bool(flags & AEC_DATA_PREPROCESS)
    xmax = (1 << n) - 1
    idlen = id_length(n)
    r = _Bits(stream)
    n_blocks = -(-n_values // J)
    samples = np.zeros(n_blocks * J, dtype=np.int64)  # δ (or X without PREPROCESS)
    refs = {}
    blk = 0
    while blk < n_blocks:
        if blk % rsi == 0 and blk > 0 and flags & AEC_PAD_RSI:
            r.pos = -(-r.pos // 8) * 8
        b = blk % rsi
        ref = pre and b == 0
        ident = r.read(idlen)
        nref = 1 if ref else 0
        s = samples[blk * J : (blk + 1) * J]
        if ident == 0:
            selector = r.read(1)
            if ref:
                refs[blk] = r.read(n)
            if selector == 0:
                z = int(r.fs(1)[0]) + 1
                run = min(rsi - b, SEGMENT - b % SEGMENT) if z == ROS else z - 1 if z > ROS else z
                if b + run > rsi:
                    raise ValueError("AEC zero-block run leaves its RSI")
                blk += run  # samples are already 0
                continue
            m = r.fs(J // 2)
            sq = np.floor((np.sqrt(8.0 * m + 1.0) - 1.0) / 2.0).astype(np.int64)
            sq -= (sq * (sq + 1) // 2 > m).astype(np.int64)  # guard the float estimate
            sq += ((sq + 1) * (sq + 2) // 2 <= m).astype(np.int64)
            bb = m - sq * (sq + 1) // 2
            aa = sq - bb
            pairs = np.stack([aa, bb], axis=1).reshape(-1)
            s[nref:] = pairs[nref:]
        elif ident == (1 << idlen) - 1:
            v = r.read_many(J, n)
            if ref:
                refs[blk] = int(v[0])
            s[nref:] = v[nref:]
        else:
            k = ident - 1
            if k >= n:
                raise ValueError(f"AEC option k = {k} for {n}-bit samples")
            if ref:
                refs[blk] = r.read(n)
            fs = r.fs(J - nref)
            lsb = r.read_many(J - nref, k)
            s[nref:] = (fs << k) | lsb
        blk += 1
    if (samples > xmax).any():
        raise ValueError("AEC sample out of range")
    samples = samples[:n_values]
    if not pre:
        return samples.astype(np.uint64)
    x = np.zeros(n_values, dtype=np.int64)
    prev = 0
    for i in range(n_values):
        if i % (rsi * J) == 0:
            prev = refs[i // J]
        else:
            prev = postprocess_one(int(samples[i]), prev, xmax)
        x[i] = prev
    return x.astype(np.uint64)


# ------------------------------------------------------------------ encoder ---------------
def _se_codes(pairs_a: np.ndarray, pairs_b: np.ndarray) -> np.ndarray:
    s = pairs_a + pairs_b
    return s * (s + 1) // 2 + pairs_b


def aec_encode(X, n: int, J: int, rsi: int, flags: int, option=None, pad: str = "block") -> bytes:
    """One AEC stream of the unsigned samples X.

    option None: per block the cheapest option, as libaec chooses (all-zero blocks become
    zero-block runs).  Otherwise every block that is not all zero is coded with `option`: an
    int k (split-sample), "se" (second extension) or "uncompressed".
    pad "block": the last block is filled with the last sample; "rsi": the last RSI is filled
    with blocks of the last sample too.  Both are what libaec may write."""
    check_parameters(n, J, rsi, flags)
    x = np.asarray(X, dtype=np.int64).reshape(-1)
    if n == 0 or x.size == 0:
        return b""
    xmax = (1 << n) - 1
    if x.min() < 0 or x.max() > xmax:
        raise ValueError("sample out of range")
    pre = bool(flags & AEC_DATA_PREPROCESS)
    idlen = id_length(n)
    n_blocks = -(-x.size // J)
    if pad == "rsi":
        n_blocks = -(-n_blocks // rsi) * rsi
    elif pad != "block":
        raise ValueError(pad)
    x = np.concatenate([x, np.full(n_blocks * J - x.size, x[-1], dtype=np.int64)])
    d = preprocess(x, n, J, rsi) if pre else x.copy()
    D = d.reshape(n_blocks, J)
    blocks = np.arange(n_blocks)
    b_in_rsi = blocks % rsi
    is_ref = (b_in_rsi == 0) & pre
    nref = is_ref.astype(np.int64)
    zero = (D == 0).all(axis=1)
    kmax = min((1 << idlen) - 3, n - 1)
    # costs in bits beyond the ID and the reference, per block
    ks = np.arange(kmax + 1)
    split_cost = np.stack([(D >> k).sum(axis=1) + (J - nref) * (k + 1) for k in ks], axis=1).astype(np.float64)
    Df = D.astype(np.float64)
    a, b = Df[:, 0::2], Df[:, 1::2]
    se_cost = ((a + b) * (a + b + 1) / 2 + b + 1).sum(axis=1) + 1
    unc_cost = ((J - nref) * n).astype(np.float64)
    if option is None:
        best_k = split_cost.argmin(axis=1)
        best_split = split_cost[blocks, best_k]
        kind = np.where(se_cost < np.minimum(best_split, unc_cost), 1, np.where(best_split < unc_cost, 2, 3))
        kk = best_k
    else:
        if option == "se":
            kind = np.full(n_blocks, 1)
        elif option == "uncompressed":
            kind = np.full(n_blocks, 3)
        else:
            k = int(option)
            if not 0 <= k <= kmax:
                raise ValueError(f"split option k = {k} for {n}-bit samples")
            kind = np.full(n_blocks, 2)
        kk = np.full(n_blocks, int(option) if kind[0] == 2 else 0)
    kind = np.where(zero, 0, kind)  # 0 zero, 1 SE, 2 split, 3 uncompressed

    # fields (value, width, key): key orders them block by block
    K = 2 * J + 4
    vals, wids, keys = [], [], []

    def emit(v, w, blk, local):
        vals.append(np.asarray(v, dtype=np.int64).reshape(-1))
        wids.append(np.broadcast_to(np.asarray(w, dtype=np.int64), np.shape(v)).reshape(-1))
        keys.append((np.asarray(blk, dtype=np.int64) * K + local).reshape(-1))

    # zero-block runs: consecutive zero blocks inside an RSI, cut at 64-block segments
    zb = np.flatnonzero(kind == 0)
    run_first = np.zeros(n_blocks, dtype=bool)
    if zb.size:
        starts = [zb[0]]
        for p, q in zip(zb[:-1], zb[1:]):
            if q != p + 1 or q % rsi == 0 or (q % rsi) % SEGMENT == 0:
                starts.append(q)
        starts = np.array(starts)
        ends = np.append(zb[np.searchsorted(zb, starts[1:]) - 1], zb[-1]) + 1  # exclusive
        for s0, e0 in zip(starts, ends):
            r = int(e0 - s0)
            b0 = int(s0 % rsi)
            nominal = min(rsi - b0, SEGMENT - b0 % SEGMENT)
            if r >= ROS and (r == nominal or e0 == n_blocks):
                m = ROS - 1
            else:
                m = r - 1 if r < ROS else r
            run_first[s0] = True
            emit(0, idlen, s0, 0)
            emit(0, 1, s0, 1)
            if is_ref[s0]:
                emit(x[s0 * J], n, s0, 2)
            emit(1, m + 1, s0, 3)
    nz = np.flatnonzero(kind != 0)
    ids = np.where(kind == 1, 0, np.where(kind == 2, kk + 1, (1 << idlen) - 1))
    emit(ids[nz], idlen, nz, 0)
    se = nz[kind[nz] == 1]
    emit(np.ones(se.size), 1, se, 1)
    refb = nz[is_ref[nz]]
    emit(x[refb * J], n, refb, 2)
    if se.size:
        m = _se_codes(D[se][:, 0::2], D[se][:, 1::2])
        emit(np.ones(m.shape), m + 1, np.repeat(se, J // 2), 3 + np.tile(np.arange(J // 2), se.size))
    for kind_id in (2, 3):
        sel = nz[kind[nz] == kind_id]
        if not sel.size:
            continue
        j = np.tile(np.arange(J), sel.size)
        bl = np.repeat(sel, J)
        keep = ~(is_ref[bl] & (j == 0))
        dv = D[sel].reshape(-1)[keep]
        bl, j = bl[keep], j[keep]
        if kind_id == 3:
            emit(dv, n, bl, 3 + j)
        else:
            k = kk[bl]
            emit(np.ones(dv.size), (dv >> k) + 1, bl, 3 + j)
            emit(dv & ((1 << k) - 1), k, bl, 3 + J + j)
    v = np.concatenate(vals)
    w = np.concatenate(wids)
    key = np.concatenate(keys)
    order = np.argsort(key, kind="stable")
    v, w, key = v[order], w[order], key[order]
    if flags & AEC_PAD_RSI:
        # every RSI starts on an octet: pad after the last field of each RSI
        rsi_of = key // K // rsi
        last = np.flatnonzero(np.append(rsi_of[1:] != rsi_of[:-1], True))
        totals = np.add.reduceat(w, np.concatenate(([0], last[:-1] + 1)))
        pads = (-totals) % 8
        v = np.insert(v, last + 1, 0)
        w = np.insert(w, last + 1, pads)
    return _pack(v.astype(np.uint64), w)


def _pack(v: np.ndarray, w: np.ndarray) -> bytes:
    total = int(w.sum())
    bits = np.zeros(-(-total // 8) * 8, dtype=np.uint8)
    end = np.cumsum(w)  # one past each field's last bit
    for j in range(33):
        sel = (w > j) & (((v >> np.uint64(j)) & np.uint64(1)) != 0)
        if not sel.any():
            if j > 0 and not (w > j).any():
                break
            continue
        bits[end[sel] - 1 - j] = 1
    return np.packbits(bits).tobytes()


__all__ = [
    "AEC_DATA_3BYTE",
    "AEC_DATA_MSB",
    "AEC_DATA_PREPROCESS",
    "AEC_DATA_SIGNED",
    "AEC_PAD_RSI",
    "AEC_RESTRICTED",
    "aec_decode",
    "aec_encode",
    "check_parameters",
    "id_length",
    "postprocess_one",
    "preprocess",
]
