"""Oracle: GRIB2 complex packing (data representation templates 5.2 and 5.3) — messages in numpy.

TEST INFRASTRUCTURE — see oracle/__init__.py.

WMO Manual on Codes I.2, FM 92 GRIB edition 2, templates 5.2 ("grid point data - complex
packing") and 5.3 ("complex packing and spatial differencing") with data templates 7.2 / 7.3.
Octets are numbered from the start of section 5:

    12-15 R   16-17 E   18-19 D   20 bits per group reference (may be 0)
    21 type of original values   22 group splitting method   23 missing value management
    24-31 missing value substitutes   32-35 NG, the number of groups
    36 reference for group widths   37 bits for group widths
    38-41 reference for group lengths   42 length increment
    43-46 true length of the last group   47 bits for scaled group lengths
    5.3 only:  48 order of spatial differencing (1 or 2)   49 octets per extra descriptor (ww)

Section 7 holds, in order: (5.3 only) the extra descriptors h1, [h2 for order 2,] gmin, each
ww octets in sign and magnitude; the NG group references; the NG group widths; the NG scaled
group lengths (each of those three parts padded to an octet); then the values of every group
back to back, value i of group g in width_g bits.  Decoding:

    width_g  = width_ref + packed width_g
    length_g = length_ref + increment · scaled length_g   (g < NG - 1; the last group has the
                                                           true last length)
    X_i      = ref_g + packed_i                            (a width-0 group is all ref_g)
    5.3, order 1:  X_0 = h1,  X_n = X_{n-1} + (X_n + gmin)
    5.3, order 2:  X_0 = h1,  X_1 = h2,  X_n = (X_n + gmin) + 2·X_{n-1} - X_{n-2}

in two's-complement int64, and then Y = ((X · 2^E) + R) · 10^-D as for simple packing.  With a
section-6 bitmap, section 5's value count is the number of packed values and the differencing
runs over those.  Only missing value management 0 is restated.

So this module works by conversion, like oracle/grib_ccsds.py: `from_simple` recodes the X of
a simple-packed message as 5.2 or 5.3 (same R, E, D and X), and `to_simple` / `decode` turn a
complex message back into the 5.0 message of the same X and hand it to oracle/grib.py: the
host arithmetic is exactly simple packing's.  `to_simple` writes X in `nbits` bits, by default
in `bits_per_value` bits (octet 20) when they hold every X and otherwise in the fewest bits that
do (at least 1: a 5.2 / 5.3 field is never simple packing's constant field, every value goes
through the formula).  `from_simple` writes octet 20 as at least the simple message's width.  A final X outside
[0, 2^32) cannot be written as simple packing and is refused (ValueError); no encoder that
takes R as the minimum produces one.

PARITY UNPINNED: ecCodes and NCEP's g2lib cannot be run here; hand-derived messages in
tests/test_oracle_grib_complex.py pin this restatement of the regulations.
"""

from __future__ import annotations

import struct

import numpy as np

from . import grib as ogrib
from . import grib_ccsds as ogc

_sections = ogc._sections
_rebuild = ogc._rebuild


def _bit_length(v: int) -> int:
    return int(v).bit_length()


def is_complex(msg: bytes) -> bool:
    if msg[:4] != b"GRIB" or msg[7] != 2:
        return False
    for pos, length, number in _sections(msg):
        if number == 5:
            return length >= 11 and struct.unpack(">H", msg[pos + 9 : pos + 11])[0] in (2, 3)
    return False


def _section5_params(msg: bytes, pos: int, length: int) -> dict:
    o = lambda k: msg[pos + k - 1]  # octet k of the section  # noqa: E731
    be = lambda a, b: int.from_bytes(msg[pos + a - 1 : pos + b], "big")  # octets a..b  # noqa: E731
    (template,) = struct.unpack(">H", msg[pos + 9 : pos + 11])
    need = 47 if template == 2 else 49
    if length < need:
        raise NotImplementedError(f"template 5.{template} section of {length} octets ({need} needed)")
    p = dict(
        n_values=be(6, 9),
        template=template,
        reference_value=float(struct.unpack(">f", msg[pos + 11 : pos + 15])[0]),
        binary_scale=ogrib.from_sign_magnitude16(msg[pos + 15 : pos + 17]),
        decimal_scale=ogrib.from_sign_magnitude16(msg[pos + 17 : pos + 19]),
        bits_per_value=o(20),
        missing_management=o(23),
        complex_groups=be(32, 35),
        complex_width_ref=o(36),
        complex_width_bits=o(37),
        complex_length_ref=be(38, 41),
        complex_length_incr=o(42),
        complex_last_length=be(43, 46),
        complex_length_bits=o(47),
        complex_order=o(48) if template == 3 else 0,
        complex_ww=o(49) if template == 3 else 0,
    )
    if p["missing_management"] != 0:
        raise NotImplementedError(f"missing value management {p['missing_management']}")
    if template == 3 and p["complex_order"] not in (1, 2):
        raise NotImplementedError(f"spatial differencing of order {p['complex_order']}")
    if template == 3 and not 1 <= p["complex_ww"] <= 4:
        raise NotImplementedError(f"{p['complex_ww']} octets per extra descriptor")
    return p


def scan(msg: bytes) -> dict:
    """`oracle.grib_ccsds.scan` (packing, CCSDS parameters) plus the complex-packing parameters
    `at_grib_scan` reports (all 0 for other packings): packing 2, NG, references, bit counts,
    order, ww and the octet offsets of the four parts inside section 7."""
    zero = dict(
        complex_groups=0,
        complex_length_ref=0,
        complex_last_length=0,
        complex_width_ref=0,
        complex_width_bits=0,
        complex_length_incr=0,
        complex_length_bits=0,
        complex_order=0,
        complex_ww=0,
        complex_refs_offset=0,
        complex_widths_offset=0,
        complex_lengths_offset=0,
        complex_values_offset=0,
    )
    if not is_complex(msg):
        info = ogc.scan(msg)
        info.update(zero)
        return info
    (total,) = struct.unpack(">Q", msg[8:16])
    info = dict(edition=2, bitmap_offset=-1, has_bitmap=0, message_length=total, packing=2, ccsds_flags=0, ccsds_block_size=0, ccsds_rsi=0)
    info.update(zero)
    seen7 = 0
    for pos, length, number in _sections(msg):
        if number == 3:
            (info["n_points"],) = struct.unpack(">I", msg[pos + 6 : pos + 10])
        elif number == 5:
            p = _section5_params(msg, pos, length)
            del p["template"], p["missing_management"]
            info.update(p)
        elif number == 6:
            indicator = msg[pos + 5]
            if indicator == 0:
                info["has_bitmap"], info["bitmap_offset"] = 1, pos + 6
            elif indicator != 255:
                raise NotImplementedError(f"bitmap indicator {indicator}")
        elif number == 7:
            seen7 += 1
            info["data_offset"], info["data_length"] = pos + 5, length - 5
    if seen7 != 1:
        raise NotImplementedError("messages with several fields")
    if msg[total - 4 : total] != b"7777":
        raise ValueError("end section missing")
    ng, order, ww = info["complex_groups"], info["complex_order"], info["complex_ww"]
    if ng == 0 and info["n_values"] > 0:
        raise ValueError("complex packing with no groups")
    if ng > info["n_values"]:
        raise ValueError("complex packing with more groups than values")
    refs = (order + 1) * ww if order else 0
    widths = refs + (ng * info["bits_per_value"] + 7) // 8
    lengths = widths + (ng * info["complex_width_bits"] + 7) // 8
    values = lengths + (ng * info["complex_length_bits"] + 7) // 8
    if values > info["data_length"]:
        raise ValueError("the group descriptors overrun section 7")
    info.update(complex_refs_offset=refs, complex_widths_offset=widths, complex_lengths_offset=lengths, complex_values_offset=values)
    return info


# ------------------------------------------------------------------------ bit fields ---
def _unpack_varying(bits: np.ndarray, offsets: np.ndarray, widths: np.ndarray) -> np.ndarray:
    """Value i: widths[i] bits (0..32) of the bit array from offsets[i], MSB first."""
    out = np.zeros(offsets.size, dtype=np.int64)
    for b in range(int(widths.max(initial=0))):
        live = widths > b
        out[live] = (out[live] << 1) | bits[offsets[live] + b].astype(np.int64)
    return out


def _pack_varying(values: np.ndarray, widths: np.ndarray) -> bytes:
    """Unsigned values in widths[i] bits each, back to back, zero padded to an octet."""
    widths = widths.astype(np.int64)
    offsets = np.concatenate([[0], np.cumsum(widths)]).astype(np.int64)
    bits = np.zeros(int(offsets[-1]), dtype=np.uint8)
    v = values.astype(np.uint64)
    for b in range(int(widths.max(initial=0))):
        live = widths > b
        shift = (widths[live] - 1 - b).astype(np.uint64)
        bits[offsets[:-1][live] + b] = ((v[live] >> shift) & np.uint64(1)).astype(np.uint8)
    return np.packbits(bits).tobytes()


def _descriptor(buf: bytes, k: int, ww: int) -> int:
    u = int.from_bytes(buf[k * ww : (k + 1) * ww], "big")
    sign = 1 << (8 * ww - 1)
    return -(u & (sign - 1)) if u & sign else u


def _sign_magnitude(v: int, ww: int) -> bytes:
    sign = 1 << (8 * ww - 1)
    if abs(v) >= sign:
        raise ValueError(f"extra descriptor {v} does not fit {ww} octets")
    return ((abs(v) | (sign if v < 0 else 0))).to_bytes(ww, "big")


# ------------------------------------------------------------------------ decoding -----
def undifference_loop(x: np.ndarray, order: int, h1: int, h2: int, gmin: int) -> np.ndarray:
    """The recurrence of the regulation, value by value, in two's-complement int64."""
    mask = (1 << 64) - 1
    wrap = lambda v: ((v + (1 << 63)) & mask) - (1 << 63)  # noqa: E731
    out = [int(v) for v in x]
    for n in range(len(out)):
        if n == 0:
            out[n] = wrap(h1)
        elif n == 1 and order == 2:
            out[n] = wrap(h2)
        elif order == 1:
            out[n] = wrap(out[n - 1] + (out[n] + gmin))
        else:
            out[n] = wrap((out[n] + gmin) + 2 * out[n - 1] - out[n - 2])
    return np.array(out, dtype=np.int64)


def undifference(x: np.ndarray, order: int, h1: int, h2: int, gmin: int) -> np.ndarray:
    """`undifference_loop` as prefix sums: with e_0 = h1, e_1 = h2 - 2·h1 and e_n = X_n + gmin
    after the first `order` values, order 1 is cumsum(e) and order 2 is cumsum(cumsum(e)) —
    the same int64 ring, so the same bits even where the sums wrap."""
    e = x.astype(np.int64) + np.int64(gmin)
    if e.size:
        e[0] = np.int64(h1)
    if order == 2 and e.size > 1:
        e[1] = np.int64(h2) - np.int64(2) * np.int64(h1)
    with np.errstate(over="ignore"):
        d = np.cumsum(e, dtype=np.int64)
        return d if order == 1 else np.cumsum(d, dtype=np.int64)


def decode_x(msg: bytes) -> np.ndarray:
    """The integers X (int64) of a 5.2 / 5.3 message.  ValueError for what the device reports
    as malformed: group lengths that do not sum to the value count, value bits past section 7,
    a group width above 32, a final X outside [0, 2^32)."""
    info = scan(msg)
    n, ng, nb = info["n_values"], info["complex_groups"], info["bits_per_value"]
    if n == 0:
        return np.zeros(0, dtype=np.int64)
    s7 = np.frombuffer(msg, dtype=np.uint8, offset=info["data_offset"], count=info["data_length"])
    part = lambda a, b: s7[info[a] : info[b]].tobytes()  # noqa: E731
    refs = ogrib.unpack_bits(part("complex_refs_offset", "complex_widths_offset"), ng, nb).astype(np.int64)
    widths = info["complex_width_ref"] + ogrib.unpack_bits(part("complex_widths_offset", "complex_lengths_offset"), ng, info["complex_width_bits"]).astype(np.int64)
    scaled = ogrib.unpack_bits(part("complex_lengths_offset", "complex_values_offset"), ng, info["complex_length_bits"]).astype(np.int64)
    lengths = info["complex_length_ref"] + info["complex_length_incr"] * scaled
    lengths[-1] = info["complex_last_length"]
    if (widths > 32).any():
        raise ValueError("a group width above 32 bits")
    if int(lengths.sum()) != n:
        raise ValueError(f"group lengths add up to {int(lengths.sum())}, not {n}")
    value_bits = s7.size * 8 - info["complex_values_offset"] * 8
    if int((widths * lengths).sum()) > value_bits:
        raise ValueError("the packed values run past section 7")
    group = np.repeat(np.arange(ng), lengths)
    first_bit = np.concatenate([[0], np.cumsum(widths * lengths)[:-1]])
    first_value = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    w = widths[group]
    offsets = first_bit[group] + (np.arange(n) - first_value[group]) * w
    bits = np.unpackbits(s7[info["complex_values_offset"] :])
    x = refs[group] + _unpack_varying(bits, offsets, w)
    order = info["complex_order"]
    if order:
        ww = info["complex_ww"]
        desc = s7[: (order + 1) * ww].tobytes()
        h1 = _descriptor(desc, 0, ww)
        h2 = _descriptor(desc, 1, ww) if order == 2 else 0
        x = undifference(x, order, h1, h2, _descriptor(desc, order, ww))
    if ((x < 0) | (x >= 1 << 32)).any():
        raise ValueError("a decoded integer outside [0, 2^32)")
    return x


def to_simple(msg: bytes, nbits: int | None = None) -> bytes:
    """A template 5.2 / 5.3 message → the template 5.0 message of the same R, E, D and X, X in
    `nbits` bits (default: see the module docstring)."""
    info = scan(msg)
    x = decode_x(msg)
    top = int(x.max(initial=0))
    if nbits is None:
        nbits = info["bits_per_value"] if top < (1 << info["bits_per_value"]) else _bit_length(top)
        nbits = max(nbits, 1)
    if top >= (1 << nbits):
        raise ValueError(f"X up to {top} does not fit {nbits} bits")
    s5 = next(pos for pos, _, number in _sections(msg) if number == 5)
    body5 = msg[s5 + 5 : s5 + 9] + struct.pack(">H", 0) + msg[s5 + 11 : s5 + 19] + bytes([nbits, msg[s5 + 20]])
    return _rebuild(msg, {5: body5, 7: ogrib.pack_bits(x.astype(np.uint64), nbits)})


# ------------------------------------------------------------------------ encoding -----
def group_lengths(n: int, size: int) -> list[int]:
    """Groups of `size` values and a ragged last group."""
    if n == 0:
        return []
    return [size] * ((n - 1) // size) + [n - size * ((n - 1) // size)]


def encode_x(
    x: np.ndarray,
    order: int = 2,
    lengths: list[int] | None = None,
    group_size: int = 16,
    increment: int = 1,
    ww: int | None = None,
    min_ref_bits: int = 0,
) -> tuple[bytes, bytes]:
    """(section 5 octets 20-49 after R, E, D — from octet 20 —, section 7) for integers X.

    `order` 0 is template 5.2, 1 or 2 template 5.3.  `lengths`: the group lengths (default:
    `group_size` and a ragged last group); every length but the last must be the smallest of
    them plus a multiple of `increment`.  Each group's reference is its minimum and its width the
    fewest bits for the rest.  Octet 20 is the fewest bits for the references, or
    `min_ref_bits` if that is more.  `ww` defaults to the fewest octets for the descriptors."""
    x = np.asarray(x, dtype=np.int64)
    n = x.size
    lengths = list(lengths) if lengths is not None else group_lengths(n, group_size)
    if sum(lengths) != n:
        raise ValueError("group lengths must add up to the value count")
    desc = b""
    v = x.copy()
    if order:
        h1 = int(x[0]) if n else 0
        h2 = int(x[1]) if order == 2 and n > 1 else 0
        d = x.copy()
        if order == 1:
            d[1:] = x[1:] - x[:-1]
        else:
            d[2:] = x[2:] - 2 * x[1:-1] + x[:-2]
        rest = d[order:]
        gmin = int(rest.min()) if rest.size else 0
        v = d - gmin
        v[:order] = 0  # placeholders: the decoder replaces them
        if ww is None:
            ww = next((k for k in (1, 2, 3, 4) if max(abs(h1), abs(h2), abs(gmin)) < 1 << (8 * k - 1)), 4)
        desc = _sign_magnitude(h1, ww) + (_sign_magnitude(h2, ww) if order == 2 else b"") + _sign_magnitude(gmin, ww)
    ng = len(lengths)
    bounds = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    refs = np.array([int(v[a:b].min()) if b > a else 0 for a, b in zip(bounds[:-1], bounds[1:])], dtype=np.int64)
    widths = np.array([_bit_length(int(v[a:b].max()) - r) if b > a else 0 for a, b, r in zip(bounds[:-1], bounds[1:], refs)], dtype=np.int64)
    nb = max(_bit_length(int(refs.max(initial=0))), min_ref_bits)
    width_ref = int(widths.min(initial=0))
    width_bits = _bit_length(int(widths.max(initial=0)) - width_ref)
    length_ref = min(lengths[:-1]) if ng > 1 else (lengths[0] if ng else 0)
    scaled = [(L - length_ref) // increment for L in lengths[:-1]] + [0]
    if any(length_ref + increment * s != L for s, L in zip(scaled[:-1], lengths[:-1])):
        raise ValueError("group lengths are not the reference plus multiples of the increment")
    length_bits = _bit_length(max(scaled, default=0))
    s7 = (
        desc
        + ogrib.pack_bits(refs.astype(np.uint64), nb)
        + ogrib.pack_bits((widths - width_ref).astype(np.uint64), width_bits)
        + ogrib.pack_bits(np.array(scaled, dtype=np.uint64), length_bits)
        + _pack_varying(v - np.repeat(refs, lengths), np.repeat(widths, lengths))
    )
    s5 = bytes([nb, 0, 1, 0]) + b"\xff" * 8  # octets 20-31: type 0, general group splitting, no missing values
    s5 += struct.pack(">IBBIBIB", ng, width_ref, width_bits, length_ref, increment, lengths[-1] if ng else 0, length_bits)
    if order:
        s5 += bytes([order, ww])
    return s5, s7


def from_simple(msg: bytes, order: int = 2, lengths=None, group_size: int = 16, increment: int = 1, ww: int | None = None) -> bytes:
    """A template 5.0 edition-2 message → the template 5.2 (order 0) or 5.3 message of the same
    R, E, D and X.  Octet 20 is at least the simple message's bits per value, so `to_simple`
    gives the simple message back — except for a constant (0-bit) message, whose X = 0 comes
    back in 1 bit and decodes through the formula, (0 · 2^E + R) · 10^-D."""
    info = ogrib.scan(msg)
    if info["edition"] != 2:
        raise ValueError("complex packing is a GRIB edition 2 template")
    nb = info["bits_per_value"]
    x = ogrib.unpack_bits(msg[info["data_offset"] : info["data_offset"] + info["data_length"]], info["n_values"], nb).astype(np.int64)
    s5_rest, s7 = encode_x(x, order, lengths, group_size, increment, ww, min_ref_bits=nb)
    s5 = next(pos for pos, _, number in _sections(msg) if number == 5)
    body5 = msg[s5 + 5 : s5 + 9] + struct.pack(">H", 3 if order else 2) + msg[s5 + 11 : s5 + 19] + s5_rest
    return _rebuild(msg, {5: body5, 7: s7})


def encode_grib2(values: np.ndarray, nbits: int = 16, decimal_scale: int = 0, bitmap: np.ndarray | None = None, **kw) -> bytes:
    """One GRIB edition 2 message, template 5.2 / 5.3, with the R, E and X that
    `oracle.grib.encode_grib2(values, nbits, decimal_scale, bitmap)` writes; `kw` as in
    `from_simple` (default: order 2, groups of 16)."""
    return from_simple(ogrib.encode_grib2(values, nbits, decimal_scale, bitmap), **kw)


def decode(msg: bytes, n_points: int | None = None, missing=np.nan) -> np.ndarray:
    """float64 values of one message of any template oracle/grib.py, oracle/grib_ccsds.py or
    this module reads, as `GribField.to_numpy(flatten=True)` gives them."""
    if is_complex(msg):
        return ogrib.decode(to_simple(msg), n_points=n_points, missing=missing)
    return ogc.decode(msg, n_points=n_points, missing=missing)


__all__ = ["decode", "decode_x", "encode_grib2", "encode_x", "from_simple", "group_lengths", "is_complex", "scan", "to_simple", "undifference", "undifference_loop"]
