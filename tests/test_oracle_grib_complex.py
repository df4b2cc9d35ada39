"""Complex packing (GRIB2 templates 5.2 and 5.3): the oracle against two messages derived by
hand from the WMO regulations, encoder and decoder against each other over orders, descriptor
widths, group counts, widths 0-32 and the ends of the X range, the messages against simple
packing of the same X, and the C scan (`at_grib_scan`, host only) against the oracle's."""

import ctypes
import struct

import numpy as np
import pytest

from oracle import grib as ogrib
from oracle import grib_ccsds as ogc
from oracle import grib_complex as ogx


def _message(template: int, s5_rest: bytes, s7: bytes, n_values: int, r: float = 0.0, e: int = 0, d: int = 0, bitmap=None) -> bytes:
    """An edition-2 message around a hand-written section 5 tail (octets 20 on) and section 7."""
    base = ogrib.encode_grib2(np.zeros(n_values), 16, 0, bitmap)
    s5 = next(pos for pos, _, number in ogc._sections(base) if number == 5)
    body5 = base[s5 + 5 : s5 + 9] + struct.pack(">H", template) + struct.pack(">f", r) + ogrib.sign_magnitude16(e) + ogrib.sign_magnitude16(d) + s5_rest
    return ogc._rebuild(base, {5: body5, 7: s7})


# ------------------------------------------------------------------ hand-derived messages ----
# 5.2: X = [5, 5, 5, 7, 4, 6, 9, 3, 3]; group lengths 2, 4, 3 (reference 2, increment 2, scaled
# 0 and 1, true last length 3); group references 5, 4, 3 in 3 bits; widths 0, 3, 0 (reference 0,
# 2 bits).  Group 0 is [5, 5] at width 0; group 1 is [5, 7, 4, 6] - 4 = [1, 3, 0, 2]... ;
# group 2 is [9, 3, 3] - 3 = [6, 0, 0] at width 3.
HAND_52_X = [5, 5, 5, 7, 4, 6, 9, 3, 3]
# group 0 = [5, 5] (width 0); group 1 = [5, 7, 4, 6] -> ref 4, packed [1, 3, 0, 2], width 2;
# group 2 = [9, 3, 3] -> ref 3, packed [6, 0, 0], width 3.
#   refs  5, 4, 3 in 3 bits: 101 100 011 -> 1011 0001 1(000 0000) = 0xB1 0x80
#   widths 0, 2, 3 - 0 in 2 bits: 00 10 11 -> 0010 11(00) = 0x2C
#   scaled lengths (L - 2) / 2 for groups 0, 1: 0, 1 (last ignored, 0) in 1 bit: 0 1 0 -> 010(0 0000) = 0x40
#   values: group 1 in 2 bits: 01 11 00 10; group 2 in 3 bits: 110 000 000
#           0111 0010 1100 0000 0(000 0000) = 0x72 0xC0 0x00
HAND_52_S5 = bytes([3, 0, 1, 0]) + b"\xff" * 8 + struct.pack(">IBBIBIB", 3, 0, 2, 2, 2, 3, 1)
HAND_52_S7 = bytes([0xB1, 0x80, 0x2C, 0x40, 0x72, 0xC0, 0x00])

# 5.3 order 2, ww = 2: X = [10, 12, 13, 13, 12, 10, 7, 7]; h1 = 10, h2 = 12.  Second
# differences from n = 2: 13-24+10 = -1, 13-26+12 = -1, 12-26+13 = -1, 10-24+13 = -1,
# 7-20+12 = -1, 7-14+10 = 3, so gmin = -1 and the packed values are [p, p, 0, 0, 0, 0, 0, 4]
# (p: placeholders, written 0).  Two groups of 4 (reference 4, no increment bits, last length
# 4): group 0 = [0]*4, width 0; group 1 = [0, 0, 0, 4] -> ref 0, width 3.  References in 0 bits.
#   descriptors: h1 = 0x000A, h2 = 0x000C, gmin = -1 -> 0x8001
#   refs: none (0 bits); widths 0, 3 in 2 bits: 00 11 -> 0x30; lengths: 0 bits
#   values: group 1 in 3 bits: 000 000 000 100 -> 0000 0000 0100 = 0x00 0x40
HAND_53_X = [10, 12, 13, 13, 12, 10, 7, 7]
HAND_53_S5 = bytes([0, 0, 1, 0]) + b"\xff" * 8 + struct.pack(">IBBIBIB", 2, 0, 2, 4, 1, 4, 0) + bytes([2, 2])
HAND_53_S7 = bytes([0x00, 0x0A, 0x00, 0x0C, 0x80, 0x01, 0x30, 0x00, 0x40])


def test_hand_messages_decode_to_their_defining_x():
    m52 = _message(2, HAND_52_S5, HAND_52_S7, 9, r=100.0, e=1)
    assert ogx.decode_x(m52).tolist() == HAND_52_X
    assert ogx.decode(m52).tolist() == [100.0 + 2.0 * x for x in HAND_52_X]
    m53 = _message(3, HAND_53_S5, HAND_53_S7, 8, r=-3.0, e=0, d=1)
    assert ogx.decode_x(m53).tolist() == HAND_53_X
    assert ogx.decode(m53).tolist() == [(x - 3.0) * 0.1 for x in HAND_53_X]
    info = ogx.scan(m53)
    assert (info["complex_refs_offset"], info["complex_widths_offset"], info["complex_lengths_offset"], info["complex_values_offset"]) == (6, 6, 7, 7)


def test_hand_messages_are_what_the_encoder_writes():
    assert ogx.encode_x(np.array(HAND_52_X), order=0, lengths=[2, 4, 3], increment=2) == (HAND_52_S5, HAND_52_S7)
    assert ogx.encode_x(np.array(HAND_53_X), order=2, lengths=[4, 4], ww=2) == (HAND_53_S5, HAND_53_S7)


def test_recurrence_and_prefix_sums_agree_even_where_int64_wraps():
    rng = np.random.default_rng(0)
    for order in (1, 2):
        for scale in (10, 1 << 40, 1 << 62):
            x = rng.integers(0, scale, 50, dtype=np.int64)
            h1, h2, gmin = (int(v) for v in rng.integers(-scale, scale, 3))
            assert np.array_equal(ogx.undifference(x, order, h1, h2, gmin), ogx.undifference_loop(x, order, h1, h2, gmin))


# ------------------------------------------------------------------ round trips ---------------
def _x_message(x: np.ndarray, **kw) -> bytes:
    s5, s7 = ogx.encode_x(x, **kw)
    return _message(3 if kw.get("order", 2) else 2, s5, s7, x.size)


@pytest.mark.parametrize("order", [0, 1, 2])
@pytest.mark.parametrize("ww", [1, 2, 3, 4])
def test_round_trip_over_orders_and_descriptor_widths(order, ww):
    rng = np.random.default_rng(order * 10 + ww)
    top = (1 << (8 * ww - 1)) - 1  # h1, h2 and gmin fit ww octets
    for n in (1, 2, 3, 17, 300):
        x = rng.integers(0, min(top // 4, 1 << 20) + 1, n, dtype=np.int64)  # differences of order 2 within ±top / 2
        if order and n > 3:
            x = np.clip(np.cumsum(rng.integers(-3, 4, n)) + top // 4, 0, top // 4)
        for kw in (dict(group_size=1), dict(group_size=n), dict(group_size=7), dict(lengths=ogx.group_lengths(n, 5))):
            msg = _x_message(x, order=order, ww=ww if order else None, **kw)
            assert np.array_equal(ogx.decode_x(msg), x), (order, ww, n, kw)
            if order:
                assert ogx.scan(msg)["complex_ww"] == ww


def test_variable_group_lengths_with_an_increment():
    rng = np.random.default_rng(3)
    lengths = [3, 9, 3, 15, 21, 3, 6]
    x = rng.integers(0, 1000, sum(lengths), dtype=np.int64)
    for order in (0, 1, 2):
        msg = _x_message(x, order=order, lengths=lengths, increment=3)
        info = ogx.scan(msg)
        assert (info["complex_length_ref"], info["complex_length_incr"], info["complex_last_length"]) == (3, 3, 6)
        assert np.array_equal(ogx.decode_x(msg), x)
    with pytest.raises(ValueError, match="increment"):
        ogx.encode_x(x, order=0, lengths=lengths, increment=4)


@pytest.mark.parametrize("width", range(33))
def test_every_group_width(width):
    """Groups of width w (a spread of 2^w - 1, up to X = 2^32 - 1 for 5.2); spatial
    differencing over X below 2^28, whose differences fit four-octet descriptors."""
    rng = np.random.default_rng(width)
    spread = (1 << width) - 1
    lo = (1 << 32) - 1 - spread
    x = np.concatenate([[lo, lo + spread], rng.integers(lo, lo + spread + 1, 62, dtype=np.int64)])
    msg = _x_message(x, order=0, group_size=32)
    assert np.array_equal(ogx.decode_x(msg), x)
    s5 = ogx.encode_x(x, order=0, group_size=32)[0]
    assert s5[16] + s5[17] > 0 or width == 0  # width reference, width bits: some group is w wide
    small = x - lo if width <= 28 else rng.integers(0, 1 << 28, 64, dtype=np.int64)
    for order in (1, 2):
        assert np.array_equal(ogx.decode_x(_x_message(small, order=order, group_size=8)), small)


def test_x_at_the_range_ends():
    top = (1 << 32) - 1
    x = np.array([0, top, 0, 1, top - 1, 7], dtype=np.int64)
    for size in (1, 2, 6):
        assert np.array_equal(ogx.decode_x(_x_message(x, order=0, group_size=size)), x)
    # with differencing, steps to 2^32 - 1 of less than 2^31 (what four-octet descriptors hold)
    x = np.array([0, (1 << 31) - 1, top - 1, top, top, top - 5, (1 << 31) + 3], dtype=np.int64)
    for order in (1, 2):
        for size in (1, 2, 7):
            assert np.array_equal(ogx.decode_x(_x_message(x, order=order, group_size=size)), x)
    s = ogx.to_simple(_x_message(x, order=0, group_size=2))
    assert ogrib.scan(s)["bits_per_value"] == 32


def test_x_outside_the_32_bit_range_is_refused():
    # order 1: h1 = 2^32 - 1, one more step of +1
    msg = _x_message(np.array([5, 6], dtype=np.int64), order=1, ww=4)
    s7 = bytearray(msg[ogx.scan(msg)["data_offset"] :])
    s7[0:4] = ((1 << 31) - 1).to_bytes(4, "big")  # h1 = 2^31 - 1: fine
    ok = ogx.decode_x(msg[: ogx.scan(msg)["data_offset"]] + bytes(s7))
    assert ok.tolist() == [(1 << 31) - 1, 1 << 31]
    x = np.array([3, 1, 0], dtype=np.int64)
    bad = _x_message(x, order=1, ww=1)
    info = ogx.scan(bad)
    b = bytearray(bad)
    b[info["data_offset"]] = 0x81  # h1 = -1
    with pytest.raises(ValueError, match=r"outside \[0, 2\^32\)"):
        ogx.decode_x(bytes(b))


@pytest.mark.parametrize("order", [0, 1, 2])
def test_messages_equal_simple_packing_of_the_same_x(order):
    rng = np.random.default_rng(order)
    for nbits in (1, 7, 12, 16, 24) + ((32,) if order == 0 else ()):  # 32-bit differences overflow four-octet descriptors
        for bitmap in (None, rng.uniform(size=500) > 0.3):
            n = 500 if bitmap is None else int(bitmap.sum())
            v = np.cumsum(rng.normal(0.0, 1.0, n)) + 280.0
            simple = ogrib.encode_grib2(v, nbits, order % 2, bitmap)
            cx = ogx.from_simple(simple, order=order, group_size=11)
            assert np.array_equal(ogx.decode(cx, n_points=500), ogrib.decode(simple, n_points=500), equal_nan=True)
            assert ogx.to_simple(cx, nbits) == simple  # 5.0 -> 5.2 / 5.3 -> 5.0
            if order == 0:
                assert ogx.to_simple(cx) == simple  # octet 20 is the simple message's width


# ------------------------------------------------------------------ the C scan ---------------
def _c_scan(native_library, msg):
    from anemoi_transform_b200._cabi import GribInfo

    info = GribInfo()
    buf = np.frombuffer(msg, dtype=np.uint8)
    rc = native_library.at_grib_scan(ctypes.c_void_p(buf.ctypes.data), buf.size, ctypes.byref(info))
    return rc, info


KEYS = (
    "edition", "bits_per_value", "binary_scale", "decimal_scale", "has_bitmap", "reference_value", "data_offset", "data_length",
    "bitmap_offset", "message_length", "n_values", "n_points", "packing", "ccsds_flags", "ccsds_block_size", "ccsds_rsi",
    "complex_groups", "complex_length_ref", "complex_last_length", "complex_width_ref", "complex_width_bits", "complex_length_incr",
    "complex_length_bits", "complex_order", "complex_ww", "complex_refs_offset", "complex_widths_offset", "complex_lengths_offset",
    "complex_values_offset",
)  # fmt: skip


def test_c_scan_equals_the_oracle(native_library):
    from anemoi_transform_b200 import _cabi, grib

    rng = np.random.default_rng(1)
    bm = rng.uniform(size=700) > 0.4
    msgs = [
        _message(2, HAND_52_S5, HAND_52_S7, 9, r=100.0, e=1),
        _message(3, HAND_53_S5, HAND_53_S7, 8, r=-3.0, d=1),
        ogx.encode_grib2(rng.normal(280, 3, 700), 16, 0, order=0),
        ogx.encode_grib2(rng.normal(280, 3, 700), 12, 1, order=1, group_size=1),
        ogx.encode_grib2(rng.normal(280, 3, int(bm.sum())), 24, 0, bm, order=2, lengths=ogx.group_lengths(int(bm.sum()), 40)),
        ogc.encode_grib2(rng.normal(280, 3, 100), 16, 0),
        ogrib.encode_grib2(rng.normal(280, 3, 100), 16, 0),
    ]
    for msg in msgs:
        rc, c = _c_scan(native_library, msg)
        assert rc == 0, native_library.at_last_error()
        o = ogx.scan(msg)
        for key in KEYS:
            assert getattr(c, key) == o[key], (key, getattr(c, key), o[key])
        assert grib.scan(msg) is not None
    assert _c_scan(native_library, msgs[0])[1].packing == _cabi.AT_GRIB_COMPLEX


def _patch5(msg: bytes, octet: int, value: bytes) -> bytes:
    s5 = next(pos for pos, _, number in ogc._sections(msg) if number == 5)
    b = bytearray(msg)
    b[s5 + octet - 1 : s5 + octet - 1 + len(value)] = value
    return bytes(b)


def _truncate5(msg: bytes, length: int) -> bytes:
    s5, l5 = next((pos, length) for pos, length, number in ogc._sections(msg) if number == 5)
    return ogc._rebuild(msg, {5: msg[s5 + 5 : s5 + length]})


def test_c_scan_refusals(native_library):
    from anemoi_transform_b200 import _cabi, grib

    rng = np.random.default_rng(2)
    m53 = ogx.encode_grib2(rng.normal(280, 3, 300), 16, 0, order=2)
    m52 = ogx.encode_grib2(rng.normal(280, 3, 300), 16, 0, order=0)
    unsupported = [
        (_patch5(m53, 23, b"\x01"), b"missing value management 1"),
        (_patch5(m52, 23, b"\x02"), b"missing value management 2"),
        (_patch5(m53, 49, b"\x00"), b"0 octets per extra descriptor"),
        (_patch5(m53, 49, b"\x05"), b"5 octets per extra descriptor"),
        (_patch5(m53, 48, b"\x03"), b"order 3"),
        (_patch5(m53, 48, b"\x00"), b"order 0"),
        (_truncate5(m52, 46), b"5.2 section of 46 octets"),
        (_truncate5(m53, 48), b"5.3 section of 48 octets"),
    ]
    for msg, what in unsupported:
        rc, _ = _c_scan(native_library, msg)
        assert rc == _cabi.AT_ERR_UNSUPPORTED and what in native_library.at_last_error(), (what, native_library.at_last_error())
        assert grib.scan(msg) is None
    # GRIB1 complex / second-order packing (BDS flag 0x40) stays unsupported
    g1 = bytearray(ogrib.encode_grib1(np.arange(50.0), 16, 0))
    bds = 8 + 28 + 32
    g1[bds + 3] |= 0x40
    rc, _ = _c_scan(native_library, bytes(g1))
    assert rc == _cabi.AT_ERR_UNSUPPORTED and b"BDS flags 0x40" in native_library.at_last_error()
    # section 7 too short for the group descriptors, no groups, more groups than values
    info = ogx.scan(m52)
    short = ogc._rebuild(m52, {7: m52[info["data_offset"] : info["data_offset"] + info["complex_values_offset"] - 1]})
    invalid = [
        (short, b"group descriptors need"),
        (_patch5(m52, 32, struct.pack(">I", 0)), b"no groups"),
        (_patch5(m52, 32, struct.pack(">I", 301)), b"301 groups for 300 values"),
    ]
    for msg, what in invalid:
        rc, _ = _c_scan(native_library, msg)
        assert rc == _cabi.AT_ERR_INVALID and what in native_library.at_last_error(), (what, native_library.at_last_error())


def test_unpack_entry_refuses_complex(native_library):
    from anemoi_transform_b200 import _cabi

    rc, info = _c_scan(native_library, ogx.encode_grib2(np.arange(100.0), 16, 0))
    assert rc == 0
    offs = (ctypes.c_int64 * 1)(0)
    dummy = ctypes.c_void_p(16)
    rc = native_library.at_grib_unpack(dummy, offs, ctypes.byref(info), 1, 100, _cabi.AT_F64, dummy, 1, None)
    assert rc == _cabi.AT_ERR_UNSUPPORTED and b"5.2 / 5.3" in native_library.at_last_error()


def test_packed_route_takes_complex_fields(native_library):
    from grib_complex_fields import ComplexGribField

    from anemoi_transform_b200 import grib

    rng = np.random.default_rng(4)
    msgs = [ogx.encode_grib2(rng.normal(280, 3, 400), 16, 0, order=k % 3) for k in range(3)] + [ogrib.encode_grib2(rng.normal(280, 3, 400), 16, 0)]
    fields = [ComplexGribField(m, 400, dict(param="t", step=k)) for k, m in enumerate(msgs)]
    packed = grib.packed_of(fields)
    assert packed is not None and packed.n_points == 400
    want = sum(ogx.scan(m)["data_length"] for m in msgs[:3]) + 800
    assert packed.packed_bytes == want
    assert np.array_equal(fields[0].to_numpy(), ogx.decode(msgs[0]))
