"""CCSDS packing (GRIB2 template 5.42): the AEC oracle against two bitstreams derived by hand
from CCSDS 121.0-B, encoder and decoder against each other over the parameter grid, every
coding option on purpose, the GRIB messages against simple packing of the same X, and the C
scan (`at_grib_scan`, host only) against the oracle's."""

import ctypes
import struct

import numpy as np
import pytest

from oracle import ccsds
from oracle import grib as ogrib
from oracle import grib_ccsds as ogc

PRE, PAD = ccsds.AEC_DATA_PREPROCESS, ccsds.AEC_PAD_RSI


# ------------------------------------------------------------------ hand-derived vectors ---
def test_hand_vector_split_k0():
    # n = 8, J = 8, RSI = 1, PREPROCESS: ID 001 (k = 0), reference 00001010, then the FS codes of
    # δ = 2, 0, 2, 3, 0, 0, 0 (x̂ = 10 → 11: Δ = +1, δ = 2; 11 → 11: 0; 11 → 12: 2; 12 → 10: Δ = −2,
    # δ = 2·2 − 1 = 3; then 0, 0, 0): 001 00001010 001 1 001 0001 1 1 1, zero padded
    x = [10, 11, 11, 12, 10, 10, 10, 10]
    stream = bytes.fromhex("21464780")
    assert ccsds.aec_encode(x, 8, 8, 1, PRE, option=0) == stream
    np.testing.assert_array_equal(ccsds.aec_decode(stream, 8, 8, 1, PRE, 8), x)


def test_hand_vector_zero_block():
    # eight 10s: ID 000, selector 0 (zero-block), reference 00001010, FS(0) (z = 1: one block)
    stream = bytes.fromhex("00a8")
    assert ccsds.aec_encode([10] * 8, 8, 8, 1, PRE) == stream
    np.testing.assert_array_equal(ccsds.aec_decode(stream, 8, 8, 1, PRE, 8), [10] * 8)


def test_predictor_mapping_inverts_at_the_range_ends():
    # x̂ at 0 and at xmax: every branch of the θ mapping (δ <= 2θ even / odd, δ > 2θ both sides)
    for n in (1, 3, 8, 16, 32):
        xmax = (1 << n) - 1
        pts = sorted({0, 1, xmax // 2, xmax // 2 + 1, xmax - 1, xmax} & set(range(0, xmax + 1)) if n < 20 else {0, 1, xmax // 2, xmax - 1, xmax})
        for prev in pts:
            for x in pts:
                d = int(ccsds.preprocess(np.array([prev, x]), n, 8, 4096)[1])
                assert 0 <= d <= xmax
                assert ccsds.postprocess_one(d, prev, xmax) == x


# ------------------------------------------------------------------ round trips ------------
def _samples(rng, n, nv, kind):
    xmax = (1 << n) - 1
    if kind == "smooth":
        return (np.cumsum(rng.integers(-3, 4, nv)) % (xmax + 1)).astype(np.int64)
    if kind == "noise":
        return rng.integers(0, xmax + 1, nv, dtype=np.int64)
    # pinned at 0 and at xmax, with steps across the whole range
    x = rng.choice(np.array([0, xmax, xmax // 2, 1 if xmax else 0, max(xmax - 1, 0)]), nv)
    x[: nv // 3] = 0
    x[nv // 3 : 2 * nv // 3] = xmax
    return x.astype(np.int64)


@pytest.mark.parametrize("n", [1, 2, 3, 7, 8, 9, 15, 16, 17, 24, 25, 31, 32])
def test_round_trip_parameter_grid(n):
    rng = np.random.default_rng(n)
    for J in (8, 16, 32, 64):
        for rsi in (1, 2, 3, 128, 4096):
            for flags in (0, PRE, PAD, PRE | PAD, PRE | 6):
                # n_values not a multiple of J nor of J·RSI, and one that is
                for nv in (int(rng.integers(1, 2500)), J * 3 + 1, J * min(rsi, 4) * 2):
                    kind = ("smooth", "noise", "edges")[int(rng.integers(0, 3))]
                    x = _samples(rng, n, nv, kind)
                    for pad in ("block", "rsi"):
                        s = ccsds.aec_encode(x, n, J, rsi, flags, pad=pad)
                        np.testing.assert_array_equal(ccsds.aec_decode(s, n, J, rsi, flags, nv), x, err_msg=f"{n} {J} {rsi} {flags} {nv} {kind} {pad}")


@pytest.mark.parametrize("option", ["se", "uncompressed", 0, 1, 2, 4, 6, 13, 29])
@pytest.mark.parametrize("flags", [0, PRE, PRE | PAD])
def test_every_option_forced(option, flags):
    rng = np.random.default_rng(7)
    for n in (3, 8, 12, 16, 24, 32):
        kmax = min((1 << ccsds.id_length(n)) - 3, n - 1)
        if isinstance(option, int) and option > kmax:
            continue
        for J in (8, 32):
            # split k and second extension want x >> k (or δ >> k) small: values below 2^(k+3)
            k = 0 if option == "se" else option if isinstance(option, int) else n
            x = rng.integers(0, 1 << min(n, k + 3), 1000, dtype=np.int64)
            s = ccsds.aec_encode(x, n, J, 16, flags, option=option)
            np.testing.assert_array_equal(ccsds.aec_decode(s, n, J, 16, flags, x.size), x)


@pytest.mark.parametrize("flags", [0, PRE, PAD, PRE | PAD])
def test_zero_block_runs(flags):
    # runs of 1 .. 4 blocks (FS code z = r), 5 .. 9 blocks (z = r + 1), the remainder of a
    # segment crossing the 64-block boundary inside a 128-block RSI, and the end of an RSI
    J, rsi, n = 16, 128, 12
    rng = np.random.default_rng(flags)
    blocks = []
    runs = [1, 2, 3, 4, 5, 6, 7, 9]
    b = 0
    for r in runs:
        blocks.append(rng.integers(1, 4000, J))
        blocks.extend([np.zeros(J, dtype=np.int64)] * r)
        b += 1 + r
    while b < 58:
        blocks.append(rng.integers(1, 4000, J))
        b += 1
    blocks.extend([np.zeros(J, dtype=np.int64)] * (128 - b + 20))  # to the 64 boundary, the RSI end, then on
    blocks.append(rng.integers(1, 4000, J))
    blocks.extend([np.zeros(J, dtype=np.int64)] * 70)
    x = np.concatenate(blocks).astype(np.int64)
    if flags & PRE:  # zero blocks of δ: constant runs of x
        x = np.concatenate([np.cumsum(blk) % 4096 if blk.any() else np.full(J, -1) for blk in blocks]).astype(np.int64)
        for i in range(x.size):
            if x[i] < 0:
                x[i] = x[i - 1]
    for pad in ("block", "rsi"):
        s = ccsds.aec_encode(x, n, J, rsi, flags, pad=pad)
        np.testing.assert_array_equal(ccsds.aec_decode(s, n, J, rsi, flags, x.size), x)


def test_remainder_of_segment_code_is_used():
    # 64 zero blocks from block 0 of a 128-block RSI: one ROS code (ID 000, selector 0, FS(4))
    J, n = 8, 8
    x = np.zeros(J * 64 + J, dtype=np.int64)
    x[-J:] = np.arange(1, J + 1)
    s = ccsds.aec_encode(x, n, J, 128, 0)
    assert s[0] == 0 and s[1] & 0x80  # 000 0 0000 1: ID, selector, FS(4) (not 64 zeros and a one)
    np.testing.assert_array_equal(ccsds.aec_decode(s, n, J, 128, 0, x.size), x)


def test_malformed_streams_are_refused():
    x = np.arange(100, dtype=np.int64) % 50
    s = ccsds.aec_encode(x, 8, 8, 4, PRE)
    with pytest.raises(ValueError):
        ccsds.aec_decode(s[: len(s) // 2], 8, 8, 4, PRE, x.size)
    # a zero-block run of 9 blocks in an RSI of 4: 000 0 FS(9)
    bad = bytes([0b00000000, 0b00000100])
    with pytest.raises(ValueError):
        ccsds.aec_decode(bad + bytes(8), 8, 8, 4, 0, 32)
    for flags, n, J, rsi in ((1, 8, 8, 4), (16, 4, 8, 4), (0, 8, 12, 4), (0, 8, 8, 0), (0, 8, 8, 4097)):
        with pytest.raises(NotImplementedError):
            ccsds.aec_decode(s, n, J, rsi, flags, x.size)


# ------------------------------------------------------------------ GRIB messages ----------
@pytest.mark.parametrize("nbits", [1, 7, 12, 16, 24, 32])
@pytest.mark.parametrize("flags", [14, 8, 0, 46])
def test_ccsds_message_decodes_like_simple_packing(nbits, flags):
    rng = np.random.default_rng(nbits + flags)
    v = np.cumsum(rng.normal(0, 0.3, 4000)) + 280.0
    bm = rng.uniform(size=4000) > 0.25
    for bitmap, vals in ((None, v[:3001]), (bm, v[: int(bm.sum())])):
        for decimal in (0, 2):
            simple = ogrib.encode_grib2(vals, nbits, decimal, bitmap)
            packed = ogc.encode_grib2(vals, nbits, decimal, bitmap, block_size=16, rsi=32, flags=flags)
            info = ogc.scan(packed)
            assert info["packing"] == 1 and (info["ccsds_flags"], info["ccsds_block_size"], info["ccsds_rsi"]) == (flags, 16, 32)
            a, b = ogrib.decode(simple), ogc.decode(packed)
            np.testing.assert_array_equal(a.view(np.uint64), b.view(np.uint64))
    const = ogc.encode_grib2(np.full(50, 2.5), 16, 0)
    assert (ogc.decode(const) == 2.5).all()


def test_smooth_16_bit_field_compresses():
    rng = np.random.default_rng(3)
    lat = np.linspace(-1.5, 1.5, 20000)
    v = 250.0 + 40.0 * np.cos(lat) + np.cumsum(rng.normal(0, 0.01, lat.size))
    simple = ogrib.encode_grib2(v, 16, 0)
    packed = ogc.encode_grib2(v, 16, 0)
    assert ogc.scan(packed)["data_length"] < 0.7 * ogrib.scan(simple)["data_length"]


# ------------------------------------------------------------------ the C scan -------------
def _c_scan(native_library, msg):
    from anemoi_transform_b200._cabi import GribInfo

    info = GribInfo()
    buf = np.frombuffer(msg, dtype=np.uint8)
    rc = native_library.at_grib_scan(ctypes.c_void_p(buf.ctypes.data), buf.size, ctypes.byref(info))
    return rc, info


def test_c_scan_equals_the_oracle_on_5_42(native_library):
    from anemoi_transform_b200 import _cabi, grib

    rng = np.random.default_rng(1)
    bm = rng.uniform(size=500) > 0.4
    cases = [
        ogc.encode_grib2(rng.normal(280, 5, 777), nb, d, block_size=J, rsi=rsi, flags=fl)
        for nb, d, J, rsi, fl in ((16, 0, 32, 128, 14), (12, 1, 8, 1, 8), (24, -1, 64, 4096, 46), (5, 0, 16, 3, 0), (32, 0, 32, 7, 40))
    ]
    cases.append(ogc.encode_grib2(rng.normal(0, 1, int(bm.sum())), 16, 0, bm))
    cases.append(ogc.encode_grib2(np.full(64, -7.25), 16, 0))
    for msg in cases:
        rc, c = _c_scan(native_library, msg)
        assert rc == 0, native_library.at_last_error()
        o = ogc.scan(msg)
        for key in ("edition", "bits_per_value", "binary_scale", "decimal_scale", "has_bitmap", "reference_value", "data_offset",
                    "data_length", "bitmap_offset", "message_length", "n_values", "n_points", "packing", "ccsds_flags", "ccsds_block_size", "ccsds_rsi"):
            assert getattr(c, key) == o[key], (key, getattr(c, key), o[key])
        assert c.packing == _cabi.AT_GRIB_CCSDS
        assert grib.scan(msg) is not None
    # simple packing still scans as AT_GRIB_SIMPLE with zero CCSDS parameters
    rc, c = _c_scan(native_library, ogrib.encode_grib2(rng.normal(0, 1, 10), 16, 0))
    assert rc == 0 and c.packing == _cabi.AT_GRIB_SIMPLE and (c.ccsds_flags, c.ccsds_block_size, c.ccsds_rsi) == (0, 0, 0)


def _with_section5(msg: bytes, flags: int, J: int, rsi: int) -> bytes:
    o = ogc.scan(msg)
    pos = 16
    b = bytearray(msg)
    while True:
        (length,) = struct.unpack(">I", msg[pos : pos + 4])
        if msg[pos + 4] == 5:
            b[pos + 21], b[pos + 22] = flags, J
            b[pos + 23 : pos + 25] = struct.pack(">H", rsi)
            return bytes(b)
        pos += length
        assert pos < o["message_length"]


def test_c_scan_refuses_what_the_device_does_not_decode(native_library):
    from anemoi_transform_b200 import _cabi, grib

    msg = ogc.encode_grib2(np.arange(100.0), 16, 0, block_size=32, rsi=128, flags=14)
    assert _c_scan(native_library, msg)[0] == 0
    for flags, J, rsi, what in (
        (15, 32, 128, b"signed"),
        (14 | 16, 32, 128, None),  # restricted is refused only for n <= 4
        (14, 12, 128, b"block size"),
        (14, 128, 128, b"block size"),
        (14, 32, 0, b"reference sample interval"),
        (14, 32, 4097, b"reference sample interval"),
    ):
        rc = _c_scan(native_library, _with_section5(msg, flags, J, rsi))[0]
        if what is None:
            assert rc == 0
            continue
        assert rc == _cabi.AT_ERR_UNSUPPORTED and what in native_library.at_last_error(), (flags, J, rsi)
        assert grib.scan(_with_section5(msg, flags, J, rsi)) is None
    low = ogc.encode_grib2(np.arange(10.0), 4, 0, flags=8)
    assert _c_scan(native_library, low)[0] == 0
    rc = _c_scan(native_library, _with_section5(low, 8 | 16, 32, 128))[0]
    assert rc == _cabi.AT_ERR_UNSUPPORTED and b"restricted" in native_library.at_last_error()


def test_packed_route_takes_ccsds_fields(native_library):
    from grib_ccsds_fields import CcsdsGribField as GribMessageField

    from anemoi_transform_b200 import grib

    rng = np.random.default_rng(4)
    v = np.cumsum(rng.normal(0, 0.2, 4000)) + 270
    simple = GribMessageField(ogrib.encode_grib2(v, 16, 0), v.size, {"param": "t"})
    packed = GribMessageField(ogc.encode_grib2(v, 16, 0), v.size, {"param": "t"})
    both = grib.packed_of([simple, packed])
    assert both is not None and both.n_points == v.size
    info = both.infos[1]
    assert info.packing == 1
    # PCIe carries the AEC stream, not n·nbits/8
    assert both.packed_bytes == 2 * v.size + info.data_length
    assert info.data_length < 2 * v.size
    # host route: the test field decodes through the oracle unchanged
    np.testing.assert_array_equal(packed.to_numpy(), simple.to_numpy())


def test_unpack_entry_refuses_ccsds(native_library):
    from anemoi_transform_b200 import _cabi

    msg = ogc.encode_grib2(np.arange(100.0), 16, 0)
    rc, info = _c_scan(native_library, msg)
    assert rc == 0
    offs = (ctypes.c_int64 * 1)(0)
    dummy = ctypes.c_void_p(16)
    rc = native_library.at_grib_unpack(dummy, offs, ctypes.byref(info), 1, 100, _cabi.AT_F64, dummy, 1, None)
    assert rc == _cabi.AT_ERR_UNSUPPORTED and b"5.42" in native_library.at_last_error()


def test_message_conversion_round_trips():
    # 5.0 → 5.42 → 5.0 gives the simple-packed message back octet for octet
    rng = np.random.default_rng(11)
    bm = rng.uniform(size=900) > 0.3
    for vals, bitmap, nb in ((rng.normal(280, 5, 900), None, 16), (rng.normal(0, 1, int(bm.sum())), bm, 11), (np.full(9, 1.5), None, 16)):
        simple = ogrib.encode_grib2(vals, nb, 1, bitmap)
        packed = ogc.from_simple(simple, 16, 8, 40)
        assert ogc.is_ccsds(packed) and not ogc.is_ccsds(simple)
        assert ogc.to_simple(packed) == simple
        assert ogc.scan(simple)["packing"] == 0 and ogc.scan(packed)["message_length"] == len(packed)
