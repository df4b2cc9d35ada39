"""Oracle: GRIB2 CCSDS packing (data representation template 5.42) — messages in numpy.

TEST INFRASTRUCTURE — see oracle/__init__.py.

Template 5.42 is section 5 of template 5.0 (simple packing, oracle/grib.py) followed by three
more fields (octets numbered from the start of the section):

    22  CCSDS flags (libaec's AEC_* values)      23  block size J
    24-25  reference sample interval (RSI, in blocks)

and section 7 is one AEC stream (CCSDS 121.0-B, oracle/ccsds.py) of the same unsigned integers
X simple packing would store.  Decoded values are Y = ((X · 2^E) + R) · 10^-D, as for 5.0.

So this module works by conversion: `encode_grib2` writes the simple-packed message with
`oracle.grib.encode_grib2` and recodes its X as an AEC stream (same R, E, D and X, so the two
messages can be compared value for value), and `decode` turns a 5.42 message back into the 5.0
message of the same X and hands it to `oracle.grib.decode` — the arithmetic, bitmaps and
missing values are exactly simple packing's.  Messages of any other template go to
oracle/grib.py unchanged.

PARITY UNPINNED: libaec and ecCodes cannot be run here (see oracle/ccsds.py).
"""

from __future__ import annotations

import struct

import numpy as np

from . import ccsds
from . import grib as ogrib


def _sections(msg: bytes):
    """(position, length, number) of every section of an edition-2 message between 0 and 8."""
    (total,) = struct.unpack(">Q", msg[8:16])
    pos = 16
    while pos < total - 4:
        (length,) = struct.unpack(">I", msg[pos : pos + 4])
        yield pos, length, msg[pos + 4]
        pos += length


def _rebuild(msg: bytes, bodies: dict) -> bytes:
    """The message with the bodies (octets after the 5-octet header) of some sections replaced."""
    parts = []
    for pos, length, number in _sections(msg):
        if number in bodies:
            parts.append(struct.pack(">IB", 5 + len(bodies[number]), number) + bodies[number])
        else:
            parts.append(msg[pos : pos + length])
    body = b"".join(parts) + b"7777"
    return msg[:8] + struct.pack(">Q", 16 + len(body)) + body


def is_ccsds(msg: bytes) -> bool:
    if msg[:4] != b"GRIB" or msg[7] != 2:
        return False
    for pos, length, number in _sections(msg):
        if number == 5:
            return length >= 11 and struct.unpack(">H", msg[pos + 9 : pos + 11])[0] == 42
    return False


def scan(msg: bytes) -> dict:
    """`oracle.grib.scan` plus `packing` (0 simple, 1 CCSDS) and the CCSDS parameters
    (`ccsds_flags`, `ccsds_block_size`, `ccsds_rsi`; 0 for simple packing)."""
    if not is_ccsds(msg):
        info = ogrib.scan(msg)
        info.update(packing=0, ccsds_flags=0, ccsds_block_size=0, ccsds_rsi=0)
        return info
    (total,) = struct.unpack(">Q", msg[8:16])
    info = dict(edition=2, bitmap_offset=-1, has_bitmap=0, message_length=total, packing=1)
    seen7 = 0
    for pos, length, number in _sections(msg):
        if number == 3:
            (info["n_points"],) = struct.unpack(">I", msg[pos + 6 : pos + 10])
        elif number == 5:
            if length < 25:
                raise NotImplementedError(f"template 5.42 section of {length} octets")
            (info["n_values"],) = struct.unpack(">I", msg[pos + 5 : pos + 9])
            info["reference_value"] = float(struct.unpack(">f", msg[pos + 11 : pos + 15])[0])
            info["binary_scale"] = ogrib.from_sign_magnitude16(msg[pos + 15 : pos + 17])
            info["decimal_scale"] = ogrib.from_sign_magnitude16(msg[pos + 17 : pos + 19])
            info["bits_per_value"] = msg[pos + 19]
            info["ccsds_flags"], info["ccsds_block_size"] = msg[pos + 21], msg[pos + 22]
            (info["ccsds_rsi"],) = struct.unpack(">H", msg[pos + 23 : pos + 25])
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
    return info


def from_simple(msg: bytes, block_size: int = 32, rsi: int = 128, flags: int = 14, option=None, pad: str = "block") -> bytes:
    """A template 5.0 edition-2 message → the template 5.42 message of the same R, E, D and X."""
    info = ogrib.scan(msg)
    if info["edition"] != 2:
        raise ValueError("CCSDS packing is a GRIB edition 2 template")
    nb = info["bits_per_value"]
    x = ogrib.unpack_bits(msg[info["data_offset"] : info["data_offset"] + info["data_length"]], info["n_values"], nb)
    stream = ccsds.aec_encode(x.astype(np.int64), nb, block_size, rsi, flags, option=option, pad=pad)
    s5 = next(pos for pos, _, number in _sections(msg) if number == 5)
    body5 = msg[s5 + 5 : s5 + 9] + struct.pack(">H", 42) + msg[s5 + 11 : s5 + 21] + struct.pack(">BBH", flags, block_size, rsi)
    return _rebuild(msg, {5: body5, 7: stream})


def to_simple(msg: bytes) -> bytes:
    """A template 5.42 message → the template 5.0 message of the same X (the AEC stream decoded)."""
    info = scan(msg)
    nb = info["bits_per_value"]
    stream = msg[info["data_offset"] : info["data_offset"] + info["data_length"]]
    x = ccsds.aec_decode(stream, nb, info["ccsds_block_size"], info["ccsds_rsi"], info["ccsds_flags"], info["n_values"])
    s5 = next(pos for pos, _, number in _sections(msg) if number == 5)
    body5 = msg[s5 + 5 : s5 + 9] + struct.pack(">H", 0) + msg[s5 + 11 : s5 + 21]
    return _rebuild(msg, {5: body5, 7: ogrib.pack_bits(x, nb)})


def encode_grib2(
    values: np.ndarray,
    nbits: int = 16,
    decimal_scale: int = 0,
    bitmap: np.ndarray | None = None,
    block_size: int = 32,
    rsi: int = 128,
    flags: int = 14,
    option=None,
    pad: str = "block",
) -> bytes:
    """One GRIB edition 2 message, template 5.42, with the R, E and X that
    `oracle.grib.encode_grib2(values, nbits, decimal_scale, bitmap)` writes.  Defaults are
    ECMWF's (J = 32, RSI = 128, flags 14 = PREPROCESS | MSB | 3BYTE); `option` and `pad` as in
    `ccsds.aec_encode`."""
    return from_simple(ogrib.encode_grib2(values, nbits, decimal_scale, bitmap), block_size, rsi, flags, option, pad)


def decode(msg: bytes, n_points: int | None = None, missing=np.nan) -> np.ndarray:
    """float64 values of one message of any template oracle/grib.py or this module reads, as
    `GribField.to_numpy(flatten=True)` gives them."""
    return ogrib.decode(to_simple(msg) if is_ccsds(msg) else msg, n_points=n_points, missing=missing)


__all__ = ["decode", "encode_grib2", "from_simple", "is_ccsds", "scan", "to_simple"]
