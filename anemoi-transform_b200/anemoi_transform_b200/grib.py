"""GRIB-backed fields: hand the packed message to the device instead of decoding on the host.

In the reference a GRIB FieldList reaches a filter as earthkit-data `GribField`s and every
`field.to_numpy(flatten=True)` (`filters/fields/regrid.py:309`, `matching.py:242-246`) has
ecCodes decode one message to float64 on one core.  A field whose *class* provides
`message()` (earthkit-data's `GribField.message()` returns the encoded message) and whose
message is grid-point simple packing, complex packing with or without spatial differencing,
or CCSDS packing (templates 5.0, 5.2, 5.3 and 5.42, with or without a bitmap) is uploaded
packed — 2 bytes per point at 16 bits instead of 8, less for complex and CCSDS — and decoded on
the device straight into the [points x fields] batch (`csrc/grib.cu`: the complex and CCSDS
kernels turn section 7 into 32-bit words, `grib_unpack_kernel` applies the packing formula).
Everything else keeps the `to_numpy()` route.

Wrapper fields (`NewDataField` and friends) forward unknown attributes to the field they
wrap, so `message()` of a wrapper would return the *original* data; only a `message` defined
on the field's own class counts.

`AT_B200_GRIB_DEVICE_DECODE=0` switches the packed route off.  `AT_B200_GRIB_DTYPE=float32`
(or `set_decode_dtype(np.float32)`) makes the device write the decoded values as float32 —
`to_numpy(dtype=np.float32)` instead of `to_numpy()`: the regridded fields then come back as
float32 when the matrix is float32, half the bytes in HBM and on the way out.  The default is
float64, what the reference's `to_numpy(flatten=True)` hands to the matrix.
"""

from __future__ import annotations

import math
import os
from ctypes import byref, c_int32, c_size_t, c_void_p
from typing import Any, Sequence

import numpy as np

from . import _cabi
from ._cabi import GribInfo


def enabled() -> bool:
    return os.environ.get("AT_B200_GRIB_DEVICE_DECODE", "1") != "0"


_decode_dtype: np.dtype | None = None


def set_decode_dtype(dtype) -> None:
    """float64 (default, the reference's `to_numpy()`), float32, or None for the environment's choice."""
    global _decode_dtype
    if dtype is not None and np.dtype(dtype) not in (np.dtype(np.float32), np.dtype(np.float64)):
        raise ValueError("GRIB values decode to float32 or float64")
    _decode_dtype = None if dtype is None else np.dtype(dtype)


def decode_dtype() -> np.dtype:
    if _decode_dtype is not None:
        return _decode_dtype
    return np.dtype(np.float32 if os.environ.get("AT_B200_GRIB_DTYPE", "float64") in ("float32", "f32") else np.float64)


def scan(message) -> GribInfo | None:
    """Packing parameters of one message, or None when it is not something the device decodes
    (not GRIB, another packing, several fields).  Host only."""
    return _scan_buffer(np.frombuffer(message, dtype=np.uint8))


def _scan_buffer(buf: np.ndarray) -> GribInfo | None:
    info = GribInfo()
    rc = _cabi.load().at_grib_scan(buf.__array_interface__["data"][0], buf.size, byref(info))
    return info if rc == _cabi.AT_OK else None


def _message_of(field: Any):
    method = getattr(type(field), "message", None)
    if method is None or not callable(method):
        return None
    try:
        m = field.message()
    except Exception:
        return None
    if isinstance(m, (bytes, bytearray, memoryview)) and len(m) >= 16:
        return m
    return None


def is_packed_message(field: Any) -> bool:
    """Would `packed_of([field])` take the packed route?"""
    return packed_of([field]) is not None


class PackedFields:
    """The messages of a FieldList the device can decode, with their scans."""

    def __init__(self, buffers: list[np.ndarray], infos, n_points: int, pointers=None):
        self.buffers = buffers  # uint8 views on the messages: keep them alive while in use
        self.infos = infos  # ctypes array of GribInfo
        self.n_points = n_points
        self.n_fields = len(buffers)
        self.pointers = pointers if pointers is not None else (c_void_p * self.n_fields)(*[b.__array_interface__["data"][0] for b in buffers])
        #: dtype the device decodes to: float64 = what `GribField.to_numpy()` returns
        self.dtype = decode_dtype()

    @property
    def packed_bytes(self) -> int:
        """Octets that cross PCIe: packed values (the whole section 7 of a CCSDS or complex
        field), plus one bit per point for fields with a bitmap."""
        total = 0
        for i in self.infos:
            values = i.n_values if (i.has_bitmap and i.n_values >= 0) else self.n_points
            packed = i.data_length if _is_stream(i) else (values * i.bits_per_value + 7) // 8
            total += packed + ((self.n_points + 7) // 8 if i.has_bitmap else 0)
        return int(total)


def _is_stream(info: GribInfo) -> bool:
    """Section 7 goes up whole and is decoded on the device (CCSDS and complex packing)."""
    return info.packing == _cabi.AT_GRIB_COMPLEX or (info.packing == _cabi.AT_GRIB_CCSDS and info.bits_per_value > 0)


def packed_of(fields: Sequence[Any]) -> PackedFields | None:
    """`PackedFields` when *every* field is a simple-, complex- or CCSDS-packed GRIB message of the same grid size,
    else None (the caller then uses `to_numpy()` for all of them).  Points a bitmap marks as
    missing decode to NaN."""
    if not fields or not enabled():
        return None
    n = len(fields)
    buffers: list[np.ndarray] = []
    for f in fields:
        m = _message_of(f)
        if m is None:
            return None
        buffers.append(np.frombuffer(m, dtype=np.uint8))
    pointers = (c_void_p * n)(*[b.__array_interface__["data"][0] for b in buffers])
    lengths = (c_size_t * n)(*[b.size for b in buffers])
    infos = (GribInfo * n)()
    status = (c_int32 * n)()
    _cabi.call("at_grib_scan_many", pointers, lengths, n, infos, status)  # one call: the per-message parse is C
    if any(status):
        return None
    n_points = -1
    for f, info in zip(fields, infos):
        # grid points of the field: with a bitmap the message says (n_points), the packed stream
        # then holds only the n_values points that are present (the device decodes the rest to NaN)
        if info.has_bitmap:
            count, packed_values = info.n_points, info.n_values
        else:
            count = info.n_values if info.n_values >= 0 else info.n_points
            packed_values = count
        shape = getattr(f, "shape", None)
        if shape is not None:
            declared = math.prod(shape)
            if count >= 0 and count != declared:
                return None
            count = declared
            if not info.has_bitmap:
                packed_values = count
        if count < 0 or (n_points >= 0 and count != n_points):
            return None
        if packed_values > count:
            return None
        # a simple-packed section holds at least its values; the length of an AEC stream or a
        # complex section 7 says nothing about the count (the device checks it as it decodes)
        if not _is_stream(info) and packed_values >= 0 and info.data_length < (packed_values * info.bits_per_value + 7) // 8:
            return None
        n_points = count
    return PackedFields(buffers, infos, n_points, pointers)


def split(fields: Sequence[Any]) -> tuple[PackedFields | None, list[int], list[int]]:
    """Partition a FieldList: (the messages the device decodes, their positions, the positions of
    the fields that keep the `to_numpy()` route — other packings, wrappers, numpy fields)."""
    if not fields or not enabled():
        return None, [], list(range(len(fields)))
    candidates = [i for i, f in enumerate(fields) if _message_of(f) is not None]
    if not candidates:
        return None, [], list(range(len(fields)))
    whole = packed_of(fields) if len(candidates) == len(fields) else None
    if whole is not None:
        return whole, list(range(len(fields))), []
    # field by field: keep those that scan as simple, complex or CCSDS packing and share the size of the first such field
    keep: list[int] = []
    n_points = -1
    for i in candidates:
        one = packed_of([fields[i]])
        if one is not None and (n_points < 0 or one.n_points == n_points):
            n_points = one.n_points
            keep.append(i)
    if not keep:
        return None, [], list(range(len(fields)))
    packed = packed_of([fields[i] for i in keep])
    if packed is None:  # pragma: no cover - each member was accepted on its own
        return None, [], list(range(len(fields)))
    kept = set(keep)
    return packed, keep, [i for i in range(len(fields)) if i not in kept]


def upload(packed: PackedFields, dtype=None):
    """→ `DeviceBatch` holding the decoded fields as columns (`at_hostio_upload_grib`)."""
    from .device import AT_F32, AT_F64, DeviceBatch, HostIO, _ptr, empty_batch, require_cuda, stream_ptr

    torch = require_cuda()
    dtype = np.dtype(dtype) if dtype is not None else packed.dtype
    tdtype = torch.float32 if dtype == np.float32 else torch.float64
    pm = empty_batch(packed.n_points, packed.n_fields, tdtype, "cuda")
    _cabi.call(
        "at_hostio_upload_grib",
        HostIO.get().handle,
        packed.pointers,
        packed.infos,
        packed.n_fields,
        packed.n_points,
        AT_F32 if dtype == np.float32 else AT_F64,
        _ptr(pm),
        int(pm.stride(0)),
        stream_ptr(),
    )
    return DeviceBatch(pm, packed.n_fields)


__all__ = ["GribInfo", "PackedFields", "decode_dtype", "enabled", "is_packed_message", "packed_of", "scan", "set_decode_dtype", "split", "upload"]
