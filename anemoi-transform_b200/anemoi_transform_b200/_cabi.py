"""ctypes binding of libat_b200.so — the C-ABI declared in include/at_b200.h.

The library is the only compute path of this package: if it is missing, or no CUDA device
is usable, calls fail loudly (`NativeLibraryError`); there is no CPU fallback.
"""

from __future__ import annotations

import ctypes
import os
import threading
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint8, c_uint32, c_uint64, c_void_p
from pathlib import Path

LIB_NAME = "libat_b200.so"
LIB_PATH = Path(__file__).resolve().parent / "lib" / LIB_NAME

AT_OK = 0
AT_ERR_INVALID, AT_ERR_CUDA, AT_ERR_NOMEM, AT_ERR_UNSUPPORTED, AT_ERR_INDEX = 1, 2, 3, 4, 5
AT_GRIB_SIMPLE, AT_GRIB_CCSDS, AT_GRIB_COMPLEX = 0, 1, 2  # at_grib_field_t.packing
AT_F32, AT_F64 = 0, 1
AT_I32, AT_I64 = 0, 1

EPI_PLAIN, EPI_UV2DDFF, EPI_DDFF2UV, EPI_QT2R, EPI_QT2QTR, EPI_RT2Q, EPI_RT2RTQ = range(7)
EPI_AFFINE, EPI_AFFINE_INV, EPI_EXP, EPI_LOG, EPI_IMPUTE_NAN, EPI_COSSIN, EPI_ATAN2 = range(7, 14)
EPI_RT2D, EPI_RT2RTD, EPI_DT2R, EPI_DT2DTR = range(14, 18)
# outputs per 4 input columns of each kind
EPI_OUT_PER_GROUP = {
    EPI_PLAIN: 4, EPI_UV2DDFF: 4, EPI_DDFF2UV: 4, EPI_QT2R: 2, EPI_QT2QTR: 6, EPI_RT2Q: 2, EPI_RT2RTQ: 6,
    EPI_AFFINE: 4, EPI_AFFINE_INV: 4, EPI_EXP: 4, EPI_LOG: 4, EPI_IMPUTE_NAN: 4, EPI_COSSIN: 8, EPI_ATAN2: 2,
    EPI_RT2D: 2, EPI_RT2RTD: 6, EPI_DT2R: 2, EPI_DT2DTR: 6,
}  # fmt: skip
HOSTIO_SPMM, HOSTIO_GATHER, HOSTIO_SPMM_MISSING_ALL, HOSTIO_SPMM_MISSING_HEAVIEST = 0, 1, 2, 3
MISSING_PROPAGATE, MISSING_ALL, MISSING_HEAVIEST = 0, 1, 2
EXCHANGE_INLINE, EXCHANGE_BULK = 0, 1
CMP_NOT_NAN = 6
COL_CLIP_LO, COL_CLIP_HI, COL_MASK = 1, 2, 4


class NativeLibraryError(RuntimeError):
    """libat_b200.so is missing or unusable."""


class NativeCallError(RuntimeError):
    """A C-ABI call returned a non-zero status."""

    def __init__(self, func: str, code: int, message: str):
        super().__init__(f"{func} failed (status {code}): {message}")
        self.func, self.code, self.message = func, code, message


class EpiSegment(Structure):
    _fields_ = [("kind", c_int32), ("in_col", c_int32), ("n_in", c_int32), ("out_col", c_int32), ("pa", c_double), ("pb", c_double)]


class EpiCol(Structure):
    _fields_ = [("lo", c_double), ("hi", c_double), ("pressure", c_double), ("flags", c_uint32), ("reserved", c_uint32)]


class GribInfo(Structure):
    """`at_grib_field_t`: packing parameters and the location of the packed values of one message."""

    _fields_ = [
        ("edition", c_int32),
        ("bits_per_value", c_int32),
        ("binary_scale", c_int32),
        ("decimal_scale", c_int32),
        ("has_bitmap", c_int32),
        ("packing", c_int32),
        ("reference_value", c_double),
        ("n_points", c_int64),
        ("n_values", c_int64),
        ("data_offset", c_int64),
        ("data_length", c_int64),
        ("bitmap_offset", c_int64),
        ("message_length", c_int64),
        ("ccsds_flags", c_int32),
        ("ccsds_block_size", c_int32),
        ("ccsds_rsi", c_int32),
        ("ccsds_pad", c_int32),
        ("complex_groups", c_int64),
        ("complex_length_ref", c_int64),
        ("complex_last_length", c_int64),
        ("complex_width_ref", c_int32),
        ("complex_width_bits", c_int32),
        ("complex_length_incr", c_int32),
        ("complex_length_bits", c_int32),
        ("complex_order", c_int32),
        ("complex_ww", c_int32),
        ("complex_refs_offset", c_int64),
        ("complex_widths_offset", c_int64),
        ("complex_lengths_offset", c_int64),
        ("complex_values_offset", c_int64),
    ]


# name -> (restype, argtypes); mirrors include/at_b200.h one to one
PROTOTYPES = {
    "at_last_error": (c_char_p, []),
    "at_version": (c_int, []),
    "at_device_count": (c_int, [POINTER(c_int)]),
    "at_set_device": (c_int, [c_int]),
    "at_device_cache_trim": (c_int, []),
    "at_host_register": (c_int, [c_void_p, c_size_t]),
    "at_host_unregister": (c_int, [c_void_p]),
    "at_csr_create": (c_int, [c_int64, c_int64, c_int64, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, POINTER(c_void_p)]),
    "at_csr_destroy": (c_int, [c_void_p]),
    "at_csr_info": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64), POINTER(c_int), POINTER(c_int)]),
    "at_spmm": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p]),
    "at_spmm_missing": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p]),
    "at_epilogue_create": (c_int, [POINTER(EpiSegment), c_int32, POINTER(EpiCol), c_int32, POINTER(c_void_p)]),
    "at_epilogue_destroy": (c_int, [c_void_p]),
    "at_spmm_fused": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "at_pointwise": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "at_gather_pointwise": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "at_transpose": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "at_gather_rows": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "at_gather_cols": (c_int, [c_void_p, c_int32, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "at_compare_mask": (c_int, [c_void_p, c_int, c_int64, c_int64, c_int, c_double, c_void_p, c_void_p]),
    "at_sum_cols": (c_int, [c_void_p, c_int32, c_int32, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "at_range_flags": (c_int, [c_void_p, c_int64, c_int64, c_int32, c_int32, c_int, c_double, c_double, c_void_p, c_void_p]),
    "at_pipeline_create": (c_int, [c_void_p, c_int32, POINTER(c_void_p)]),
    "at_pipeline_destroy": (c_int, [c_void_p]),
    "at_pipeline_regrid": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p), c_int64]),
    "at_bilinear_matrix": (c_int, [c_double, c_double, c_int64, c_double, c_double, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "at_structured_matrix": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int32, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "at_conservative_matrix_count": (c_int, [*[c_void_p] * 5, c_int64, c_int64, *[c_void_p] * 5, c_int64, c_int64, c_void_p, c_void_p]),
    "at_conservative_matrix_fill": (c_int, [*[c_void_p] * 5, c_int64, c_int64, *[c_void_p] * 5, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "at_healpix_conservative_count": (c_int, [c_int64, c_int32, *[c_void_p] * 5, c_int64, c_int64, c_int64, c_int32, *[c_void_p] * 5, c_int64, c_int64, c_void_p, c_void_p]),
    "at_healpix_conservative_fill": (c_int, [c_int64, c_int32, *[c_void_p] * 5, c_int64, c_int64, c_int64, c_int32, *[c_void_p] * 5, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "at_healpix_reorder": (c_int, [c_int64, c_int32, c_void_p, c_int64, c_void_p, c_void_p]),
    "at_pinned_alloc": (c_int, [c_size_t, POINTER(c_void_p)]),
    "at_pinned_alloc_many": (c_int, [c_size_t, c_int64, POINTER(c_void_p)]),
    "at_pinned_free": (c_int, [c_void_p]),
    "at_pinned_trim": (c_int, []),
    "at_pinned_stats": (c_int, [POINTER(c_size_t), POINTER(c_size_t)]),
    "at_hostio_create": (c_int, [c_int32, POINTER(c_void_p)]),
    "at_hostio_destroy": (c_int, [c_void_p]),
    "at_hostio_threads": (c_int, [c_void_p, POINTER(c_int32), POINTER(c_int32)]),
    "at_hostio_upload": (c_int, [c_void_p, POINTER(c_void_p), c_int64, c_int64, c_int, c_void_p, c_int64, c_void_p]),
    "at_hostio_download": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, POINTER(c_void_p), c_void_p, POINTER(c_int64)]),
    "at_hostio_wait": (c_int, [c_void_p, c_int64]),
    "at_hostio_regrid": (
        c_int,
        [c_void_p, c_int, c_void_p, c_void_p, c_int64, POINTER(c_void_p), c_int64, c_int64, c_int, c_void_p, c_int64, POINTER(c_void_p), c_void_p, POINTER(c_int64)],
    ),
    "at_grib_scan": (c_int, [c_void_p, c_size_t, POINTER(GribInfo)]),
    "at_grib_scan_many": (c_int, [POINTER(c_void_p), POINTER(c_size_t), c_int64, POINTER(GribInfo), POINTER(c_int32)]),
    "at_grib_unpack": (c_int, [c_void_p, POINTER(c_int64), POINTER(GribInfo), c_int64, c_int64, c_int, c_void_p, c_int64, c_void_p]),
    "at_hostio_upload_grib": (c_int, [c_void_p, POINTER(c_void_p), POINTER(GribInfo), c_int64, c_int64, c_int, c_void_p, c_int64, c_void_p]),
    "at_hostio_regrid_grib": (
        c_int,
        [c_void_p, c_int, c_void_p, c_void_p, c_int64, POINTER(c_void_p), POINTER(GribInfo), c_int64, c_int64, c_int, c_void_p, c_int64, POINTER(c_void_p), c_void_p, POINTER(c_int64)],
    ),
    "at_csr_replicate": (c_int, [c_void_p, c_int, POINTER(c_void_p)]),
    "at_hostio_group_create": (c_int, [c_int32, POINTER(c_int32), c_int32, POINTER(c_void_p)]),
    "at_hostio_group_destroy": (c_int, [c_void_p]),
    "at_hostio_group_regrid": (
        c_int,
        [c_void_p, c_int, POINTER(c_void_p), POINTER(c_void_p), c_int64, POINTER(c_void_p), c_int64, c_int64, c_int, POINTER(c_void_p), POINTER(c_int64)],
    ),
    "at_hostio_group_regrid_grib": (
        c_int,
        [c_void_p, c_int, POINTER(c_void_p), POINTER(c_void_p), c_int64, POINTER(c_void_p), POINTER(GribInfo), c_int64, c_int64, c_int, POINTER(c_void_p), POINTER(c_int64)],
    ),
    "at_hostio_group_wait": (c_int, [c_void_p, c_int64]),
    "at_knn_create": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_double, POINTER(c_void_p)]),
    "at_knn_destroy": (c_int, [c_void_p]),
    "at_knn_query": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "at_knn_query_gather": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_double, POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int64, c_void_p, c_void_p, c_uint64, c_void_p, c_int, c_void_p],
    ),
    "at_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), c_void_p]),
    "at_peer_free": (c_int, [c_void_p]),
    "at_peer_open": (c_int, [c_void_p, POINTER(c_void_p)]),
    "at_peer_close": (c_int, [c_void_p]),
    "at_ball_mark": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_void_p, c_void_p]),
    "at_min_nn_distance": (c_int, [c_void_p, c_int64, c_int64, POINTER(c_double), c_void_p]),
    "at_compact_mask": (c_int, [c_void_p, c_int64, c_void_p, POINTER(c_int64), c_void_p]),
    "at_cropping_mask": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_double, c_double, c_double, c_void_p, c_void_p]),
    "at_outline_classify": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "at_cutout_classify": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_double, c_double, c_int, c_void_p, c_void_p],
    ),
}

_lock = threading.Lock()
_lib = None


def library_path() -> Path:
    return Path(os.environ.get("AT_B200_LIBRARY", LIB_PATH))


def load(check_device: bool = False) -> ctypes.CDLL:
    """Load libat_b200.so (once) and declare every prototype.

    With ``check_device`` also require a usable CUDA device.
    """
    global _lib
    with _lock:
        if _lib is None:
            path = library_path()
            if not path.exists():
                raise NativeLibraryError(
                    f"{path} not found: build it with `python anemoi-transform_b200/build.py` "
                    "(this package has no CPU fallback)"
                )
            try:
                lib = ctypes.CDLL(str(path))
            except OSError as e:
                raise NativeLibraryError(f"cannot load {path}: {e}") from e
            for name, (restype, argtypes) in PROTOTYPES.items():
                try:
                    fn = getattr(lib, name)
                except AttributeError as e:
                    raise NativeLibraryError(f"{path} does not export {name}") from e
                fn.restype = restype
                fn.argtypes = argtypes
            _lib = lib
    if check_device:
        n = c_int(0)
        call("at_device_count", ctypes.byref(n))
    return _lib


def call(name: str, *args):
    """Call a status-returning entry point; raise on failure (IndexError for AT_ERR_INDEX)."""
    lib = _lib if _lib is not None else load()
    rc = getattr(lib, name)(*args)
    if rc != AT_OK:
        msg = lib.at_last_error().decode("utf-8", "replace")
        if rc == AT_ERR_INDEX:
            raise IndexError(msg)
        if rc == AT_ERR_INVALID:
            raise ValueError(f"{name}: {msg}")
        raise NativeCallError(name, rc, msg)
    return rc


def exported_symbols() -> list[str]:
    return sorted(PROTOTYPES)
