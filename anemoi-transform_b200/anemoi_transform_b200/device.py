"""Device-side objects of the hot path: thin Python owners of the C-ABI handles.

torch is used for device memory, streams and (elsewhere) torch.distributed only; every
kernel launched from here lives in libat_b200.so.
"""

from __future__ import annotations

import ctypes
import os
import re
from ctypes import byref, c_double, c_int, c_int32, c_int64, c_void_p
from typing import Iterable, Sequence

import numpy as np

from . import _cabi
from ._cabi import AT_F32, AT_F64, AT_I32, AT_I64, EpiCol, EpiSegment, call


def _torch():
    import torch

    return torch


def require_cuda():
    """Fail loudly when the CUDA path cannot run (no silent CPU fallback)."""
    torch = _torch()
    _cabi.load()
    if not torch.cuda.is_available():
        raise _cabi.NativeLibraryError("no CUDA device available: anemoi_transform_b200 has no CPU fallback")
    return torch


def stream_ptr(device: int | None = None) -> c_void_p:
    """The current stream of `device` (default: of the current device)."""
    torch = _torch()
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


DEVICES_ENV = "AT_B200_DEVICES"


def parse_devices(value: str | None, device_count: int, local_world_size: int = 1) -> list[int] | None:
    """The engines of the streamed regrid, from the value of AT_B200_DEVICES.

    None (unset or empty) keeps the single engine of the current device.  "all" is one engine
    per visible device; "0,2" a comma list of device ordinals, where an ordinal given twice is
    one more engine on that device.  Raises ValueError on anything else, on an ordinal outside
    [0, device_count), and under torchrun (local_world_size > 1), where each process already
    owns a GPU."""
    if value is None or not value.strip():
        return None
    if local_world_size > 1:
        raise ValueError(f"{DEVICES_ENV}={value!r} cannot be combined with torchrun (LOCAL_WORLD_SIZE={local_world_size}): each process already owns a GPU")
    text = value.strip()
    if text.lower() == "all":
        if device_count < 1:
            raise ValueError(f"{DEVICES_ENV}=all: no CUDA device is visible")
        return list(range(device_count))
    devices = []
    for part in text.split(","):
        part = part.strip()
        if not re.fullmatch(r"[0-9]+", part):
            raise ValueError(f"{DEVICES_ENV}={value!r}: {part!r} is not a device ordinal (expected 'all' or a comma list such as '0,1')")
        d = int(part)
        if d >= device_count:
            raise ValueError(f"{DEVICES_ENV}={value!r}: device {d} is out of range ({device_count} visible)")
        devices.append(d)
    return devices


def fanout_devices() -> list[int] | None:
    """The devices a streamed regrid deals its chunks to (AT_B200_DEVICES), or None for the
    single engine of the current device — also when only one engine is selected."""
    value = os.environ.get(DEVICES_ENV)
    if value is None or not value.strip():
        return None
    devices = parse_devices(value, _torch().cuda.device_count(), int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1))
    return devices if len(devices) > 1 else None


def _ptr(t) -> c_void_p:
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(None)


def _np_dtype_code(a: np.ndarray, kinds: dict) -> int:
    try:
        return kinds[a.dtype.type]
    except KeyError:
        raise TypeError(f"unsupported dtype {a.dtype}") from None


_FLOAT_CODES = {np.float32: AT_F32, np.float64: AT_F64}
_INT_CODES = {np.int32: AT_I32, np.int64: AT_I64}


def round_up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def empty_batch(n_rows: int, n_cols: int, dtype, device, written: int | None = None):
    """[n_rows, round_up(n_cols, 4)] without a full memset: the kernels write every real column;
    only the (at most 3) padding columns, or whatever lies beyond `written`, are zeroed."""
    torch = _torch()
    ld = round_up(n_cols, 4)
    out = torch.empty((n_rows, ld), dtype=dtype, device=device)
    first_unwritten = n_cols if written is None else written
    if first_unwritten < ld:
        out[:, first_unwritten:].zero_()
    return out


class CsrMatrix:
    """A CSR interpolation matrix staged once in HBM (reference: MIRMatrix.__init__,
    filters/fields/regrid.py:281-285)."""

    def __init__(self, data: np.ndarray, indices: np.ndarray, indptr: np.ndarray, shape: Sequence[int]):
        require_cuda()
        data = np.ascontiguousarray(data)
        indices = np.ascontiguousarray(indices)
        indptr = np.ascontiguousarray(indptr)
        if data.dtype not in (np.float32, np.float64):
            data = data.astype(np.float64)
        if indices.dtype not in (np.int32, np.int64):
            indices = indices.astype(np.int64)
        if indptr.dtype not in (np.int32, np.int64):
            indptr = indptr.astype(np.int64)
        self.shape = (int(shape[0]), int(shape[1]))
        self.nnz = int(data.shape[0])
        self.dtype = data.dtype
        if indptr.shape[0] != self.shape[0] + 1:
            raise ValueError(f"indptr has {indptr.shape[0]} entries for {self.shape[0]} rows")
        if indices.shape[0] != self.nnz:
            raise ValueError("indices and data differ in length")
        h = c_void_p()
        call(
            "at_csr_create",
            self.shape[0],
            self.shape[1],
            self.nnz,
            indptr.ctypes.data_as(c_void_p),
            _np_dtype_code(indptr, _INT_CODES),
            indices.ctypes.data_as(c_void_p),
            _np_dtype_code(indices, _INT_CODES),
            data.ctypes.data_as(c_void_p),
            _np_dtype_code(data, _FLOAT_CODES),
            byref(h),
        )
        self._h = h
        self.device = _torch().cuda.current_device()
        self._replicas: dict[int, c_void_p] = {}
        u = c_int()
        call("at_csr_info", self._h, None, None, None, byref(u), None)
        self.uniform_nnz = u.value

    @classmethod
    def from_scipy(cls, m) -> "CsrMatrix":
        m = m.tocsr()
        return cls(m.data, m.indices, m.indptr, m.shape)

    @property
    def handle(self) -> c_void_p:
        if self._h is None:
            raise RuntimeError("CsrMatrix used after close()")
        return self._h

    def handle_on(self, device: int) -> c_void_p:
        """The matrix staged on `device`: itself, or a copy made device to device the first
        time it is asked for (`at_csr_replicate`) and kept until `close()`."""
        if device == self.device:
            return self.handle
        h = self._replicas.get(device)
        if h is None:
            h = c_void_p()
            call("at_csr_replicate", self.handle, int(device), byref(h))
            self._replicas[device] = h
        return h

    def close(self) -> None:
        for h in getattr(self, "_replicas", {}).values():
            call("at_csr_destroy", h)
        self._replicas = {}
        if getattr(self, "_h", None) is not None:
            call("at_csr_destroy", self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def result_dtype(self, x_dtype):
        torch = _torch()
        if self.dtype == np.float64 or x_dtype == torch.float64:
            return torch.float64
        return torch.float32

    def apply(self, X, n_fields: int | None = None, out=None, variant: int = 0, missing: int = 0):
        """Y[n_rows, ld] = A · X[n_cols, ld]  (point-major batches, torch CUDA tensors).

        `missing`: a missing-value policy code (`_cabi.MISSING_*`); nonzero skips NaN sources
        and renormalises the weights (`at_spmm_missing`, default kernel shape)."""
        torch = _torch()
        if X.dim() != 2 or X.shape[0] != self.shape[1]:
            raise ValueError(f"X has shape {tuple(X.shape)}, expected [{self.shape[1]}, fields]")
        if X.stride(1) != 1:
            raise ValueError("X must be row-major (unit stride along fields)")
        if missing and variant:
            raise ValueError("a kernel variant applies to the plain SpMM only, not with a missing-value policy")
        n_fields = X.shape[1] if n_fields is None else n_fields
        ydt = self.result_dtype(X.dtype)
        if out is None:
            out = torch.empty((self.shape[0], X.shape[1]), dtype=ydt, device=X.device)
        code = {torch.float32: AT_F32, torch.float64: AT_F64}
        call(
            "at_spmm_missing" if missing else "at_spmm",
            self.handle,
            _ptr(X),
            code[X.dtype],
            X.stride(0),
            _ptr(out),
            code[out.dtype],
            out.stride(0),
            n_fields,
            missing if missing else variant,
            stream_ptr(),
        )
        return out


class Epilogue:
    """A fused pointwise program (segments + per-output-column parameters)."""

    def __init__(self, segments: Iterable[tuple], cols: Iterable[tuple[float, float, float, int]]):
        """segments: (kind, in_col, n_in, out_col[, pa, pb]); cols: (lo, hi, pressure, flags) per output column."""
        require_cuda()
        segs = [tuple(s) + (0.0, 0.0)[len(s) - 4 :] for s in segments]
        cols = list(cols)
        seg_arr = (EpiSegment * len(segs))(*[EpiSegment(int(s[0]), int(s[1]), int(s[2]), int(s[3]), float(s[4]), float(s[5])) for s in segs])
        col_arr = (EpiCol * len(cols))(*[EpiCol(float(lo), float(hi), float(p), int(fl), 0) for lo, hi, p, fl in cols])
        h = c_void_p()
        call("at_epilogue_create", seg_arr, len(segs), col_arr, len(cols), byref(h))
        self._h = h
        self.n_out_cols = len(cols)
        self.n_in_cols = max(s[1] + s[2] for s in segs)

    @property
    def handle(self) -> c_void_p:
        return self._h

    def close(self) -> None:
        if getattr(self, "_h", None) is not None:
            call("at_epilogue_destroy", self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def apply(self, X, out=None, row_mask=None, gather=None):
        """Y = epilogue(X) on a resident point-major batch — or, with `gather` (device int64
        indices, every entry a valid row of X), Y[r] = epilogue(X[gather[r]])."""
        torch = _torch()
        if X.shape[1] < self.n_in_cols:
            raise ValueError(f"the epilogue reads {self.n_in_cols} input columns, X has {X.shape[1]}")
        n_rows = X.shape[0] if gather is None else int(gather.shape[0])
        if out is None:
            out = empty_batch(n_rows, self.n_out_cols, X.dtype, X.device)
        code = {torch.float32: AT_F32, torch.float64: AT_F64}[X.dtype]
        if gather is None:
            call("at_pointwise", self.handle, n_rows, _ptr(X), X.stride(0), _ptr(out), out.stride(0), code, _ptr(row_mask), stream_ptr())
        else:
            if gather.dtype != torch.int64 or not gather.is_contiguous():
                raise ValueError("gather must be a contiguous int64 CUDA tensor")
            call("at_gather_pointwise", self.handle, _ptr(gather), n_rows, X.shape[0], _ptr(X), X.stride(0), _ptr(out), out.stride(0), code, _ptr(row_mask), stream_ptr())
        return out

    def apply_fused(self, csr: CsrMatrix, X, out=None, row_mask=None):
        """Y = epilogue(A · X)."""
        torch = _torch()
        if X.dim() != 2 or X.shape[0] != csr.shape[1]:
            raise ValueError(f"dimension mismatch: matrix has {csr.shape[1]} columns, X has shape {tuple(X.shape)}")
        if X.shape[1] < self.n_in_cols:
            raise ValueError(f"the epilogue reads {self.n_in_cols} input columns, X has {X.shape[1]}")
        if X.dtype != torch.float32 or X.stride(1) != 1:
            raise ValueError("apply_fused: X must be a row-major float32 batch")
        if out is None:
            out = empty_batch(csr.shape[0], self.n_out_cols, torch.float32, X.device)
        call("at_spmm_fused", csr.handle, self.handle, _ptr(X), X.shape[0], X.stride(0), _ptr(out), out.stride(0), _ptr(row_mask), stream_ptr())
        return out


class KnnIndex:
    """Bucketed search structure over float64 xyz sources (replaces cKDTree(points))."""

    def __init__(self, xyz, cell_size: float = 0.0):
        """xyz: tuple of three float64 arrays (numpy on host or torch CUDA tensors)."""
        torch = require_cuda()
        x, y, z = xyz
        if isinstance(x, torch.Tensor):
            x, y, z = (t.contiguous().to(torch.float64) for t in (x, y, z))
            self.n = int(x.shape[0])
            ptrs = (_ptr(x), _ptr(y), _ptr(z))
            on_device = 1
            torch.cuda.current_stream().synchronize()
        else:
            x, y, z = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, z))
            self.n = int(x.shape[0])
            ptrs = tuple(a.ctypes.data_as(c_void_p) for a in (x, y, z))
            on_device = 0
        h = c_void_p()
        call("at_knn_create", *ptrs, self.n, on_device, float(cell_size), byref(h))
        self._h = h

    def close(self) -> None:
        if getattr(self, "_h", None) is not None:
            call("at_knn_destroy", self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def query(self, qxyz, k: int = 1, distance_upper_bound: float = float("inf"), want_ties: bool = False):
        """→ (idx int64[nq,k], dist float64[nq,k], ties uint8[nq] | None), CUDA tensors."""
        torch = _torch()
        qx, qy, qz = (to_device_f64(a) for a in qxyz)
        nq = int(qx.shape[0])
        idx = torch.empty((nq, k), dtype=torch.int64, device=qx.device)
        dist = torch.empty((nq, k), dtype=torch.float64, device=qx.device)
        ties = torch.empty((nq,), dtype=torch.uint8, device=qx.device) if want_ties else None
        call("at_knn_query", self._h, _ptr(qx), _ptr(qy), _ptr(qz), nq, int(k), float(distance_upper_bound), _ptr(idx), _ptr(dist), _ptr(ties), stream_ptr())
        return idx, dist, ties

    def ball_mark(self, qxyz, r: float, mark=None):
        """mark[j] |= any query within r of source j.  → uint8[n] CUDA tensor."""
        torch = _torch()
        qx, qy, qz = (to_device_f64(a) for a in qxyz)
        if mark is None:
            mark = torch.zeros((self.n,), dtype=torch.uint8, device=qx.device)
        call("at_ball_mark", self._h, _ptr(qx), _ptr(qy), _ptr(qz), int(qx.shape[0]), float(r), _ptr(mark), stream_ptr())
        return mark

    def min_nn_distance(self, first: int = 0, count: int = -1) -> float:
        """min over sources [first, first+count) of the distance to their 2nd nearest source."""
        out = c_double()
        call("at_min_nn_distance", self._h, int(first), int(count), byref(out), stream_ptr())
        return out.value


def to_device_f64(a):
    torch = _torch()
    if isinstance(a, torch.Tensor):
        return a.to(device="cuda", dtype=torch.float64).contiguous()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def compact_mask(mark):
    """Sorted int64 indices of the non-zero bytes of a uint8 CUDA tensor."""
    torch = _torch()
    n = int(mark.shape[0])
    out = torch.empty((max(n, 1),), dtype=torch.int64, device=mark.device)
    count = c_int64()
    call("at_compact_mask", _ptr(mark), n, _ptr(out), byref(count), stream_ptr())
    return out[: count.value]


def cropping_mask_device(lats, lons, north, west, south, east):
    torch = _torch()
    la, lo = to_device_f64(lats), to_device_f64(lons)
    mask = torch.empty((la.shape[0],), dtype=torch.uint8, device=la.device)
    call("at_cropping_mask", _ptr(la), _ptr(lo), int(la.shape[0]), float(north), float(west), float(south), float(east), _ptr(mask), stream_ptr())
    return mask


def transpose(src, out=None):
    """out[c, r] = src[r, c] for 2-D CUDA tensors of 4- or 8-byte elements."""
    torch = _torch()
    rows, cols = src.shape
    if src.stride(1) != 1:
        raise ValueError("transpose: source must have unit stride along its last axis")
    if out is None:
        out = torch.empty((cols, rows), dtype=src.dtype, device=src.device)
    call("at_transpose", _ptr(src), rows, cols, src.stride(0), _ptr(out), out.stride(0), src.element_size(), stream_ptr())
    return out


def gather_rows(X, idx, n_fields: int | None = None, out=None):
    """out[i, :] = X[idx[i], :] (numpy's data[..., idx] on a point-major batch)."""
    torch = _torch()
    idx = idx.to(device=X.device, dtype=torch.int64).contiguous()
    n_out = int(idx.shape[0])
    n_fields = X.shape[1] if n_fields is None else n_fields
    if out is None:
        # whole 16-byte chunks are copied, padding columns included, when the layout allows it:
        # the same test as at_gather_rows (empty_batch's rows are 16-byte aligned), so that a
        # misaligned column view of X does not leave the padding columns unwritten
        per16 = 16 // X.element_size()
        vec16 = X.stride(0) % per16 == 0 and X.data_ptr() % 16 == 0
        out = empty_batch(n_out, X.shape[1], X.dtype, X.device, written=min(X.shape[1], round_up(n_fields, per16)) if vec16 else n_fields)
    err = torch.zeros((1,), dtype=torch.int32, device=X.device)
    call("at_gather_rows", _ptr(idx), n_out, X.shape[0], _ptr(X), X.stride(0), _ptr(out), out.stride(0), n_fields, X.element_size(), _ptr(err), stream_ptr())
    if int(err.item()) != 0:
        raise IndexError(f"index out of bounds for axis with size {X.shape[0]}")
    return out


def gather_cols(X, cols: Sequence[int], out=None):
    """out[:, j] = X[:, cols[j]] — regroup the fields of a resident point-major batch."""
    torch = _torch()
    n_out = len(cols)
    if any(c < 0 or c >= X.shape[1] for c in cols):
        raise IndexError("column index out of range")
    if out is None:
        out = empty_batch(X.shape[0], n_out, X.dtype, X.device)
    index = torch.tensor(list(cols), dtype=torch.int32, device=X.device)
    call("at_gather_cols", _ptr(index), n_out, X.shape[0], _ptr(X), X.stride(0), _ptr(out), out.stride(0), X.element_size(), stream_ptr())
    return out


def sum_cols(X, cols: Sequence[int], n_groups: int, n_terms: int, out=None):
    """out[:, g] = X[:, cols[g*n_terms]] + X[:, cols[g*n_terms+1]] + … (sequential, X's dtype)."""
    torch = _torch()
    if len(cols) != n_groups * n_terms or any(c < 0 or c >= X.shape[1] for c in cols):
        raise IndexError("sum_cols: bad column list")
    if out is None:
        out = empty_batch(X.shape[0], n_groups, X.dtype, X.device)
    index = torch.tensor(list(cols), dtype=torch.int32, device=X.device)
    code = AT_F32 if X.dtype == torch.float32 else AT_F64
    call("at_sum_cols", _ptr(index), n_groups, n_terms, X.shape[0], _ptr(X), X.stride(0), _ptr(out), out.stride(0), code, stream_ptr())
    return out


def range_flags(X, first_col: int, n_cols: int, lo: float, hi: float) -> list[int]:
    """Per column: bit 0 any value < lo, bit 1 any value > hi, bit 2 any NaN."""
    torch = _torch()
    flags = torch.zeros((max(n_cols, 1),), dtype=torch.int32, device=X.device)
    code = AT_F32 if X.dtype == torch.float32 else AT_F64
    call("at_range_flags", _ptr(X), X.stride(0), X.shape[0], int(first_col), int(n_cols), code, float(lo), float(hi), _ptr(flags), stream_ptr())
    return [int(v) for v in flags[:n_cols].cpu().tolist()]


def compare_mask(values, op: int, threshold: float):
    """uint8 mask = OP(values, threshold) for a 1-D (possibly strided) float CUDA tensor.

    As numpy compares an array with a Python float (NEP 50): in the array's own float dtype,
    in float64 for integer and bool arrays."""
    torch = _torch()
    if values.dtype == torch.float16:
        # float16 values widen to float64 exactly; the threshold is rounded to float16 first
        with np.errstate(over="ignore"):
            threshold = float(np.float16(threshold))
    if values.dtype not in (torch.float32, torch.float64):
        values = values.to(torch.float64)
    n = int(values.shape[0])
    mask = torch.empty((n,), dtype=torch.uint8, device=values.device)
    code = AT_F32 if values.dtype == torch.float32 else AT_F64
    call("at_compare_mask", _ptr(values), code, values.stride(0) if n > 1 else 1, n, int(op), float(threshold), _ptr(mask), stream_ptr())
    return mask


# ---------------------------------------------------------------- host <-> device -------
class PinnedBlock:
    """A block of the library's page-locked host pool, exposed to numpy through the array
    interface; the block returns to the pool when the last array viewing it is collected."""

    __slots__ = ("ptr", "nbytes", "__array_interface__", "__weakref__")

    def __init__(self, ptr: int, nbytes: int):
        self.ptr, self.nbytes = ptr, nbytes
        self.__array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}

    def __del__(self):
        try:
            _cabi.load().at_pinned_free(c_void_p(self.ptr))
        except Exception:  # interpreter shutdown
            pass


def _array_on_block(ptr: int, n: int, dtype) -> np.ndarray:
    dtype = np.dtype(dtype)
    return np.asarray(PinnedBlock(ptr, n * dtype.itemsize)).view(dtype)


def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
    """np.empty in page-locked host memory (a block of the library's pool): uploads of such
    arrays and downloads into them are DMA-ed in place, without a staging copy.  Decoders that
    feed the filters of this package can allocate their field arrays here."""
    require_cuda()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape))
    p = c_void_p()
    call("at_pinned_alloc", max(1, n * dtype.itemsize), byref(p))
    return _array_on_block(p.value, n, dtype).reshape(shape)


def pinned_fields(n_fields: int, n_points: int, dtype) -> tuple[list[np.ndarray] | None, object]:
    """n_fields pool arrays of n_points elements and the ctypes pointer array naming them, or
    (None, None) when the pool is exhausted (callers then use ordinary numpy memory)."""
    dtype = np.dtype(dtype)
    ptrs = (c_void_p * n_fields)()
    try:
        call("at_pinned_alloc_many", max(1, n_points * dtype.itemsize), n_fields, ptrs)
    except _cabi.NativeCallError as e:
        if e.code != _cabi.AT_ERR_NOMEM:
            raise
        return None, None
    return [_array_on_block(ptrs[j], n_points, dtype) for j in range(n_fields)], ptrs


def pinned_pool_stats() -> tuple[int, int]:
    """(bytes in use, bytes reserved) of the page-locked pool."""
    from ctypes import c_size_t

    a, b = c_size_t(), c_size_t()
    call("at_pinned_stats", byref(a), byref(b))
    return a.value, b.value


def pinned_pool_trim() -> None:
    call("at_pinned_trim")


def _host_ptr(a: np.ndarray) -> int:
    return a.__array_interface__["data"][0]


def _pointer_array(arrays: Sequence[np.ndarray]):
    return (c_void_p * len(arrays))(*[a.__array_interface__["data"][0] for a in arrays])


class HostIO:
    """Owner of the process's `at_hostio_t` engine of one device (by default the current one)."""

    _engines: dict[int, "HostIO"] = {}

    def __init__(self, n_threads: int = 0):
        torch = require_cuda()
        self.device = torch.cuda.current_device()
        h = c_void_p()
        call("at_hostio_create", int(n_threads), byref(h))
        self._h = h
        from ctypes import c_int32

        t, nt = c_int32(), c_int32()
        call("at_hostio_threads", self._h, byref(t), byref(nt))
        self.n_threads, self.nontemporal = t.value, bool(nt.value)

    @classmethod
    def get(cls, device: int | None = None) -> "HostIO":
        torch = require_cuda()
        dev = torch.cuda.current_device() if device is None else int(device)
        io = cls._engines.get(dev)
        if io is None:
            n = int(os.environ.get("AT_B200_COPY_THREADS", 0))
            local = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
            if n <= 0 and local > 1:
                # several ranks on one box share its cores: an equal share each (the native call
                # runs on a helper thread that stages too; the Python thread mostly waits)
                n = max(1, min(8, len(os.sched_getaffinity(0)) // local))
            with torch.cuda.device(dev):
                io = cls._engines[dev] = cls(n)  # 0: one staging thread per physical core
        return io

    @property
    def handle(self) -> c_void_p:
        return self._h

    def upload(self, arrays: Sequence[np.ndarray], pm, col0: int = 0) -> None:
        """pm[:, col0 + j] = arrays[j] (contiguous 1-D host arrays of pm's dtype)."""
        n = len(arrays)
        if n == 0:
            return
        esz = pm.element_size()
        call("at_hostio_upload", self._h, _pointer_array(arrays), n, int(arrays[0].size), esz, c_void_p(pm.data_ptr() + col0 * esz), pm.stride(0), stream_ptr())

    def download(self, pm, col0: int, dests: Sequence[np.ndarray], ptrs=None) -> int:
        """dests[j][:] = pm[:, col0 + j]; → ticket (-1 when already complete)."""
        n = len(dests)
        if n == 0:
            return -1
        esz = pm.element_size()
        ticket = c_int64(-1)
        call("at_hostio_download", self._h, c_void_p(pm.data_ptr() + col0 * esz), pm.stride(0), n, int(pm.shape[0]), esz, ptrs if ptrs is not None else _pointer_array(dests), stream_ptr(self.device), byref(ticket))
        return ticket.value

    def wait(self, ticket: int) -> None:
        if ticket >= 0:
            call("at_hostio_wait", self._h, ticket)


class HostIOGroup:
    """Owner of an `at_hostio_group_t`: one engine per entry of `devices` and one pool of
    staging threads for all of them (the streamed regrid over several GPUs)."""

    _groups: dict[tuple[int, ...], "HostIOGroup"] = {}

    def __init__(self, devices: Sequence[int]):
        require_cuda()
        self.devices = tuple(int(d) for d in devices)
        h = c_void_p()
        call("at_hostio_group_create", len(self.devices), (c_int32 * len(self.devices))(*self.devices), 0, byref(h))
        self._h = h

    @classmethod
    def get(cls, devices: Sequence[int]) -> "HostIOGroup":
        key = tuple(int(d) for d in devices)
        group = cls._groups.get(key)
        if group is None:
            group = cls._groups[key] = cls(key)
        return group

    @property
    def handle(self) -> c_void_p:
        return self._h

    def wait(self, ticket: int) -> None:
        if ticket >= 0:
            call("at_hostio_group_wait", self._h, ticket)


class Transfer:
    """An asynchronous device-to-host transfer: a ticket of the engine (or group) that issued it."""

    __slots__ = ("ticket", "done", "engine")

    def __init__(self, ticket: int, engine: "HostIO | HostIOGroup"):
        self.ticket, self.done, self.engine = ticket, ticket < 0, engine

    def wait(self) -> None:
        if not self.done:
            self.done = True
            self.engine.wait(self.ticket)


class DeviceBatch:
    """A batch of fields resident in HBM, point-major: data[n_points, ld], ld % 4 == 0.

    Host copies of the columns (`_host`) appear when they are first needed — or ahead of need,
    when a filter knows its results are headed for the host (`prefetch`, the streamed regrid)
    — as arrays of the page-locked pool that the DMA engine fills directly; `_ticket[j]` is the
    transfer column j's array is waiting for."""

    #: host bytes fetched per lazy download (a reader walking the columns misses once per window)
    window_bytes = 256 << 20

    def __init__(self, data, n_fields: int):
        self.data = data
        self.n_fields = int(n_fields)
        self._host: list | None = None
        self._ticket: list[Transfer | None] | None = None
        self._n_points = int(data.shape[0]) if data is not None else 0
        self._dtype = None

    @property
    def n_points(self) -> int:
        return int(self.data.shape[0]) if self.data is not None else self._n_points

    @property
    def resident(self) -> bool:
        return self.data is not None

    @classmethod
    def from_host_fields(cls, arrays: Sequence[np.ndarray], chunk: int | None = None) -> "DeviceBatch":
        """Upload F host fields (each [n_points]) and pack them point-major (`at_hostio_upload`:
        worker threads stage pageable arrays into pinned slots, one H2D per piece, one
        `at_transpose` per chunk; page-locked arrays are read in place).  All fields take the
        batch's dtype — the widest of theirs; callers that must keep per-field dtypes batch
        runs of equal dtype (`batching.group_by_dtype`)."""
        torch = require_cuda()
        n_fields = len(arrays)
        if n_fields == 0:
            raise ValueError("empty batch")
        views = [np.asarray(a).reshape(-1) for a in arrays]
        n_points = int(views[0].size)
        dtype = np.result_type(*{v.dtype for v in views})
        if dtype not in (np.float32, np.float64):
            dtype = np.dtype(np.float64)
        tdtype = torch.float32 if dtype == np.float32 else torch.float64
        for i, v in enumerate(views):
            if v.size != n_points:
                raise ValueError(f"field {i} has {v.size} points, expected {n_points}")
        views = [v if (v.dtype == dtype and v.flags.c_contiguous) else np.ascontiguousarray(v, dtype=dtype) for v in views]
        pm = empty_batch(n_points, n_fields, tdtype, "cuda")
        HostIO.get().upload(views, pm)
        return cls(pm, n_fields)

    def _np_dtype(self):
        if self.data is None:
            return self._dtype
        return np.dtype(np.float32 if self.data.dtype == _torch().float32 else np.float64)

    # -- host copies ----------------------------------------------------------------------
    def _ensure_host_lists(self) -> None:
        if self._host is None:
            self._host = [None] * self.n_fields
            self._ticket = [None] * self.n_fields

    def _start_download(self, first: int, count: int) -> None:
        """Begin moving columns [first, first + count) that have no host copy yet into pool
        arrays (asynchronous); pageable arrays when the pool is exhausted (synchronous)."""
        self._ensure_host_lists()
        cols = [j for j in range(first, first + count) if self._host[j] is None]
        io = HostIO.get(self.data.device.index)
        # runs of consecutive columns go in one call
        run: list[int] = []
        for j in cols + [-1]:
            if run and j == run[-1] + 1:
                run.append(j)
                continue
            if run:
                arrays, ptrs = pinned_fields(len(run), self.n_points, self._np_dtype())
                if arrays is None:
                    arrays, ptrs = [np.empty((self.n_points,), dtype=self._np_dtype()) for _ in run], None
                transfer = Transfer(io.download(self.data, run[0], arrays, ptrs), io)
                for k, c in enumerate(run):
                    self._host[c], self._ticket[c] = arrays[k], transfer
            run = [j] if j >= 0 else []

    def adopt_host_arrays(self, arrays: Sequence[np.ndarray], transfer: "Transfer") -> None:
        """Host copies produced together with the batch (the streamed regrid's outputs)."""
        self._host = list(arrays)
        self._ticket = [transfer] * len(arrays)
        if self.data is None and arrays:
            self._n_points, self._dtype = int(arrays[0].size), arrays[0].dtype

    def prefetch(self) -> None:
        """Start the download of every column now: the caller expects `to_numpy()` soon."""
        if self.data is not None:
            self._start_download(0, self.n_fields)

    def prefetch_columns(self, cols: Sequence[int]) -> None:
        """`prefetch` of the listed (sorted) columns only — a fused launch leaves padding
        columns between its segments that belong to no field."""
        if self.data is None or not cols:
            return
        start = prev = cols[0]
        for c in list(cols[1:]) + [None]:
            if c is not None and c == prev + 1:
                prev = c
                continue
            self._start_download(start, prev - start + 1)
            if c is not None:
                start = prev = c

    def _wait(self, col: int) -> None:
        t = self._ticket[col]
        if t is not None:
            t.wait()

    def _wait_all(self) -> None:
        if self._ticket:
            for t in {id(t): t for t in self._ticket if t is not None and not t.done}.values():
                t.wait()

    def __del__(self):
        # a DMA still writing into pool arrays must finish before they are recycled
        try:
            self._wait_all()
        except Exception:
            pass

    def to_host_fields(self, chunk: int | None = None) -> np.ndarray:
        """→ numpy [n_fields, n_points] (field-major), a fresh array."""
        host = np.empty((self.n_fields, self.n_points), dtype=self._np_dtype())
        if self.data is None:
            self._wait_all()
            for j in range(self.n_fields):
                host[j] = self._host[j]
            return host
        HostIO.get(self.data.device.index).download(self.data, 0, [host[j] for j in range(self.n_fields)])
        return host

    def offload(self) -> None:
        """Move the batch to host memory and free its HBM (used when a FieldList is larger than
        the device: outputs of finished sub-batches must not pile up in HBM).  From then on
        `take_column` hands out copies of the host arrays."""
        if self.data is None:
            return
        self._start_download(0, self.n_fields)
        self._wait_all()
        self._n_points, self._dtype = self.n_points, self._np_dtype()
        self.data = None

    def take_column(self, col: int) -> np.ndarray:
        """A fresh host array with the values of column `col`, owned by the caller.

        A column without a host copy triggers the download of a window of columns starting at
        it (not of the whole batch); each array is handed out once without a further copy.  A
        column asked for again is downloaded again (the device copy is the source of truth —
        callers may mutate what they were given, e.g. apply_mask.py:184-185)."""
        if not 0 <= col < self.n_fields:
            raise IndexError(f"column {col} of a batch of {self.n_fields} fields")
        if self.data is None:  # offloaded: the host arrays are the only copy
            self._wait(col)
            return self._host[col].copy()
        self._ensure_host_lists()
        if self._host[col] is None:
            per_field = max(1, self.n_points * self.data.element_size())
            self._start_download(col, min(self.n_fields - col, max(1, self.window_bytes // per_field)))
        self._wait(col)
        arr, self._host[col] = self._host[col], None
        return arr

    def host_column(self, col: int) -> np.ndarray:
        return self.take_column(col)

    def locate(self, col: int) -> tuple["DeviceBatch", int]:
        """(batch, column) of output `col` — itself (see pointwise.SplitOutput)."""
        return self, col


_HOST_BOUND = [True]


def results_are_host_bound() -> bool:
    """Whether a filter should start moving its results to the host as it produces them (the
    caller of a stand-alone `forward` reads them next) or leave them in HBM for the next
    filter of a pipeline."""
    return _HOST_BOUND[0]


class results_stay_on_device:
    """Context of the non-final filters of a `Pipeline`: no eager download of their results."""

    def __enter__(self):
        self._saved, _HOST_BOUND[0] = _HOST_BOUND[0], False

    def __exit__(self, *exc):
        _HOST_BOUND[0] = self._saved


class StreamedRegrid:
    """One `at_hostio_regrid` job: host fields in, a `DeviceBatch` with host copies out.

    The native call runs on a helper thread (it releases the GIL for its whole duration), so
    the caller can build the output FieldList while the fields stream through the GPU;
    `join()` returns once every input byte has been consumed — the results keep arriving in
    their pool arrays behind the batch's transfer.

    `devices` (more than one entry): the job runs on the engines of a `HostIOGroup`
    (`at_hostio_group_regrid`), which deals chunks of fields to those devices; `index` is then
    one device index per entry, and the results go to the host only."""

    def __init__(self, op: int, csr: "CsrMatrix | None", index, n_tgt: int, y_dtype, arrays: Sequence[np.ndarray], keep_resident: bool, to_host: bool, devices: Sequence[int] | None = None):
        import threading

        torch = require_cuda()
        if not (keep_resident or to_host):
            raise ValueError("StreamedRegrid: nothing to produce")
        if devices is not None and (keep_resident or not to_host):
            raise ValueError("StreamedRegrid: a job over several devices produces host results only")
        # `arrays` is either the fields' host values or a grib.PackedFields (messages decoded on
        # the device: at_hostio_regrid_grib)
        packed = arrays if hasattr(arrays, "infos") else None
        n = packed.n_fields if packed is not None else len(arrays)
        n_src = packed.n_points if packed is not None else int(arrays[0].size)
        x_np = packed.dtype if packed is not None else arrays[0].dtype
        y_np = np.dtype(np.float32 if y_dtype == torch.float32 else np.float64)
        self._io = HostIO.get() if devices is None else HostIOGroup.get(devices)
        self._keep = (arrays, csr, index)  # alive until the native call returns
        data = empty_batch(n_tgt, n, y_dtype, "cuda") if keep_resident else None
        self.batch = DeviceBatch(data, n)
        if data is None:
            self.batch._n_points, self.batch._dtype = n_tgt, y_np
        self._out, out_ptrs, pooled = None, None, False
        if to_host:
            # raw pool blocks now, numpy views on them once the native call is running
            out_ptrs = (c_void_p * n)()
            try:
                call("at_pinned_alloc_many", max(1, n_tgt * y_np.itemsize), n, out_ptrs)
                pooled = True
            except _cabi.NativeCallError as e:
                if e.code != _cabi.AT_ERR_NOMEM:
                    raise
                # pool exhausted: pageable destinations, filled synchronously
                self._out = [np.empty((n_tgt,), dtype=y_np) for _ in range(n)]
                out_ptrs = _pointer_array(self._out)
        self._ticket = c_int64(-1)
        self._error: BaseException | None = None
        inputs = (packed.pointers, packed.infos) if packed is not None else (_pointer_array(arrays),)
        x_code = AT_F32 if x_np == np.float32 else AT_F64
        if devices is not None:
            n_eng = len(devices)
            csrs = (c_void_p * n_eng)(*[csr.handle_on(d).value for d in devices]) if csr is not None else None
            indices = (c_void_p * n_eng)(*[t.data_ptr() for t in index]) if index is not None else None
            args = ("at_hostio_group_regrid_grib" if packed is not None else "at_hostio_group_regrid", self._io.handle, int(op), csrs, indices, int(n_tgt), *inputs, n, n_src, x_code, out_ptrs, byref(self._ticket))
        else:
            args = (
                "at_hostio_regrid_grib" if packed is not None else "at_hostio_regrid",
                self._io.handle,
                int(op),
                csr.handle if csr is not None else None,
                _ptr(index),
                int(n_tgt),
                *inputs,
                n,
                n_src,
                x_code,
                _ptr(data),
                int(data.stride(0)) if data is not None else 0,
                out_ptrs,
                stream_ptr(),
                byref(self._ticket),
            )

        def run():
            try:
                call(*args)
            except BaseException as e:  # re-raised by join()
                self._error = e

        self._thread = threading.Thread(target=run, name="at-regrid-stream", daemon=True)
        self._thread.start()
        if pooled:
            self._out = [_array_on_block(out_ptrs[j], n_tgt, y_np) for j in range(n)]

    def join(self) -> DeviceBatch:
        self._thread.join()
        self._keep = None
        if self._error is not None:
            raise self._error
        if self._out is not None:
            self.batch.adopt_host_arrays(self._out, Transfer(self._ticket.value, self._io))
        return self.batch


class HostPipeline:
    """Streaming regrid of host-resident fields (at_pipeline_*)."""

    def __init__(self, csr: CsrMatrix, chunk_fields: int = 64):
        require_cuda()
        self.csr = csr
        h = c_void_p()
        call("at_pipeline_create", csr.handle, int(chunk_fields), byref(h))
        self._h = h

    def close(self) -> None:
        if getattr(self, "_h", None) is not None:
            call("at_pipeline_destroy", self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def regrid(self, fields_in: Sequence[np.ndarray], fields_out: Sequence[np.ndarray] | None = None) -> list[np.ndarray]:
        n = len(fields_in)
        n_src, n_tgt = self.csr.shape[1], self.csr.shape[0]
        ins = []
        for i, a in enumerate(fields_in):
            a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1)
            if a.size != n_src:
                raise ValueError(f"field {i} has {a.size} points, matrix expects {n_src}")
            ins.append(a)
        if fields_out is None:
            fields_out = [np.empty((n_tgt,), dtype=np.float32) for _ in range(n)]
        for i, a in enumerate(fields_out):
            if a.dtype != np.float32 or a.size != n_tgt or not a.flags.c_contiguous:
                raise ValueError(f"output field {i} must be contiguous float32[{n_tgt}]")
        in_ptrs = (c_void_p * n)(*[a.ctypes.data for a in ins])
        out_ptrs = (c_void_p * n)(*[a.ctypes.data for a in fields_out])
        call("at_pipeline_regrid", self._h, in_ptrs, out_ptrs, n)
        return list(fields_out)
