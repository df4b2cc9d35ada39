"""`regrid` — reference `filters/fields/regrid.py:87-516`.

Same constructor arguments, same interpolator precedence (matrix > mask > method=="nearest"
> earthkit, `_interpolator` 432-467) and the same output wrapping
(`NewLatLonField(NewMetadataField(NewDataField…))`, regrid.py:312).  What changes is where
the arithmetic runs: the per-field Python loop of `_interpolate` (regrid.py:204-208) becomes
one batched device pass —

    MIRMatrix                     CSR staged once in HBM, `at_spmm` over all fields
                                  (`at_spmm_missing` with `missing_values=`)
    ScipyKDTreeNearestNeighbours  `spatial.nearest_grid_points` (device kNN) + `at_gather_rows`
    MaskedRegrid                  `at_gather_rows` with the mask's indices

Host fields are uploaded in chunks and packed point-major; fields already resident in HBM
(outputs of another filter of this package) are used in place.  Outputs stay resident and
are downloaded when `to_numpy()` is first called.

With AT_B200_DEVICES naming more than one engine (`device.parse_devices`), the streamed route
— host fields in, results headed to the host — deals its chunks to several GPUs from this one
process (`at_hostio_group_regrid`); its results are then host arrays only.  The batch route,
fused pipelines, kNN and the masks stay on the current device.
"""

from __future__ import annotations

import logging
from typing import Any

import numpy as np

from ... import ekd
from ... import grib
from ...batching import fields_to_batch
from ... import _cabi
from ...device import CsrMatrix, DeviceBatch, StreamedRegrid, fanout_devices, gather_rows, require_cuda, results_are_host_bound
from ...fields import new_field_from_device_column, new_field_from_latitudes_longitudes, new_fieldlist_from_list
from ...filter import Filter
from . import filter_registry

LOG = logging.getLogger(__name__)

#: `missing_values=` of `regrid` -> the policy of `at_spmm_missing` (the names are MIR's
#: `nonlinear` options; the semantics are this package's, see DESIGN.md §3.11)
MISSING_VALUES = {
    "propagate": _cabi.MISSING_PROPAGATE,
    "missing-if-all-missing": _cabi.MISSING_ALL,
    "missing-if-heaviest-missing": _cabi.MISSING_HEAVIEST,
}
_MATRIX_OPS = {
    _cabi.MISSING_PROPAGATE: _cabi.HOSTIO_SPMM,
    _cabi.MISSING_ALL: _cabi.HOSTIO_SPMM_MISSING_ALL,
    _cabi.MISSING_HEAVIEST: _cabi.HOSTIO_SPMM_MISSING_HEAVIEST,
}


def missing_policy(missing_values: str | None) -> int:
    """The policy code of a `missing_values` argument (None: "propagate")."""
    name = "propagate" if missing_values is None else missing_values
    if not isinstance(name, str) or name not in MISSING_VALUES:
        raise ValueError(f"regrid: missing_values={missing_values!r} is not one of {tuple(MISSING_VALUES)}")
    return MISSING_VALUES[name]


def _free_device_bytes() -> int:
    """HBM this process can still use, from torch's own counters (cudaMemGetInfo takes tens of
    milliseconds on a 180 GB device — too slow for every forward call)."""
    torch = require_cuda()
    total = torch.cuda.get_device_properties(torch.cuda.current_device()).total_memory
    return int(0.95 * total - torch.cuda.memory_allocated())


def as_gridspec(grid: Any) -> dict[str, Any] | None:
    if grid is None:
        return None
    if isinstance(grid, (str, list, tuple)):
        return {"grid": grid}
    return grid


def as_griddata(grid: Any) -> dict[str, Any] | None:
    """Grid given as a field, a {latitudes, longitudes} dict, a named grid or a gridspec dict
    ({"grid": "H128", "ordering": "nested"}, `grids.lookup`)."""
    if grid is None:
        return None
    if isinstance(grid, ekd.Field) or (hasattr(grid, "grid_points") and hasattr(grid, "to_numpy")):
        lat, lon = grid.grid_points()
        return dict(latitudes=lat, longitudes=lon)
    if isinstance(grid, dict) and "latitudes" in grid and "longitudes" in grid:
        return grid
    if isinstance(grid, (str, list, tuple)) or (isinstance(grid, dict) and "grid" in grid):
        from ...grids import lookup

        return lookup(grid)
    raise ValueError(f"Invalid grid: {grid}")


@filter_registry.register("regrid")
class RegridFilter(Filter):
    """Regrid fields with a precomputed matrix, a nearest-neighbour search or an index mask."""

    def __init__(
        self,
        *,
        in_grid: Any | None = None,
        out_grid: Any | None = None,
        method: str | None = None,
        matrix: str | None = None,
        mask: str | None = None,
        check: bool = False,
        missing_values: str | None = None,
    ) -> None:
        """`missing_values`: what a matrix regrid does with missing (NaN) source values.
        "propagate" (None, the default): y = A·x, a NaN reaches every target that references it.
        "missing-if-all-missing": the NaN sources are skipped and the row's remaining weights
        renormalised; NaN only when every source is missing (or the remaining weights do not
        sum to > 0).  "missing-if-heaviest-missing": the same, and NaN whenever the row's
        heaviest source is missing.  Nearest and mask regrids copy one source per target, which
        every policy leaves as it is."""
        self.in_grid = in_grid
        self.out_grid = out_grid
        self.method = method
        self.missing_values = missing_values
        self.interpolator = make_interpolator(
            in_grid=in_grid, out_grid=out_grid, method=method, matrix=matrix, mask=mask, check=check, missing_values=missing_values
        )

    def forward(self, data: Any) -> Any:
        return self._interpolate(data)

    def _interpolate(self, data: Any) -> Any:
        fields = list(data)
        if not fields:
            return new_fieldlist_from_list([])
        if hasattr(self.interpolator, "regrid_batch"):
            return new_fieldlist_from_list(self.interpolator.regrid_batch(fields))
        return new_fieldlist_from_list([self.interpolator(f) for f in fields])


class _BatchedInterpolator:
    """Shared driver: batch the FieldList, transform on the device, wrap the outputs."""

    def __call__(self, field: Any) -> Any:
        return self.regrid_batch([field])[0]

    #: fraction of the free HBM one sub-batch (inputs + outputs) may take
    memory_fraction = 0.4

    def regrid_batch(self, fields: list[Any]) -> list[Any]:
        """All fields in one device pass.

        Fields that arrive from the host and whose results are headed back to it are *streamed*
        (`at_hostio_regrid`: staging, H2D, compute and D2H of consecutive chunks overlap; only
        the results stay in HBM, and not even those when they would not fit).  Anything else —
        fields already resident, results wanted by the next filter of a pipeline — takes the
        batch path, in sub-batches whose outputs are moved to host memory as soon as they are
        computed when the FieldList does not fit in HBM."""
        from ...fields import device_column_of

        if results_are_host_bound() and all(device_column_of(f) is None for f in fields):
            return self._regrid_streamed(fields)
        per_field = self.bytes_per_field(fields[0])
        limit = max(4, int(self.memory_fraction * _free_device_bytes() // max(1, per_field)) // 4 * 4)
        if len(fields) <= limit:
            return self._regrid_resident(fields)
        LOG.info("regrid: %d fields exceed the device budget (%d per pass): streaming in sub-batches", len(fields), limit)
        out: list[Any] = []
        for i in range(0, len(fields), limit):
            part = self._regrid_resident(fields[i : i + limit])
            for batch in {id(b): b for b, _ in filter(None, (device_column_of(f) for f in part))}.values():
                batch.offload()
            out.extend(part)
        return out

    def bytes_per_field(self, field: Any) -> int:
        """Device bytes one field costs: its input column plus its output column (float64 worst case)."""
        n_in = int(np.prod(field.shape)) if hasattr(field, "shape") else 0
        return 8 * (n_in + self.output_points(n_in))

    def output_points(self, n_in: int) -> int:
        return n_in

    @staticmethod
    def _host_values(field: Any) -> np.ndarray:
        # reshape(-1) instead of flatten=True: no host copy when the field is contiguous
        v = np.asarray(field.to_numpy()).reshape(-1)
        if v.dtype != np.float32 and v.dtype != np.float64:
            v = v.astype(np.float64)
        return v if v.flags.c_contiguous else np.ascontiguousarray(v)

    def _wrap(self, fields: list[Any], idxs: list[int], result: DeviceBatch, out: list[Any]) -> None:
        lat, lon = self.output_grid(fields[idxs[0]])
        for j, i in enumerate(idxs):
            out[i] = new_field_from_latitudes_longitudes(new_field_from_device_column(result, j, template=fields[i]), latitudes=lat, longitudes=lon)

    def _regrid_streamed(self, fields: list[Any]) -> list[Any]:
        torch = require_cuda()
        self.prepare(fields[0])
        out: list[Any] = [None] * len(fields)
        packed, packed_idx, other_idx = grib.split(fields)
        if packed is not None:
            # simple-packed GRIB messages: the packed octets cross PCIe, the device decodes them
            # to float64 (what `to_numpy()` of a GRIB field returns) in front of the transform
            op, csr, index, n_tgt, y_dtype = self.stream_spec(packed.n_points, torch.float32 if packed.dtype == np.float32 else torch.float64)
            keep = 8 * n_tgt * len(packed_idx) <= self.memory_fraction * _free_device_bytes()
            job = self._stream(op, csr, index, n_tgt, y_dtype, packed, keep)
            try:
                self._wrap(fields, packed_idx, job.batch, out)
            finally:
                job.join()
            if not other_idx:
                return out
        # everything else (numpy fields, other packings, bitmaps): values fetched on the host
        values: dict[int, np.ndarray] = {i: self._host_values(fields[i]) for i in other_idx}
        by_dtype: dict[Any, list[int]] = {}
        for i, v in values.items():
            by_dtype.setdefault(v.dtype, []).append(i)
        for dtype, idxs in by_dtype.items():
            arrays = [values[i] for i in idxs]
            n_src = int(arrays[0].size)
            for i in idxs:
                if values[i].size != n_src:
                    raise ValueError(f"field {i} has {values[i].size} points, expected {n_src}")
            op, csr, index, n_tgt, y_dtype = self.stream_spec(n_src, torch.float32 if dtype == np.float32 else torch.float64)
            keep = 8 * n_tgt * len(arrays) <= self.memory_fraction * _free_device_bytes()
            job = self._stream(op, csr, index, n_tgt, y_dtype, arrays, keep)
            try:
                self._wrap(fields, idxs, job.batch, out)  # while the fields stream through the GPU
            finally:
                job.join()
        return out

    def _stream(self, op: int, csr: CsrMatrix | None, index: Any, n_tgt: int, y_dtype: Any, inputs: Any, keep: bool) -> StreamedRegrid:
        devices = fanout_devices()
        if devices is None:
            return StreamedRegrid(op, csr, index, n_tgt, y_dtype, inputs, keep_resident=keep, to_host=True)
        if index is not None:
            index = [self._index_on(index, d) for d in devices]
        return StreamedRegrid(op, csr, index, n_tgt, y_dtype, inputs, keep_resident=False, to_host=True, devices=devices)

    def _index_on(self, index: Any, device: int) -> Any:
        """The device index `index` on `device`, copied there once per index (the cache holds
        `index`, so its memory cannot be reused by another index while it is cached)."""
        cache = self.__dict__.setdefault("_index_by_device", {})
        hit = cache.get(device)
        if hit is None or hit[0].data_ptr() != index.data_ptr() or hit[0].shape != index.shape:
            hit = cache[device] = (index, index if index.device.index == device else index.to(f"cuda:{device}"))
        return hit[1]

    def stream_spec(self, n_src: int, x_dtype: Any):
        """→ (op, csr, device index, n_tgt, result dtype) of `at_hostio_regrid`."""
        raise NotImplementedError

    def _regrid_resident(self, fields: list[Any]) -> list[Any]:
        self.prepare(fields[0])
        # numpy dtypes differ per field in principle; batch runs of equal dtype together.
        # Host values are fetched once here (to_numpy decodes / copies) and handed to the upload.
        from ...fields import device_column_of

        out: list[Any] = [None] * len(fields)
        if all(device_column_of(f) is None for f in fields):
            packed = grib.packed_of(fields)
            if packed is not None:  # decoded on the device, see _regrid_streamed
                result = self.apply(grib.upload(packed))
                if results_are_host_bound():
                    result.prefetch()
                self._wrap(fields, list(range(len(fields))), result, out)
                return out
        by_dtype: dict[Any, list[int]] = {}
        host_values: dict[int, np.ndarray] = {}
        for i, f in enumerate(fields):
            col = device_column_of(f)
            if col is not None:
                key = str(col[0].data.dtype)
            else:
                host_values[i] = v = self._host_values(f)
                key = "torch.float32" if v.dtype == np.float32 else "torch.float64"
            by_dtype.setdefault(key, []).append(i)
        for _, idxs in by_dtype.items():
            batch = fields_to_batch([fields[i] for i in idxs], host_values=[host_values.get(i) for i in idxs])
            result = self.apply(batch)
            if results_are_host_bound():
                result.prefetch()
            self._wrap(fields, idxs, result, out)
        return out

    def prepare(self, first_field: Any) -> None:
        pass

    def apply(self, batch: DeviceBatch) -> DeviceBatch:
        raise NotImplementedError

    def output_grid(self, field: Any):
        raise NotImplementedError


class MIRMatrix(_BatchedInterpolator):
    """Matrix created by ``anemoi-transform make-regrid-file`` (npz schema
    make-regrid-file.py:150-160), applied as a device SpMM."""

    def __init__(self, *, matrix: str, check: bool, missing_values: str | None = None) -> None:
        self.missing = missing_policy(missing_values)
        self.check = check
        if self.check:
            LOG.warning("Check is not supported by MIRMatrix")
        loaded = dict(np.load(matrix))
        self.matrix = CsrMatrix(loaded["matrix_data"], loaded["matrix_indices"], loaded["matrix_indptr"], tuple(loaded["matrix_shape"]))
        self.in_grid = dict(latitudes=loaded["in_latitudes"], longitudes=loaded["in_longitudes"])
        self.out_grid = dict(latitudes=loaded["out_latitudes"], longitudes=loaded["out_longitudes"])

    def output_points(self, n_in: int) -> int:
        return self.matrix.shape[0]

    def apply(self, batch: DeviceBatch) -> DeviceBatch:
        if batch.n_points != self.matrix.shape[1]:
            raise ValueError(f"dimension mismatch: matrix has {self.matrix.shape[1]} columns, field has {batch.n_points} points")
        return DeviceBatch(self.matrix.apply(batch.data, n_fields=batch.n_fields, missing=self.missing), batch.n_fields)

    def stream_spec(self, n_src: int, x_dtype: Any):
        return _MATRIX_OPS[self.missing], self.matrix, None, self.matrix.shape[0], self.matrix.result_dtype(x_dtype)

    def output_grid(self, field: Any):
        return self.out_grid["latitudes"], self.out_grid["longitudes"]


class ScipyKDTreeNearestNeighbours(_BatchedInterpolator):
    """Nearest-neighbour regridding for grids earthkit-regrid has no matrix for.

    The class name is the reference's (regrid.py:315); the search itself is the bucketed
    device kNN of `spatial.nearest_grid_points`, not scipy.
    """

    nearest_grid_points = None

    def __init__(self, *, in_grid: Any, out_grid: Any, method: str, check: bool = False, missing_values: str | None = None) -> None:
        missing_policy(missing_values)  # validated; one source per target is the same under every policy
        if method != "nearest":
            raise NotImplementedError(f"ScipyKDTreeNearestNeighbours does not support {method}, only 'nearest'")
        self.in_grid = as_griddata(in_grid)
        self.out_grid = as_griddata(out_grid)
        if self.out_grid is None:
            raise ValueError("out_grid is required, but not provided")
        if check:
            LOG.warning("Check is not supported by ScipyKDTreeNearestNeighbours")

    def prepare(self, first_field: Any) -> None:
        if self.in_grid is None:
            self.in_grid = as_griddata(first_field)
            assert self.in_grid is not None, first_field
        if self.nearest_grid_points is None:
            from ...spatial import nearest_grid_points

            self.nearest_grid_points = nearest_grid_points(
                self.in_grid["latitudes"],
                self.in_grid["longitudes"],
                self.out_grid["latitudes"],
                self.out_grid["longitudes"],
                _as_device=True,
            )

    def output_points(self, n_in: int) -> int:
        return int(np.size(self.out_grid["latitudes"]))

    def _check_points(self, n_points: int) -> None:
        n_in = (n_points,)
        assert n_in == np.shape(self.in_grid["latitudes"]), (n_in, np.shape(self.in_grid["latitudes"]))
        assert n_in == np.shape(self.in_grid["longitudes"]), (n_in, np.shape(self.in_grid["longitudes"]))

    def apply(self, batch: DeviceBatch) -> DeviceBatch:
        self._check_points(batch.n_points)
        return DeviceBatch(gather_rows(batch.data, self.nearest_grid_points, n_fields=batch.n_fields), batch.n_fields)

    def stream_spec(self, n_src: int, x_dtype: Any):
        self._check_points(n_src)
        idx = self.nearest_grid_points.reshape(-1)
        return _cabi.HOSTIO_GATHER, None, idx, int(idx.shape[0]), x_dtype

    def output_grid(self, field: Any):
        return self.out_grid["latitudes"], self.out_grid["longitudes"]


class MaskedRegrid(_BatchedInterpolator):
    """Select points with a precomputed index (or boolean) mask (`make-regrid-file
    global-on-lam-mask`, make-regrid-file.py:239-240)."""

    out_latitudes = None
    out_longitudes = None

    def __init__(self, *, mask: str, check: bool, missing_values: str | None = None) -> None:
        missing_policy(missing_values)  # validated; one source per target is the same under every policy
        if check:
            LOG.warning("Check is not supported by MaskedRegrid")
        self.mask = np.load(mask)["mask"]
        self._device_index = None
        self._index_points = -1

    def _index(self, n_points: int):
        """The mask as device int64 indices into a field of n_points (numpy's indexing rules)."""
        torch = require_cuda()
        if self._device_index is None or self._index_points != n_points:
            m = self.mask
            if m.dtype == np.bool_:
                if m.shape[0] != n_points:
                    raise IndexError(f"boolean index did not match indexed array along axis 0; size of axis is {n_points} but size of corresponding boolean axis is {m.shape[0]}")
                m = np.nonzero(m)[0]
            m = np.asarray(m).astype(np.int64).reshape(-1)
            bad = m[(m < -n_points) | (m >= n_points)]
            if bad.size:
                raise IndexError(f"index {int(bad[0])} is out of bounds for axis 0 with size {n_points}")
            m = np.where(m < 0, m + n_points, m)  # numpy's negative indexing
            self._device_index, self._index_points = torch.from_numpy(m).cuda(), n_points
        return self._device_index

    def apply(self, batch: DeviceBatch) -> DeviceBatch:
        return DeviceBatch(gather_rows(batch.data, self._index(batch.n_points), n_fields=batch.n_fields), batch.n_fields)

    def output_points(self, n_in: int) -> int:
        return int(self._index(n_in).shape[0])

    def stream_spec(self, n_src: int, x_dtype: Any):
        idx = self._index(n_src)
        return _cabi.HOSTIO_GATHER, None, idx, int(idx.shape[0]), x_dtype

    def output_grid(self, field: Any):
        if self.out_latitudes is None or self.out_longitudes is None:
            in_latitudes, in_longitudes = field.grid_points()
            self.out_latitudes = in_latitudes[self.mask]
            self.out_longitudes = in_longitudes[self.mask]
        return self.out_latitudes, self.out_longitudes


class EarthkitRegrid(_BatchedInterpolator):
    """The `in_grid` / `out_grid` / `method` recipes (reference regrid.py:211-259).

    The reference hands these to `earthkit.regrid.interpolate`, i.e. to earthkit-regrid's
    inventory of MIR matrices; neither the package nor the inventory exists offline.  Here the
    matrix is built locally on the device the first time it is needed and applied like any
    other (`MIRMatrix` machinery: one SpMM over the whole FieldList):

        method="linear"                      4-point bilinear weights, regular lat-lon sources
                                             (`regrid_files.make_bilinear_matrix`)
        method="structured-bilinear"         2 rows × 2 points (4 entries per target) on any
                                             global structured source: octahedral / reduced /
                                             full Gaussian, regular lat-lon
                                             (`regrid_files.make_structured_matrix`)
        method="structured-bicubic"          4 rows × 4 points, cubic Lagrange in longitude
                                             then latitude (16 entries), same sources
        method="structured-conservative"     first-order conservative grid-box averages (area
                                             weighted, rows sum to 1, the area integral kept)
                                             between two global structured grids: for
                                             accumulated / flux fields and coarsening
                                             (`regrid_files.make_conservative_matrix`); its
                                             boxes are latitude bands on every grid, HEALPix
                                             included
        method="healpix-conservative"        the same with the true HEALPix pixels: between a
                                             HEALPix grid (ring or nested, any nside) and a
                                             HEALPix or global structured grid
                                             (`regrid_files.make_healpix_conservative_matrix`)
        method="nearest-neighbour" | "nn"    the nearest source point (`make_knn_matrix`, k = 1)

    (`method="nearest"` is dispatched to `ScipyKDTreeNearestNeighbours`, as in the reference.)
    The class name is the reference's so that `_interpolator` / configuration dumps read the
    same; other schemes (MIR's "grid-box-average" among them), and grids a method cannot take
    (non-regular sources for "linear", non-structured sources for the structured methods and
    non-structured targets for "structured-conservative"), raise NotImplementedError and still
    need a `matrix=` made with MIR.
    """

    METHODS = ("linear", "structured-bilinear", "structured-bicubic", "structured-conservative", "healpix-conservative", "nearest-neighbour", "nn")

    def __init__(self, *, in_grid: Any = None, out_grid: Any = None, method: str = "linear", check: bool = False, missing_values: str | None = None) -> None:
        self.missing = missing_policy(missing_values)
        if method not in self.METHODS:
            raise NotImplementedError(f"regrid: method {method!r} is not built locally (have {self.METHODS} and 'nearest'); pass `matrix=`")
        if out_grid is None:
            raise ValueError("out_grid is required, but not provided")
        self.in_gridspec = as_gridspec(in_grid)
        self.out_gridspec = as_gridspec(out_grid)
        self.in_grid = as_griddata(in_grid)
        self.out_grid = as_griddata(out_grid)
        self.method = method
        self.matrix: CsrMatrix | None = None
        if check:
            LOG.warning("Check is not supported by EarthkitRegrid")

    def prepare(self, first_field: Any) -> None:
        if self.matrix is not None:
            return
        if self.in_grid is None:  # earthkit-regrid reads the grid off the field; so do we
            self.in_grid = as_griddata(first_field)
        from ...regrid_files import make_bilinear_matrix, make_conservative_matrix, make_healpix_conservative_matrix, make_knn_matrix, make_structured_matrix

        src = (self.in_grid["latitudes"], self.in_grid["longitudes"])
        dst = (self.out_grid["latitudes"], self.out_grid["longitudes"])
        if self.method == "linear":
            data, indices, indptr, shape = make_bilinear_matrix(*src, *dst)
        elif self.method == "structured-conservative":
            data, indices, indptr, shape = make_conservative_matrix(*src, *dst)
        elif self.method == "healpix-conservative":
            data, indices, indptr, shape = make_healpix_conservative_matrix(*src, *dst)
        elif self.method.startswith("structured-"):
            data, indices, indptr, shape = make_structured_matrix(*src, *dst, self.method)
        else:
            data, indices, indptr, shape = make_knn_matrix(*src, *dst, k=1)
        self.matrix = CsrMatrix(data, indices, indptr, shape)

    def output_points(self, n_in: int) -> int:
        return int(np.size(self.out_grid["latitudes"]))

    def apply(self, batch: DeviceBatch) -> DeviceBatch:
        if batch.n_points != self.matrix.shape[1]:
            raise ValueError(f"dimension mismatch: matrix has {self.matrix.shape[1]} columns, field has {batch.n_points} points")
        return DeviceBatch(self.matrix.apply(batch.data, n_fields=batch.n_fields, missing=self.missing), batch.n_fields)

    def stream_spec(self, n_src: int, x_dtype: Any):
        return _MATRIX_OPS[self.missing], self.matrix, None, self.matrix.shape[0], self.matrix.result_dtype(x_dtype)

    def output_grid(self, field: Any):
        return self.out_grid["latitudes"], self.out_grid["longitudes"]


def _interpolator(*, method: str | None = None, matrix: str | None = None, mask: str | None = None) -> str:
    if matrix is not None:
        return "MIRMatrix"
    if mask is not None:
        return "MaskedRegrid"
    if method == "nearest":
        return "ScipyKDTreeNearestNeighbours"
    return "EarthkitRegrid"


def make_interpolator(
    in_grid: Any = None,
    out_grid: Any = None,
    method: str | None = None,
    matrix: str | None = None,
    mask: str | None = None,
    check: bool | None = None,
    missing_values: str | None = None,
) -> Any:
    name = _interpolator(method=method, matrix=matrix, mask=mask)
    kwargs = {"in_grid": in_grid, "out_grid": out_grid, "method": method, "matrix": matrix, "mask": mask, "check": check, "missing_values": missing_values}
    kwargs = {k: v for k, v in kwargs.items() if v is not None}
    return globals()[name](**kwargs)
