"""Fusing `regrid | uv_to_ddff | q_to_r | clip | apply_mask` into one kernel launch.

(Matrix regrids — from a file or built locally — run `at_spmm_fused`; nearest-neighbour and
mask regrids run `at_gather_pointwise`, the same epilogue behind a row gather.  Followers:
wind, humidity, dewpoint, cos/sin -> angle, clip, mask and the one-field conversions.)

In the reference every filter of a pipeline materialises a complete new FieldList
(`workflows/pipeline.py:33-48`), so a regrid followed by four pointwise filters reads and
writes every field five times.  `at_spmm_fused` applies the pointwise program in the SpMM
epilogue instead: one read of X, one write of Y.

`fuse(filters)` rewrites a flat filter list: a `RegridFilter` that applies a float32 matrix,
followed by pointwise filters of this package, becomes one `FusedRegrid`.  The fused filter
*plans* on metadata only — it runs the followers' own selection / grouping logic
(`GroupByParam`, `FieldSelection`) over placeholder fields, so grouping, ordering, renaming
and error behaviour are the followers' own — and then issues a single launch.  Whatever the
epilogue cannot express (a clip before a conversion, two masks, float64 fields, partial
`return_inputs`, …) raises `Unfusable` during planning and the original filters run one
after the other, device-resident, with identical results
(`tests/test_gpu_filters.py::test_pipeline_fusion_*`).
"""

from __future__ import annotations

import logging
from typing import Any

import numpy as np

from . import _cabi, grib
from .batching import fields_to_batch
from .device import DeviceBatch, Epilogue, require_cuda, results_are_host_bound, round_up
from .fields import DeviceColumnField, NewMetadataField, device_column_of, new_field_from_latitudes_longitudes, new_fieldlist_from_list
from .filter import Filter
from .grouping import GroupByParam
from .transform import ReversedTransform

LOG = logging.getLogger(__name__)


class Unfusable(Exception):
    """The pipeline needs something the fused epilogue cannot express; run it unfused."""


class _Sym:
    """A field of the pipeline during planning: metadata is real, values are a plan."""

    __slots__ = ("field", "node", "src", "inp", "lo", "hi", "masked", "pressure")

    def __init__(self, field: Any, node: DeviceColumnField, src: tuple):
        self.field = field  # what the unfused chain would hand to the next filter
        self.node = node  # the DeviceColumnField to bind to an output column
        self.src = src  # ("col", i): regridded input i | ("conv", group, slot): output of a conversion
        self.inp = src[1] if src[0] == "col" else None  # index of the input field, if it is one
        self.lo = self.hi = None
        self.masked = False
        self.pressure = 0.0

    def transformed(self, **metadata: Any) -> "_Sym":
        """A new value derived from this field (same metadata template, overridden keys)."""
        node = DeviceColumnField(self.field, None, 0, shape=self.node.shape)
        return _Sym(NewMetadataField(node, **metadata), node, ("conv", -1, 0))


class _Group:
    __slots__ = ("kind", "inputs", "outputs", "pa", "pb")

    def __init__(self, kind: int, inputs: list[_Sym], outputs: list[_Sym], pa: float = 0.0, pb: float = 0.0):
        self.kind, self.inputs, self.outputs, self.pa, self.pb = kind, inputs, outputs, pa, pb


def _direction(f: Any, cls: type) -> str | None:
    if isinstance(f, cls):
        return "forward"
    if isinstance(f, ReversedTransform) and isinstance(f.filter, cls):
        return "backward"
    return None


def _unwrap(f: Any) -> Any:
    """The field-level implementation behind a dispatcher (`clip`, `mask`)."""
    from .filters.clip import Clip
    from .filters.geopotential_to_height import GeopotentialToHeight
    from .filters.impute_nans import ImputeNaNs as ImputeNaNsDispatcher
    from .filters.mask import Mask

    if isinstance(f, (Clip, Mask)):
        return f.filter
    if isinstance(f, (GeopotentialToHeight, ImputeNaNsDispatcher)):
        return f.field_filter
    if isinstance(f, ReversedTransform) and isinstance(f.filter, GeopotentialToHeight):
        return ReversedTransform(f.filter.field_filter)
    return f


def _unary_plan(f: Any):
    """(filter, direction, kind, pa, pb, metadata) for the one-field-in / one-field-out filters
    the epilogue runs (`rescale` / `convert`, `lnsp_to_sp`, `impute_nans`, `orog_to_z`), else None.
    The metadata is what the filter's own `*_transform_batch` attaches to its outputs."""
    from .constants import g_gravitational_acceleration as g
    from .filters.fields.impute_nans import ImputeNaNs
    from .filters.fields.lnsp_to_sp import LnspToSp
    from .filters.fields.orog_to_z import Orography
    from .filters.fields.rescale import RescaleMixin

    for cls in (RescaleMixin, LnspToSp, ImputeNaNs, Orography):
        d = _direction(f, cls)
        if d is None:
            continue
        t = f if isinstance(f, cls) else f.filter
        fwd = d == "forward"
        if cls is RescaleMixin:
            kind = _cabi.EPI_AFFINE if fwd else _cabi.EPI_AFFINE_INV
            md = dict(param=t.param, units=t.forward_units) if fwd else dict(param=t.param)
            return t, d, kind, float(t.rescaler.scale), float(t.rescaler.offset), md
        if cls is LnspToSp:
            md = {"param": t.surface_pressure, "levelist": None, "level": None} if fwd else {"param": t.log_of_surface_pressure}
            return t, d, (_cabi.EPI_EXP if fwd else _cabi.EPI_LOG), 0.0, 0.0, md
        if cls is ImputeNaNs:
            if not fwd:
                return None
            return t, d, _cabi.EPI_IMPUTE_NAN, float(t.value), 0.0, {}
        md = {"param": t.geopotential} if fwd else {"param": t.orography}
        return t, d, (_cabi.EPI_AFFINE if fwd else _cabi.EPI_AFFINE_INV), g, 0.0, md
    return None


def is_fusable_follower(f: Any) -> bool:
    from .filters.fields.apply_mask import MaskVariable
    from .filters.fields.clipper import Clipper
    from .filters.fields.cos_sin_from_rad import CosSinFromRad
    from .filters.fields.dewpoint import DewPoint
    from .filters.fields.q_to_r import HumidityConversion
    from .filters.fields.uv_to_ddff import WindComponents

    f = _unwrap(f)
    if bool(_direction(f, WindComponents) or _direction(f, HumidityConversion) or _direction(f, DewPoint)) or isinstance(f, (Clipper, MaskVariable)):
        return True
    if _direction(f, CosSinFromRad) == "backward":  # forward validates the value range first (cos_sin_from_rad.py:74-77)
        return True
    return _unary_plan(f) is not None


def is_fusable_regrid(f: Any) -> bool:
    """A regrid whose interpolator the fused launch can run: a float32 matrix (from a file or
    built locally) through `at_spmm_fused`, a nearest-neighbour or mask gather through
    `at_gather_pointwise`.  A matrix regrid that skips missing values (`missing_values=`) is
    not: the fused kernel has no missing-aware accumulation, and the chain runs unfused."""
    from .filters.fields.regrid import EarthkitRegrid, MaskedRegrid, MIRMatrix, RegridFilter, ScipyKDTreeNearestNeighbours

    if not isinstance(f, RegridFilter):
        return False
    if getattr(f.interpolator, "missing", _cabi.MISSING_PROPAGATE) != _cabi.MISSING_PROPAGATE:
        return False
    if isinstance(f.interpolator, MIRMatrix):
        return f.interpolator.matrix.dtype == np.float32
    return isinstance(f.interpolator, (EarthkitRegrid, ScipyKDTreeNearestNeighbours, MaskedRegrid))


def flatten(filters: list[Any]) -> list[Any]:
    from .workflows import Pipeline

    out: list[Any] = []
    for f in filters:
        out.extend(flatten(f.filters) if isinstance(f, Pipeline) else [f])
    return out


def fuse(filters: list[Any]) -> list[Any]:
    """Replace `regrid, pointwise…` runs by `FusedRegrid`; everything else is kept as is."""
    filters = flatten(filters)
    out: list[Any] = []
    i = 0
    while i < len(filters):
        f = filters[i]
        if is_fusable_regrid(f):
            j = i + 1
            while j < len(filters) and is_fusable_follower(filters[j]):
                j += 1
            if j > i + 1:
                out.append(FusedRegrid(f, filters[i + 1 : j]))
                i = j
                continue
        out.append(f)
        i += 1
    return out


class FusedRegrid(Filter):
    """`regrid` and the pointwise filters after it, as one `at_spmm_fused` launch."""

    def __init__(self, regrid: Any, followers: list[Any]) -> None:
        self.regrid = regrid
        self.followers = list(followers)
        self.last_forward_was_fused = False

    def __repr__(self) -> str:
        return f"FusedRegrid({self.regrid}, {self.followers})"

    def forward(self, data: Any) -> Any:
        fields = list(data)
        self.last_forward_was_fused = False
        if fields:
            try:
                result = self._forward_fused(fields)
                self.last_forward_was_fused = True
                return result
            except Unfusable as why:
                LOG.info("pipeline not fused (%s); running the filters one after the other", why)
        out = self.regrid.forward(new_fieldlist_from_list(fields))
        for f in self.followers:
            out = f.forward(out)
        return out

    # ------------------------------------------------------------------ planning ------
    def _forward_fused(self, fields: list[Any]) -> Any:
        from .filters.fields.apply_mask import MaskVariable
        from .filters.fields.clipper import Clipper
        from .filters.fields.cos_sin_from_rad import CosSinFromRad
        from .filters.fields.dewpoint import DewPoint
        from .filters.fields.q_to_r import HumidityConversion
        from .filters.fields.uv_to_ddff import WindComponents

        torch = require_cuda()
        interp = self.regrid.interpolator
        interp.prepare(fields[0])
        n_tgt = interp.output_points(int(np.prod(fields[0].shape)))
        lat, lon = interp.output_grid(fields[0])

        for f in fields:
            col = device_column_of(f)
            dt = col[0].data.dtype if col is not None else None
            if dt is None and grib.is_packed_message(f):
                # decoded on the device to what to_numpy() gives; no host decode just to learn the dtype
                dt = torch.float32 if grib.decode_dtype() == np.float32 else torch.float64
            if dt is None:
                dt = torch.float32 if np.asarray(f.to_numpy()).dtype == np.float32 else torch.float64
            if dt != torch.float32:
                raise Unfusable("float64 fields")

        # the regridded fields, as the regrid filter would wrap them
        syms: list[_Sym] = []
        for i, f in enumerate(fields):
            node = DeviceColumnField(f, None, 0, shape=(n_tgt,))
            syms.append(_Sym(new_field_from_latitudes_longitudes(NewMetadataField(node), latitudes=lat, longitudes=lon), node, ("col", i)))

        groups: list[_Group] = []
        mask_filter = None
        mask_sym = None

        for follower in self.followers:
            f = _unwrap(follower)
            pair_classes = (WindComponents, HumidityConversion, DewPoint, CosSinFromRad)
            paired = next((d for d in (_direction(f, c) for c in pair_classes) if d), None)
            if paired:
                target = f if isinstance(f, pair_classes) else f.filter
                syms = self._plan_matching(target, paired, syms, groups)
            elif isinstance(f, Clipper):
                for s in syms:
                    if f._forward_selection.match(s.field):
                        if s.lo is not None or s.hi is not None or s.masked:
                            raise Unfusable("clip after another clip or a mask on the same field")
                        s.lo, s.hi = f.minimum, f.maximum
                        self._retag(s, param=s.field.metadata("param"))
            elif isinstance(f, MaskVariable):
                if mask_filter is not None:
                    raise Unfusable("more than one mask")
                mask_filter = f
                if f.mask_param is not None:
                    kept = []
                    for s in syms:
                        if s.field.metadata("param") == f.mask_param:
                            if mask_sym is None:
                                mask_sym = s
                            if not f.return_mask:
                                continue
                        kept.append(s)
                    if mask_sym is None:
                        raise ValueError(f"Mask parameter '{f.mask_param}' not found in input data.")
                    if mask_sym.src[0] != "col" or mask_sym.lo is not None or mask_sym.hi is not None:
                        raise Unfusable("mask field is itself transformed")
                    syms = kept
                for s in syms:
                    if f._forward_selection.match(s.field):
                        s.masked = True
                        md = {"param": f"{s.field.metadata('param')}_{f.rename}"} if f.rename is not None else {}
                        self._retag(s, **md)
            elif _unary_plan(f) is not None:
                target, direction, kind, pa, pb, md = _unary_plan(f)
                selection = target._forward_selection if direction == "forward" else target._backward_selection
                for pos, sym in enumerate(syms):
                    if not selection.match(sym.field):
                        continue
                    if sym.src[0] != "col" or sym.lo is not None or sym.hi is not None or sym.masked:
                        raise Unfusable("conversion of a field that was already transformed")
                    o = sym.transformed(**md)
                    o.src = ("conv", len(groups), 0)
                    groups.append(_Group(kind, [sym], [o], pa, pb))
                    syms[pos] = o
            else:  # pragma: no cover - guarded by is_fusable_follower
                raise Unfusable(f"unsupported filter {follower}")

        return self._launch(fields, syms, groups, mask_filter, mask_sym)

    @staticmethod
    def _retag(s: _Sym, **metadata: Any) -> None:
        """The filter produced a new field object from `s` (same values plan, new wrapper)."""
        node = DeviceColumnField(s.field, None, 0, shape=s.node.shape)
        s.field, s.node = NewMetadataField(node, **metadata), node

    def _plan_matching(self, f: Any, direction: str, syms: list[_Sym], groups: list[_Group]) -> list[_Sym]:
        """Mirror MatchingFieldsFilter._run on symbolic fields."""
        from .filters.fields.cos_sin_from_rad import CosSinFromRad
        from .filters.fields.dewpoint import DewPoint
        from .filters.fields.uv_to_ddff import WindComponents

        names = getattr(f.MATCHING, direction)
        params = [getattr(f, name) for name in names]
        returned = f.MATCHING.inputs(direction=direction)
        if set(returned) not in (set(), set(names)):
            raise Unfusable("partial return_inputs")
        by_field = {id(s.field): s for s in syms}
        result: list[_Sym] = []
        planned = list(GroupByParam(params).iterate([s.field for s in syms], other=lambda fld: result.append(by_field[id(fld)])))
        for members in planned:
            a, b = (by_field[id(m)] for m in members)
            for s in (a, b):
                if s.src[0] != "col" or s.lo is not None or s.hi is not None or s.masked:
                    raise Unfusable("conversion of a field that was already transformed")
            if isinstance(f, WindComponents):
                kind = _cabi.EPI_UV2DDFF if direction == "forward" else _cabi.EPI_DDFF2UV
                out_params = (f.wind_speed, f.wind_direction) if direction == "forward" else (f.u_component, f.v_component)
                outs = [a.transformed(param=out_params[0]), b.transformed(param=out_params[1])]
                for k, o in enumerate(outs):
                    o.src = ("conv", len(groups), k)
                groups.append(_Group(kind, [a, b], outs))
                result.extend(outs)
            elif isinstance(f, CosSinFromRad):  # backward only: (cos, sin) -> the angle, inputs dropped
                o = a.transformed(param=f.param)
                o.src = ("conv", len(groups), 0)
                groups.append(_Group(_cabi.EPI_ATAN2, [a, b], [o], 1.0, 0.0))
                result.append(o)
            elif isinstance(f, DewPoint):
                forward = direction == "forward"
                keep = bool(returned)
                kind = (_cabi.EPI_RT2RTD if keep else _cabi.EPI_RT2D) if forward else (_cabi.EPI_DT2DTR if keep else _cabi.EPI_DT2R)
                template = a if forward else b  # dewpoint.py: forward wraps relative_humidity, backward temperature
                o = template.transformed(param=f.dewpoint if forward else f.relative_humidity)
                o.src = ("conv", len(groups), 2 if keep else 0)
                if keep:
                    a.src, b.src = ("conv", len(groups), 0), ("conv", len(groups), 1)
                    result.extend([a, b])
                groups.append(_Group(kind, [a, b], [a, b, o] if keep else [o]))
                result.append(o)
            else:
                forward = direction == "forward"
                keep = bool(returned)
                kind = (_cabi.EPI_QT2QTR if keep else _cabi.EPI_QT2R) if forward else (_cabi.EPI_RT2RTQ if keep else _cabi.EPI_RT2Q)
                level_from = a if forward else b  # q_to_r.py:71 (humidity) / :77 (temperature)
                o = a.transformed(param=f.relative_humidity if forward else f.humidity)
                o.pressure = 100 * float(level_from.field.metadata("levelist"))
                o.src = ("conv", len(groups), 2 if keep else 0)
                if keep:
                    a.src, b.src = ("conv", len(groups), 0), ("conv", len(groups), 1)
                    result.extend([a, b])
                groups.append(_Group(kind, [a, b], [a, b, o] if keep else [o]))
                result.append(o)
        return result

    # ------------------------------------------------------------------ launch --------
    def _launch(self, fields: list[Any], syms: list[_Sym], groups: list[_Group], mask_filter: Any, mask_sym: _Sym | None) -> Any:
        torch = require_cuda()
        interp = self.regrid.interpolator
        OUT_PER_PAIR = {
            _cabi.EPI_UV2DDFF: 2, _cabi.EPI_DDFF2UV: 2, _cabi.EPI_QT2R: 1, _cabi.EPI_RT2Q: 1, _cabi.EPI_QT2QTR: 3, _cabi.EPI_RT2RTQ: 3,
            _cabi.EPI_ATAN2: 1, _cabi.EPI_RT2D: 1, _cabi.EPI_DT2R: 1, _cabi.EPI_RT2RTD: 3, _cabi.EPI_DT2DTR: 3,
        }  # fmt: skip

        # input columns: plain fields first, then the pairs of each conversion kind
        plain = [s for s in syms if s.src[0] == "col"]
        in_fields: list[Any] = [fields[s.inp] for s in plain]
        segments: list[tuple] = []
        out_cols: list[tuple[float, float, float, int]] = []
        assign: list[tuple[_Sym, int]] = []

        def col_params(s: _Sym | None) -> tuple[float, float, float, int]:
            if s is None:
                return (0.0, 0.0, 0.0, 0)
            flags = (_cabi.COL_CLIP_LO if s.lo is not None else 0) | (_cabi.COL_CLIP_HI if s.hi is not None else 0) | (_cabi.COL_MASK if s.masked else 0)
            return (s.lo or 0.0, s.hi or 0.0, s.pressure, flags)

        def pad_inputs(to: int) -> None:
            while len(in_fields) % to:
                in_fields.append(in_fields[-1])  # padding column: any real field

        if plain:
            pad_inputs(4)
            segments.append((_cabi.EPI_PLAIN, 0, len(in_fields), 0))
            for k, s in enumerate(plain):
                assign.append((s, k))
            out_cols = [col_params(s) for s in plain] + [col_params(None)] * (len(in_fields) - len(plain))
        live = set(id(s) for s in syms)
        # one-in / one-out kinds: a segment per (kind, constants), columns 1:1
        unary = [g for g in groups if g.kind not in OUT_PER_PAIR]
        for key in sorted({(g.kind, g.pa, g.pb) for g in unary}):
            same = [g for g in unary if (g.kind, g.pa, g.pb) == key]
            in0, out0 = len(in_fields), round_up(len(out_cols), 4)
            out_cols += [col_params(None)] * (out0 - len(out_cols))
            for g in same:
                if g.inputs[0].inp is None:
                    raise Unfusable("conversion input that is itself a conversion output")
                in_fields.append(fields[g.inputs[0].inp])
            while (len(in_fields) - in0) % 4:
                in_fields.append(in_fields[-1])
            seg_out = [col_params(None)] * (len(in_fields) - in0)
            for k, g in enumerate(same):
                seg_out[k] = col_params(g.outputs[0])
                if id(g.outputs[0]) in live:
                    assign.append((g.outputs[0], out0 + k))
            segments.append((key[0], in0, len(in_fields) - in0, out0, key[1], key[2]))
            out_cols += seg_out
        for kind, pa, pb in sorted({(g.kind, g.pa, g.pb) for g in groups if g.kind in OUT_PER_PAIR}):
            same = [g for g in groups if (g.kind, g.pa, g.pb) == (kind, pa, pb)]
            in0, out0 = len(in_fields), len(out_cols)
            out0 = round_up(out0, 4)
            out_cols += [col_params(None)] * (out0 - len(out_cols))
            for g in same:
                for s in g.inputs:
                    if s.inp is None:
                        raise Unfusable("conversion input that is itself a conversion output")
                    in_fields.append(fields[s.inp])
            if len(same) % 2:
                in_fields.extend(in_fields[-2:])  # pad with a copy of the last pair
            n_pairs = (len(in_fields) - in0) // 2
            per = OUT_PER_PAIR[kind]
            seg_out = [col_params(None)] * (n_pairs * per)
            for p, g in enumerate(same):
                for o in g.outputs:
                    slot = o.src[2]
                    seg_out[p * per + slot] = col_params(o)
                    if id(o) in live:
                        assign.append((o, out0 + p * per + slot))
            segments.append((kind, in0, len(in_fields) - in0, out0, pa, pb))
            out_cols += seg_out
        out_cols += [col_params(None)] * (round_up(len(out_cols), 4) - len(out_cols))

        x = fields_to_batch(in_fields)
        # (matrix | None, gather index | None): validates the number of source points as the
        # stand-alone regrid does (scipy's dimension mismatch, numpy's IndexError)
        op, csr, index, n_tgt, _ = interp.stream_spec(x.n_points, torch.float32)
        if csr is not None and x.n_points != csr.shape[1]:
            raise ValueError(f"dimension mismatch: matrix has {csr.shape[1]} columns, field has {x.n_points} points")

        row_mask = None
        if mask_filter is not None:
            if mask_filter.mask_param is None:
                row_mask = mask_filter.mask
            else:
                one = fields_to_batch([fields[mask_sym.inp]])
                regridded = interp.apply(one).data
                row_mask = mask_filter._compute_mask(regridded[:, 0])
            if row_mask is None or int(row_mask.shape[0]) != n_tgt:
                have = None if row_mask is None else int(row_mask.shape[0])
                raise IndexError(f"boolean index did not match indexed array: mask has {have} points, field has {n_tgt}")
            mask_filter.mask = row_mask

        epi = Epilogue(segments, out_cols)
        try:
            if op == _cabi.HOSTIO_SPMM:
                y = epi.apply_fused(csr, x.data, row_mask=row_mask)
            else:
                y = epi.apply(x.data, row_mask=row_mask, gather=index.contiguous())
        finally:
            epi.close()
        # the launch writes round_up(len(out_cols), 4) columns; only those bound to a field count
        out_batch = DeviceBatch(y, max((col for _, col in assign), default=-1) + 1)
        if results_are_host_bound():
            out_batch.prefetch_columns(sorted({col for _, col in assign}))
        for s, col in assign:
            s.node._batch, s.node._col = out_batch, col
        placed = {id(s) for s, _ in assign}
        missing = [s for s in syms if id(s) not in placed]
        if missing:  # pragma: no cover - a planning bug must not produce silent garbage
            raise RuntimeError(f"fusion planner lost {len(missing)} output field(s)")
        return new_fieldlist_from_list([s.field for s in syms])
