"""`sum` — reference `filters/fields/sum.py:22-122`.

Sums a set of params per matching key (the mars namespace minus `param`, optionally minus
`levelist`), in field order, one device pass per dtype for all keys (`at_sum_cols`:
`s = c0; s += c1; …` in the batch's dtype).  The summed inputs are consumed, every other field
passes through first, the sums follow in first-seen key order (sum.py:88-118).

numpy's in-place `s += c` keeps the first term's dtype and rounds to it after every step,
also when a later term is wider.  Groups whose terms share one dtype run on the device, one
batch per dtype, so a float32 group stays float32 next to a float64 one.  A group that mixes
dtypes (float32 `lsp` with float64 `cp`, say) runs that statement on the host.
"""

from __future__ import annotations

import logging
from collections import defaultdict
from collections.abc import Hashable
from typing import Any

import numpy as np

from ...batching import fields_to_batch, numpy_dtype_of
from ...device import DeviceBatch, results_are_host_bound, sum_cols
from ...fields import device_column_of, new_field_from_device_column, new_field_from_numpy, new_fieldlist_from_list
from ...filter import Filter
from . import filter_registry

LOG = logging.getLogger(__name__)


@filter_registry.register("sum")
class Sum(Filter):
    """Computes the sum over a set of variables."""

    def __init__(self, *, params: list[str], output: str, ignore_level: bool = False):
        self.params = params
        self.output = output
        self.ignore_level = ignore_level

    def forward(self, fields: Any) -> Any:
        result = []
        needed_fields: dict[tuple[Hashable, ...], dict[str, Any]] = defaultdict(dict)
        for f in fields:
            key = dict(f.metadata(namespace="mars"))
            param = key.pop("param", None)
            if self.ignore_level:
                ll = key.pop("levelist", None)
                LOG.debug(f"Removing levelist ({ll}) from matching key for variable: {param}")
            if param is None:
                param = f.metadata("param")
            if param in self.params:
                key = tuple(key.items())
                if param in needed_fields[key]:
                    raise ValueError(f"Duplicate field {param} for {key}")
                needed_fields[key][param] = f
            else:
                result.append(f)

        groups = []
        for keys, values in needed_fields.items():
            if len(values) != len(self.params):
                raise ValueError("Missing fields")
            groups.append(list(values.values()))
        if groups:
            result.extend(self._sums(groups))
        return new_fieldlist_from_list(result)

    def _sums(self, groups: list[list[Any]]) -> list[Any]:
        n_terms = len(self.params)
        flat = [f for g in groups for f in g]
        cols = [device_column_of(f) for f in flat]
        if all(c is None for c in cols):
            from ... import grib

            if grib.packed_of(flat) is not None:  # GRIB messages decode to one dtype on the device
                return self._device_sums(groups, fields_to_batch(flat))
        values = [None if c is not None else np.asarray(f.to_numpy(flatten=True)) for f, c in zip(flat, cols)]
        dtypes = [np.dtype(numpy_dtype_of(c[0]) if c is not None else v.dtype) for c, v in zip(cols, values)]
        # per group: the float dtype all its terms share, else None (summed on the host)
        kinds = []
        for i in range(len(groups)):
            seen = set(dtypes[i * n_terms : (i + 1) * n_terms])
            kind = seen.pop() if len(seen) == 1 else None
            kinds.append(kind if kind in (np.float32, np.float64) else None)
        out: list[Any] = [None] * len(groups)
        for dt in dict.fromkeys(k for k in kinds if k is not None):
            idx = [i for i, k in enumerate(kinds) if k == dt]
            members = [i * n_terms + j for i in idx for j in range(n_terms)]
            host = [values[m] for m in members]
            batch = fields_to_batch([flat[m] for m in members], host_values=host if all(h is not None for h in host) else None)
            for i, f in zip(idx, self._device_sums([groups[i] for i in idx], batch)):
                out[i] = f
        for i, k in enumerate(kinds):
            if k is None:
                terms = [np.asarray(f.to_numpy(flatten=True)) if v is None else v for f, v in zip(groups[i], values[i * n_terms : (i + 1) * n_terms])]
                s = terms[0].copy()
                for t in terms[1:]:
                    s += t
                out[i] = new_field_from_numpy(s, template=groups[i][0], param=self.output)
        return out

    def _device_sums(self, groups: list[list[Any]], batch: DeviceBatch) -> list[Any]:
        n_terms = len(self.params)
        out = DeviceBatch(sum_cols(batch.data, list(range(len(groups) * n_terms)), len(groups), n_terms), len(groups))
        if results_are_host_bound():
            out.prefetch()
        # the reference sums flattened arrays (sum.py:110)
        return [new_field_from_device_column(out, i, template=g[0], shape=None, param=self.output) for i, g in enumerate(groups)]

    def backward(self, data: Any) -> Any:
        raise NotImplementedError("Sum filter is not reversible")
