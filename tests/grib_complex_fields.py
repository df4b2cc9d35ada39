"""A stand-in for earthkit-data's `GribField` that also reads complex-packed messages (test
infrastructure): `GribMessageField` (tests/grib_fields.py) whose host decode goes through
`oracle.grib_complex.decode`, which reads templates 5.2 and 5.3 and hands every other template
to `oracle.grib_ccsds.decode` (5.42) and `oracle.grib.decode`."""

from __future__ import annotations

from grib_fields import GribMessageField

from oracle import grib_complex as ogx


class ComplexGribField(GribMessageField):
    def to_numpy(self, flatten: bool = False, dtype=None, index=None):
        self.decodes += 1
        v = ogx.decode(self._message, n_points=self._n_points)
        if dtype is not None:
            v = v.astype(dtype)
        if index is not None:
            v = v[index]
        return v
