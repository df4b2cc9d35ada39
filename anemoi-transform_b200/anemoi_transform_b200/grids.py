"""Named grids.  The reference downloads `grid-{name}.npz` from get.ecmwf.int
(`grids/named.py:27-88`); offline, the grids this package can generate itself are served
from `synthetic` (octahedral O-grids and HEALPix H-grids are exact; see tests/test_grids)."""

from __future__ import annotations

import re
from typing import Any

import numpy as np

from . import synthetic


def lookup(name: Any) -> dict[str, np.ndarray]:
    """The points of a named grid: "O<n>" (octahedral), [d, d] (regular lat-lon), "H<nside>"
    (HEALPix, ring order as earthkit-regrid defaults), or a gridspec dict {"grid": name} with,
    for HEALPix, "ordering": "ring" | "nested".  ValueError for anything else, naming the key
    of a gridspec dict that cannot be honoured."""
    if isinstance(name, dict):
        if "grid" not in name:
            raise ValueError(f"Invalid grid: {name}: a gridspec dict needs a 'grid' key")
        grid, ordering = name["grid"], name.get("ordering")
        healpix = isinstance(grid, str) and re.fullmatch(r"[hH]\d+", grid) is not None
        for key in name:
            if key != "grid" and not (key == "ordering" and healpix):
                raise ValueError(f"Invalid grid: {name}: the gridspec key {key!r} is not supported for grid {grid!r}")
        if healpix:
            if ordering is not None and ordering not in ("ring", "nested"):
                raise ValueError(f"Invalid grid: {name}: 'ordering' must be 'ring' or 'nested', not {ordering!r}")
            lat, lon = synthetic.healpix(int(grid[1:]), ordering or "ring")
            return dict(latitudes=lat, longitudes=lon)
        return lookup(grid)
    if isinstance(name, (list, tuple)):
        if len(name) == 2 and float(name[0]) == float(name[1]):
            lat, lon = synthetic.regular_latlon(float(name[0]))
            return dict(latitudes=lat, longitudes=lon)
        raise ValueError(f"Invalid grid: {name}")
    key = str(name).lower()
    m = re.fullmatch(r"o(\d+)", key)
    if m:
        lat, lon = synthetic.octahedral(int(m.group(1)))
        return dict(latitudes=lat, longitudes=lon)
    m = re.fullmatch(r"h(\d+)", key)
    if m:
        lat, lon = synthetic.healpix(int(m.group(1)))
        return dict(latitudes=lat, longitudes=lon)
    raise ValueError(f"Unknown grid {name!r}: only octahedral O-grids, HEALPix H-grids and regular [d, d] grids are generated offline")


def icon_grid(path: str, refinement_level_c: int | None = None) -> tuple[np.ndarray, np.ndarray]:
    """Cell-centre latitudes / longitudes (degrees) of an ICON grid file, optionally only the
    cells with `refinement_level_c <= refinement_level_c` (reference `grids/icon.py:22-53`).

    ICON grid files are NetCDF (`clat`, `clon` in radians, `refinement_level_c`); they are read
    with xarray when it is installed.  A `.npz` with the same three arrays is accepted as well,
    so the filter can be used (and tested) where xarray / netCDF are not available."""
    if str(path).endswith(".npz"):
        ds = np.load(path)
        clat, clon, level = ds["clat"], ds["clon"], ds["refinement_level_c"] if "refinement_level_c" in ds.files else None
    else:
        try:
            import xarray as xr
        except ImportError as e:  # pragma: no cover - depends on the environment
            raise ImportError(f"reading the ICON grid {path} needs xarray (or provide clat / clon / refinement_level_c as .npz)") from e
        ds = xr.open_dataset(path)
        clat, clon, level = ds.clat.values, ds.clon.values, ds.refinement_level_c.values
    if refinement_level_c is not None:
        if level is None:
            raise ValueError(f"{path} has no refinement_level_c")
        keep = level <= refinement_level_c
        clat, clon = clat[keep], clon[keep]
    return np.rad2deg(clat), np.rad2deg(clon)
