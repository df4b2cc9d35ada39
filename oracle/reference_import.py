"""Import the UNMODIFIED reference (ecmwf/anemoi-transform 0.4.2) behind oracle/refstubs.

TEST INFRASTRUCTURE.  The reference is not part of this repository: point the environment
variable ANEMOI_REFERENCE_SRC at the `src` directory of its source tree (its tests are read
from the sibling `tests` directory).  Used by oracle/make_golden.py and by the CPU tests that
validate the oracle restatements against the live reference (skipped when it is not given).
"""

from __future__ import annotations

import importlib
import os
import sys
from pathlib import Path

REFERENCE_SRC = Path(os.environ["ANEMOI_REFERENCE_SRC"]) if os.environ.get("ANEMOI_REFERENCE_SRC") else None
REFERENCE_TESTS = REFERENCE_SRC.parent / "tests" if REFERENCE_SRC else None
STUBS = Path(__file__).resolve().parent / "refstubs"
REPO = Path(__file__).resolve().parent.parent

HOT_PATH_MODULES = (
    "anemoi.transform.workflows.pipeline",
    "anemoi.transform.spatial",
    "anemoi.transform.filters.fields.regrid",
    "anemoi.transform.filters.fields.uv_to_ddff",
    "anemoi.transform.filters.fields.q_to_r",
    "anemoi.transform.filters.fields.clipper",
    "anemoi.transform.filters.fields.apply_mask",
    # SURVEY §8(f) rank 1: the remaining pointwise field filters
    "anemoi.transform.filters.fields.rescale",
    "anemoi.transform.filters.fields.lnsp_to_sp",
    "anemoi.transform.filters.fields.impute_nans",
    "anemoi.transform.filters.fields.remove_nans",
    "anemoi.transform.filters.fields.cos_sin_from_rad",
    "anemoi.transform.filters.fields.cos_sin_mean_wave_direction",
    "anemoi.transform.filters.fields.dewpoint",
    "anemoi.transform.filters.fields.sum",
    "anemoi.transform.filters.fields.orog_to_z",
)


def available() -> bool:
    return REFERENCE_SRC is not None and (REFERENCE_SRC / "anemoi" / "transform" / "spatial.py").exists()


def load() -> dict[str, object]:
    """→ {short name: module} of the reference's hot-path modules."""
    if not available():
        raise RuntimeError(f"reference sources not found (ANEMOI_REFERENCE_SRC={REFERENCE_SRC})")
    for p in (str(REPO), str(REPO / "anemoi-transform_b200"), str(STUBS), str(REFERENCE_SRC)):
        if p not in sys.path:
            sys.path.insert(0, p)
    mods = {}
    for name in HOT_PATH_MODULES:
        mods[name.rsplit(".", 1)[1]] = importlib.import_module(name)
    return mods
