"""Boundary packaging: the entry-point metadata resolves, and the B200 filters plug into the
REFERENCE's own registry / Pipeline (the latter only when ANEMOI_REFERENCE_SRC points at the
reference's sources, see oracle/reference_import.py)."""

import importlib
import subprocess
import sys
import tomllib
from pathlib import Path

import pytest

from oracle import reference_import

REPO = Path(__file__).resolve().parent.parent
PYPROJECT = REPO / "anemoi-transform_b200" / "pyproject.toml"


def test_every_entry_point_resolves_to_a_filter_factory():
    meta = tomllib.loads(PYPROJECT.read_text())
    group = meta["project"]["entry-points"]["anemoi.transform.filters"]
    assert {"b200_regrid", "b200_uv_to_ddff", "b200_q_to_r", "b200_clip", "b200_mask"} <= set(group)
    for name, target in group.items():
        module, _, attribute = target.partition(":")
        factory = getattr(importlib.import_module(module), attribute)
        assert callable(factory), (name, target)
    from anemoi_transform_b200 import plugin
    from anemoi_transform_b200.filters.fields.regrid import RegridFilter

    assert plugin.regrid is RegridFilter
    with pytest.raises(AttributeError):
        plugin.not_a_filter
    assert meta["tool"]["setuptools"]["package-data"]["anemoi_transform_b200"] == ["lib/libat_b200.so"]


def test_install_replaces_and_adds_names_in_a_registry():
    from anemoi_transform_b200 import plugin
    from anemoi_transform_b200.filters.fields.uv_to_ddff import WindComponents
    from anemoi_transform_b200.registry import Registry

    stock = Registry("somewhere.filters")
    stock.register("uv_to_ddff", lambda **kw: "stock wind")
    stock.register("clip", lambda **kw: "stock clip", aliases=["clipper"])
    stock.register("untouched", lambda **kw: "stock other")
    added = plugin.install(stock, prefix="b200_", names=["uv_to_ddff"])
    assert added == ["b200_uv_to_ddff"] and stock.create("uv_to_ddff") == "stock wind" and isinstance(stock.create("b200_uv_to_ddff"), WindComponents)
    replaced = plugin.install(stock)
    assert "regrid" in replaced and "clipper" in replaced
    assert isinstance(stock.create("uv_to_ddff"), WindComponents) and stock.create("untouched") == "stock other"
    assert type(stock.create("clipper", param="t", minimum=0.0)).__module__.startswith("anemoi_transform_b200")


_IN_REFERENCE = r"""
import sys
sys.path.insert(0, {repo!r}); sys.path.insert(0, {pkg!r})
import numpy as np
from oracle import reference_import
ref = reference_import.load()                      # the UNMODIFIED reference, behind the stubs
import anemoi.transform.filters.fields as ref_fields
from anemoi.transform.workflows.pipeline import Pipeline as RefPipeline
from anemoi.transform.transform import Transform as RefTransform
from anemoi_transform_b200 import _cabi, ekd, plugin
from anemoi_transform_b200 import synthetic as syn

registry = ref_fields.filter_registry                 # holds the reference's regrid, uv_to_ddff, ...
stock_regrid = registry.lookup("regrid")
assert stock_regrid.__module__ == "anemoi.transform.filters.fields.regrid", stock_regrid
added = plugin.install(registry, prefix="b200_")      # next to the stock filters
assert registry.lookup("regrid") is stock_regrid and registry.lookup("b200_regrid").__module__.startswith("anemoi_transform_b200")

s_lat, s_lon = syn.regular_latlon(4.0)
t_lat, t_lon = syn.octahedral(8)
np.savez({tmp!r} + "/m.npz", mask=np.arange(0, s_lat.size, 3))   # a MaskedRegrid: no device work at construction
fields = ekd.from_source("list-of-dicts", [dict(param=q, levelist=850, values=syn.synthetic_field(q, s_lat.size, k), latitudes=s_lat, longitudes=s_lon) for k, q in enumerate(("u", "v"))])

# the reference's own regrid | uv_to_ddff through the reference's Pipeline: CPU, scipy
stock = RefPipeline(filters=[registry.create("regrid", mask={tmp!r} + "/m.npz"), registry.create("uv_to_ddff")])
out = stock.forward(fields)
assert [f.metadata("param") for f in out] == ["ws", "wdir"] and out[0].to_numpy().shape == (len(range(0, s_lat.size, 3)),)

# the same recipe with the B200 filters, assembled by the reference's machinery
mine = RefPipeline(filters=[registry.create("b200_regrid", mask={tmp!r} + "/m.npz"), registry.create("b200_uv_to_ddff")])
assert isinstance(mine, RefTransform) and all(type(f).__module__.startswith("anemoi_transform_b200") for f in mine.filters)
import torch
if torch.cuda.is_available():
    got = mine.forward(fields)
    assert [f.metadata("param") for f in got] == ["ws", "wdir"]
    assert np.allclose(got[0].to_numpy(), out[0].to_numpy(), rtol=1e-6, atol=1e-5)
    print("RAN_ON_GPU")
else:
    try:
        mine.forward(fields)
    except _cabi.NativeLibraryError as e:            # no CPU fallback: the dispatch reached the B200 filter
        assert "no CPU fallback" in str(e)
        print("DISPATCHED_TO_B200")

# install() without a prefix swaps the stock factories themselves; recipes stay as they are
plugin.install(registry)
assert registry.lookup("regrid").__module__.startswith("anemoi_transform_b200")
swapped = registry.create("uv_to_ddff")
assert type(swapped).__module__.startswith("anemoi_transform_b200")
print("OK")
"""


@pytest.mark.reference
@pytest.mark.skipif(not reference_import.available(), reason="reference sources not present")
def test_b200_filters_register_into_the_references_registry_and_run_in_its_pipeline(tmp_path):
    code = _IN_REFERENCE.format(repo=str(REPO), pkg=str(REPO / "anemoi-transform_b200"), tmp=str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    assert "OK" in r.stdout and ("DISPATCHED_TO_B200" in r.stdout or "RAN_ON_GPU" in r.stdout), r.stdout
