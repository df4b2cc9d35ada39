"""Oracle restatements and the filters' host-only behaviour against the outputs of the
UNMODIFIED reference.  The tests without a suffix compare with the reference's outputs stored in
tests/golden/ (reference_checks.npz, patch_data_request.json, oracle/make_golden.py); the
`_live` variants and test_goldens_are_reproducible re-run the reference itself, imported from
ANEMOI_REFERENCE_SRC (oracle/reference_import.py), and skip without it."""

import copy
import json

import numpy as np
import pytest
from conftest import GOLDEN

from anemoi_transform_b200 import synthetic as syn
from oracle import make_golden as mg
from oracle import reference_import
from oracle import spatial as osp

live = pytest.mark.skipif(not reference_import.available(), reason="reference sources not present")


@pytest.fixture(scope="module")
def ref():
    return reference_import.load()


@pytest.fixture(scope="module")
def stored():
    return dict(np.load(GOLDEN / "reference_checks.npz"))


def _stored_requests():
    cases = json.loads((GOLDEN / "patch_data_request.json").read_text())
    assert [(c["filter"], c["kwargs"], c["request"]) for c in cases] == [(n, kw, r) for n, kw, reqs in mg.PATCH_DATA_REQUEST_CASES for r in reqs]
    return cases


def _spatial_outputs(sp, lam, glob, cutout_default):
    return {
        "cutout": cutout_default(*lam, *glob),
        "cutout_50_900": sp.cutout_mask(*lam, *glob, min_distance_km=50, max_distance_km=900),
        "thinning": sp.thinning_mask(*lam, *glob),
        "global_on_lam": sp.global_on_lam_mask(*lam, *glob),
        "ngp_k3": sp.nearest_grid_points(*glob, *lam, num_neighbours_to_return=3),
    }


def test_spatial_functions_agree_on_random_inputs(stored):
    for seed, lam, glob in mg.spatial_random_cases(syn):
        for name, got in _spatial_outputs(osp, lam, glob, osp.cutout_mask_vectorised).items():
            assert np.array_equal(got, stored[f"spatial{seed}_{name}"]), (seed, name)


@pytest.mark.reference
@live
def test_spatial_functions_agree_on_random_inputs_live(ref, stored):
    sp = ref["spatial"]
    for seed, lam, glob in mg.spatial_random_cases(syn):
        want = _spatial_outputs(sp, lam, glob, sp.cutout_mask)
        got = _spatial_outputs(osp, lam, glob, osp.cutout_mask_vectorised)
        for name in want:
            assert np.array_equal(want[name], got[name]) and np.array_equal(want[name], stored[f"spatial{seed}_{name}"]), (seed, name)


@pytest.mark.reference
@live
def test_goldens_are_reproducible(ref, golden_spatial):
    g = golden_spatial
    sp = ref["spatial"]
    assert np.array_equal(sp.cutout_mask(g["lam_lat"], g["lam_lon"], g["o_lat"], g["o_lon"]), g["cutout_default"])
    assert np.array_equal(sp.nearest_grid_points(g["g_lat"], g["g_lon"], g["o_lat"], g["o_lon"]), g["ngp_k1"])


def test_patch_data_request_matches_the_reference_filters():
    """Host-only behaviour of the product's filters against the reference's classes: the
    `patch_data_request` rewrites (no GPU involved)."""
    from anemoi_transform_b200.filters import create_filter_by_name as F

    for case in _stored_requests():
        got = F(case["filter"], **case["kwargs"]).patch_data_request(copy.deepcopy(case["request"]))
        assert json.loads(json.dumps(got)) == case["result"], case
    for both, flt in (({"param": ["sp", "lnsp"]}, F("lnsp_to_sp")), ({"param": ["z", "orog"]}, F("orog_to_z_fields"))):
        with pytest.raises(ValueError, match="cannot contain both"):
            flt.patch_data_request(both)


@pytest.mark.reference
@live
def test_patch_data_request_matches_the_reference_filters_live(ref):
    from anemoi_transform_b200.filters import create_filter_by_name as F

    theirs = {
        "orog_to_z_fields": lambda: ref["orog_to_z"].Orography(),
        "lnsp_to_sp": lambda: ref["lnsp_to_sp"].LnspToSp(),
        "cos_sin_from_rad": lambda param: ref["cos_sin_from_rad"].CosSinFromRad(param=param),
        "cos_sin_mean_wave_direction": lambda: ref["cos_sin_mean_wave_direction"].CosSinWaveDirection(),
    }
    for case in _stored_requests():
        mine = F(case["filter"], **case["kwargs"]).patch_data_request(copy.deepcopy(case["request"]))
        want = theirs[case["filter"]](**case["kwargs"]).patch_data_request(copy.deepcopy(case["request"]))
        assert mine == want and json.loads(json.dumps(want)) == case["result"], case
