"""The drop-in spatial functions against the imported reference's golden outputs, the
reference's known-answer tests and the oracle on mid-size grids."""

import numpy as np
import pytest

from anemoi_transform_b200 import synthetic as syn
from oracle import spatial as osp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sp(cuda):
    from anemoi_transform_b200 import spatial

    return spatial


def _lam11():
    la, lo = np.meshgrid(np.linspace(44.0, 46.0, 11), np.linspace(0.0, 2.0, 11))
    return la.flatten(), lo.flatten()


# ---- reference tests/test_spatial.py ported verbatim in spirit -------------------------------
@pytest.mark.parametrize("cropping_distance", [1.0, 3.0, 5.0])
def test_cutout_mask_with_max_distance(sp, cropping_distance):
    lam_lats, lam_lons = _lam11()
    mask = sp.cutout_mask(lam_lats, lam_lons, np.array([43.1, 44.0, 45.0, 45.5, 46.0, 50.0]), np.array([359.1, 359.5, 0.0, 1.0, 2.0, 0.0]), cropping_distance=cropping_distance, max_distance_km=250.0)
    assert isinstance(mask, np.ndarray) and mask.shape == (6,)
    assert np.array_equal(mask, np.array([True, False, False, False, False, False]))


def test_cutout_mask_with_min_distance(sp):
    lam_lats, lam_lons = _lam11()
    mask = sp.cutout_mask(lam_lats, lam_lons, np.array([44.0, 45.0, 46.0, 46.1, 47.5]), np.array([0.0, 1.0, 2.0, -0.1, -1.5]), min_distance_km=100.0)
    assert np.array_equal(mask, np.array([False, False, False, False, True]))


def test_cutout_mask_array_shapes(sp):
    with pytest.raises(AssertionError):
        sp.cutout_mask(np.array([[45.0, 45.0], [46.0, 46.0]]), np.array([[0.0, 1.0], [0.0, 1.0]]), np.array([45.0]), np.array([0.0]))


def test_cutout_mask_parameter_types(sp):
    lam_lats, lam_lons = _lam11()
    g = (np.array([45.0, 46.0]), np.array([0.0, 2.0]))
    assert isinstance(sp.cutout_mask(lam_lats, lam_lons, *g, max_distance_km=100), np.ndarray)
    assert isinstance(sp.cutout_mask(lam_lats, lam_lons, *g, max_distance_km=100.0), np.ndarray)
    with pytest.raises(AssertionError, match="neighbours must be positive"):
        sp.cutout_mask(lam_lats, lam_lons, *g, neighbours=0)
    with pytest.raises(AssertionError, match="cropping_distance must be non-negative"):
        sp.cutout_mask(lam_lats, lam_lons, *g, cropping_distance=-1.0)


def test_cutout_mask_large_grid(sp):
    la, lo = np.meshgrid(np.linspace(40.0, 50.0, 21), np.linspace(0.0, 10.0, 21))
    gla, glo = np.meshgrid(np.linspace(30.0, 60.0, 31), np.linspace(-10.0, 20.0, 31))
    args = (la.flatten(), lo.flatten(), gla.flatten(), glo.flatten())
    mask = sp.cutout_mask(*args, min_distance_km=150.0, max_distance_km=300.0)
    assert mask.shape == (961,) and mask.dtype == bool and np.any(mask) and not np.all(mask)
    assert np.array_equal(mask, osp.cutout_mask(*args, min_distance_km=150.0, max_distance_km=300.0))


# ---- golden outputs of the imported reference -----------------------------------------------
def test_golden_nearest_grid_points(sp, golden_spatial):
    g = golden_spatial
    idx = sp.nearest_grid_points(g["g_lat"], g["g_lon"], g["o_lat"], g["o_lon"])
    assert idx.dtype == np.int64 and idx.shape == g["ngp_k1"].shape
    i_t, d_t, ties = sp.nearest_grid_points(g["g_lat"], g["g_lon"], g["o_lat"], g["o_lon"], _return_ties=True)
    assert not ((idx != g["ngp_k1"]) & (ties == 0)).any()
    i4, d4 = sp.nearest_grid_points(g["g_lat"], g["g_lon"], g["lam_lat"], g["lam_lon"], num_neighbours_to_return=4, return_distances=True)
    assert np.array_equal(d4, g["ngp_k4_dist"]) and i4.shape == (720, 4)
    assert np.array_equal(i4, g["ngp_k4_idx"])  # rotated LAM vs lat-lon grid: no exact ties
    iu, du = sp.nearest_grid_points(g["lam_lat"], g["lam_lon"], g["o_lat"], g["o_lon"], max_distance=0.01, return_distances=True)
    assert np.array_equal(iu, g["ngp_ub_idx"]) and np.array_equal(du, g["ngp_ub_dist"])


def test_golden_masks(sp, golden_spatial):
    g = golden_spatial
    lam, o = (g["lam_lat"], g["lam_lon"]), (g["o_lat"], g["o_lon"])
    assert np.array_equal(sp.cropping_mask(g["g_lat"], g["g_lon"], 70.0, -20.0, 40.0, 15.0), g["crop_wrap"])
    t = sp.thinning_mask(*lam, *o)
    assert t.dtype == np.int64 and np.array_equal(t, g["thinning"])
    assert np.array_equal(sp.thinning_mask(*lam, g["g_lat"], g["g_lon"], cropping_distance=6.0), g["thinning_crop6"])
    m = sp.global_on_lam_mask(*lam, *o)
    assert m.dtype == np.int64 and np.array_equal(m, g["gol_none"])
    assert np.array_equal(sp.global_on_lam_mask(*lam, *o, distance_km=150.0), g["gol_150km"])
    empty = sp.global_on_lam_mask(*lam, *o, distance_km=1.0)
    assert empty.shape == (0,) and empty.dtype == np.float64


@pytest.mark.parametrize("dot_mode", [1, 0])
def test_golden_cutout(sp, golden_spatial, dot_mode, monkeypatch):
    monkeypatch.setattr(sp, "CUTOUT_DOT_MODE", dot_mode)
    g = golden_spatial
    lam, o = (g["lam_lat"], g["lam_lon"]), (g["o_lat"], g["o_lon"])
    assert np.array_equal(sp.cutout_mask(*lam, *o), g["cutout_default"])
    assert np.array_equal(sp.cutout_mask(*lam, *o, min_distance_km=80.0, max_distance_km=400.0), g["cutout_min80_max400"])
    assert np.array_equal(sp.cutout_mask(*lam, *o, cropping_distance=5.0, neighbours=3, min_distance_km=10), g["cutout_n3_crop5"])
    assert np.array_equal(sp.cutout_mask(*lam, g["g_lat"], g["g_lon"]), g["cutout_regular_default"])


# ---- mid-size grids against the oracle -----------------------------------------------------
def test_midsize_lam_in_global(sp):
    """A 200x240 LAM at 0.05° inside O160: cutout / thinning / global-on-lam against the oracle."""
    lam = syn.rotated_lam(200, 240, 0.05, 55.0, 15.0)
    glob = syn.octahedral(160)
    assert np.array_equal(sp.cutout_mask(*lam, *glob), osp.cutout_mask_vectorised(*lam, *glob))
    assert np.array_equal(sp.cutout_mask(*lam, *glob, min_distance_km=20, max_distance_km=150), osp.cutout_mask_vectorised(*lam, *glob, min_distance_km=20, max_distance_km=150))
    assert np.array_equal(sp.thinning_mask(*lam, *glob), osp.thinning_mask(*lam, *glob))
    assert np.array_equal(sp.global_on_lam_mask(*lam, *glob), osp.global_on_lam_mask(*lam, *glob))
    assert np.array_equal(sp.global_on_lam_mask(*lam, *glob, distance_km=40.0), osp.global_on_lam_mask(*lam, *glob, distance_km=40.0))


def test_lam_straddling_longitude_zero_far_queries(sp):
    """Like BASELINE config 5: the LAM crosses lon 0, so the reference's crop box spans every
    longitude and most cropped global points are far from the LAM (tree-search path)."""
    lam = syn.rotated_lam(150, 150, 0.1, 60.0, 10.0)
    assert lam[1].min() < 1.0 and lam[1].max() > 359.0
    glob = syn.octahedral(96)
    got, want = sp.thinning_mask(*lam, *glob), osp.thinning_mask(*lam, *glob)
    assert got.shape == want.shape and got.size > 2000
    differ = np.nonzero(got != want)[0]
    if differ.size:  # only exact float64 d² ties may differ (mirror-image LAM points)
        lp = np.array(osp.latlon_to_xyz(*lam)).T
        crop = osp._crop(lam[0], lam[1], glob[0], glob[1], 2.0)
        gp = np.array(osp.latlon_to_xyz(glob[0][crop], glob[1][crop])).T[differ]
        assert np.array_equal(((lp[got[differ]] - gp) ** 2).sum(axis=1), ((lp[want[differ]] - gp) ** 2).sum(axis=1))
        assert differ.size < 50
    assert np.array_equal(sp.cutout_mask(*lam, *glob), osp.cutout_mask_vectorised(*lam, *glob))
    assert np.array_equal(sp.cutout_mask(*lam, *glob, max_distance_km=500.0), osp.cutout_mask_vectorised(*lam, *glob, max_distance_km=500.0))
    assert np.array_equal(sp.global_on_lam_mask(*lam, *glob), osp.global_on_lam_mask(*lam, *glob))
    assert np.array_equal(sp.global_on_lam_mask(*lam, *glob, distance_km="lam"), osp.global_on_lam_mask(*lam, *glob, distance_km="lam"))


def test_sharded_entry_points_equal_the_single_gpu_ones(sp, golden_spatial):
    """distributed.* with world_size 1 (no process group): same answers as spatial.*."""
    from anemoi_transform_b200 import distributed as atd

    g = golden_spatial
    lam, o = (g["lam_lat"], g["lam_lon"]), (g["o_lat"], g["o_lon"])
    assert np.array_equal(atd.nearest_grid_points(*lam, *o, num_neighbours_to_return=3), sp.nearest_grid_points(*lam, *o, num_neighbours_to_return=3))
    assert np.array_equal(atd.global_on_lam_mask(*lam, *o), g["gol_none"])
    assert np.array_equal(atd.global_on_lam_mask(*lam, *o, distance_km=150.0), g["gol_150km"])


def test_global_on_lam_mask_file_feeds_the_masked_regrid(sp, golden_spatial, tmp_path):
    """make-regrid-file global-on-lam-mask → regrid(mask=…): the file written on the device path
    selects exactly the points the reference's mask selects."""
    from anemoi_transform_b200 import ekd
    from anemoi_transform_b200.filters import create_filter_by_name
    from anemoi_transform_b200.regrid_files import make_global_on_lam_mask

    g = golden_spatial
    mask = make_global_on_lam_mask(g["lam_lat"], g["lam_lon"], g["o_lat"], g["o_lon"], str(tmp_path / "gol.npz"), distance_km=150.0)
    assert np.array_equal(mask, g["gol_150km"]) and np.array_equal(np.load(tmp_path / "gol.npz")["mask"], g["gol_150km"])
    rng = np.random.default_rng(1)
    vals = rng.normal(size=g["o_lat"].size).astype(np.float32)
    fl = ekd.from_source("list-of-dicts", [dict(param="t", levelist=1, values=vals, latitudes=g["o_lat"], longitudes=g["o_lon"])])
    out = create_filter_by_name("regrid", mask=str(tmp_path / "gol.npz")).forward(fl)
    assert np.array_equal(out[0].to_numpy(flatten=True), vals[g["gol_150km"]])
    lat, lon = out[0].grid_points()
    assert np.array_equal(lat, g["o_lat"][g["gol_150km"]]) and np.array_equal(lon, g["o_lon"][g["gol_150km"]])


def test_locally_built_knn_matrix_feeds_the_regrid_filter(sp, tmp_path):
    """regrid_files.make_knn_matrix: k = 1 is nearest-neighbour regridding as a matrix (same values
    as `regrid(method="nearest")`, up to the sign of zero); k = 4 rows are convex weights."""
    from anemoi_transform_b200 import ekd
    from anemoi_transform_b200.filters import create_filter_by_name
    from anemoi_transform_b200.regrid_files import make_knn_matrix

    s_lat, s_lon = syn.regular_latlon(2.0)
    t_lat, t_lon = syn.octahedral(24)
    rng = np.random.default_rng(5)
    vals = [rng.normal(280, 10, s_lat.size).astype(np.float32) for _ in range(5)]
    fl = ekd.from_source("list-of-dicts", [dict(param="t", levelist=k, values=v, latitudes=s_lat, longitudes=s_lon) for k, v in enumerate(vals)])
    make_knn_matrix(s_lat, s_lon, t_lat, t_lon, str(tmp_path / "nn.npz"), k=1)
    via_matrix = create_filter_by_name("regrid", matrix=str(tmp_path / "nn.npz")).forward(fl)
    via_gather = create_filter_by_name("regrid", method="nearest", in_grid=dict(latitudes=s_lat, longitudes=s_lon), out_grid=dict(latitudes=t_lat, longitudes=t_lon)).forward(fl)
    for a, b in zip(via_matrix, via_gather):
        assert np.array_equal(a.to_numpy(flatten=True), b.to_numpy(flatten=True))
    d, i, p, shape = make_knn_matrix(s_lat, s_lon, t_lat, t_lon, k=4, power=2.0)
    assert shape == (t_lat.size, s_lat.size) and d.dtype == np.float32 and i.dtype == np.int32
    w = d.reshape(-1, 4)
    assert np.all(w >= 0) and np.allclose(w.sum(axis=1), 1.0, atol=1e-6) and np.all(np.diff(i.reshape(-1, 4), axis=1) > 0)
    on_source = np.nonzero((np.isin(t_lat, s_lat)) & (np.isin(t_lon, s_lon)))[0]
    for r in on_source[:5]:  # a target on a source point takes that source alone
        assert np.sort(w[r])[-1] == 1.0


def test_outline_matches_the_reference(sp, golden_spatial):
    """spatial.outline (self-kNN + triangle fan from the second neighbour) against the reference's
    outputs on a scattered patch (no tied neighbour distances: exact) and on the rotated LAM."""
    g = golden_spatial
    assert sp.outline(g["patch_lat"], g["patch_lon"]) == g["outline_patch"].tolist()
    assert sp.outline(g["patch_lat"], g["patch_lon"], neighbours=7) == g["outline_patch_n7"].tolist()
    got = sp.outline(g["lam_lat"], g["lam_lon"])
    if got != g["outline_lam"].tolist():
        # a regular LAM has exactly tied neighbour distances: the fan order is cKDTree's traversal
        # order there; with cKDTree's own neighbour order the classification must agree exactly
        from scipy.spatial import cKDTree

        pts = np.array(osp.latlon_to_xyz(g["lam_lat"], g["lam_lon"])).T
        _, idx = cKDTree(pts).query(pts, k=5)
        assert osp.outline(g["lam_lat"], g["lam_lon"], indices=idx) == g["outline_lam"].tolist()
        d = np.sqrt(((pts[:, None, :] - pts[idx]) ** 2).sum(axis=2))
        tied = (np.diff(d, axis=1) == 0).any(axis=1)
        assert set(got) ^ set(g["outline_lam"].tolist()) <= set(np.nonzero(tied)[0].tolist())
    assert sp.outline(np.zeros(0), np.zeros(0)) == []


def test_random_lam_cases_match_the_reference_outputs(sp):
    """The reference's outputs on three random LAM / global pairs (tests/golden/reference_checks.npz)."""
    from conftest import GOLDEN

    from oracle import make_golden as mg

    stored = np.load(GOLDEN / "reference_checks.npz")
    for seed, lam, glob in mg.spatial_random_cases(syn):
        assert np.array_equal(sp.cutout_mask(*lam, *glob), stored[f"spatial{seed}_cutout"]), seed
        assert np.array_equal(sp.cutout_mask(*lam, *glob, min_distance_km=50, max_distance_km=900), stored[f"spatial{seed}_cutout_50_900"]), seed
        assert np.array_equal(sp.thinning_mask(*lam, *glob), stored[f"spatial{seed}_thinning"]), seed
        assert np.array_equal(sp.global_on_lam_mask(*lam, *glob), stored[f"spatial{seed}_global_on_lam"]), seed
        assert np.array_equal(sp.nearest_grid_points(*glob, *lam, num_neighbours_to_return=3), stored[f"spatial{seed}_ngp_k3"]), seed
