"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported behind
oracle/refstubs, see oracle/reference_import.py) on small seeded inputs.

TEST INFRASTRUCTURE.  Run:   ANEMOI_REFERENCE_SRC=<reference>/src python oracle/make_golden.py

What is pinned by these files
    spatial_*.npz    reference spatial.py on live scipy cKDTree (real arithmetic of the path)
    regrid_*.npz     reference RegridFilter (MIRMatrix / nearest / mask) on live scipy.sparse
    filters_more.npz reference Rescale / LnspToSp / ImputeNaNs / RemoveNaNs / CosSinFromRad /
                     CosSinWaveDirection / DewPoint / Sum (SURVEY §8f rank 1), same caveat for the
                     dewpoint VALUES (earthkit-meteo → oracle/pointwise.py, pinned by the
                     reference's test_dewpoint.py:23-27)
    filters.npz      reference WindComponents / HumidityConversion / Clipper / MaskVariable:
                     grouping, output ordering, metadata and dtypes are the reference's; the
                     wind / humidity VALUES come from oracle/pointwise.py through the
                     earthkit.meteo stub (earthkit-meteo itself is unavailable), so for
                     those values the pin is the reference's own golden vectors, not this file.
    reference_checks.npz, patch_data_request.json
                     reference cutout / thinning / global-on-LAM masks and k=3 neighbours on three
                     random LAM / global pairs, superob (binning and result frame) and the
                     patch_data_request rewrites of four filters: see reference_checks() below
"""

from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "anemoi-transform_b200"))

from oracle import reference_import  # noqa: E402

GOLDEN = REPO / "tests" / "golden"


def spatial_cases(sp, syn):
    lam_lat, lam_lon = syn.rotated_lam(24, 30, 0.5, 60.0, 10.0)
    g_lat, g_lon = syn.regular_latlon(3.0)
    o_lat, o_lon = syn.octahedral(24)
    out = dict(lam_lat=lam_lat, lam_lon=lam_lon, g_lat=g_lat, g_lon=g_lon, o_lat=o_lat, o_lon=o_lon)
    # cutout_mask variants (global = octahedral grid: no exact neighbour ties with the rotated LAM)
    out["cutout_default"] = sp.cutout_mask(lam_lat, lam_lon, o_lat, o_lon)
    out["cutout_min80_max400"] = sp.cutout_mask(lam_lat, lam_lon, o_lat, o_lon, min_distance_km=80.0, max_distance_km=400.0)
    out["cutout_n3_crop5"] = sp.cutout_mask(lam_lat, lam_lon, o_lat, o_lon, cropping_distance=5.0, neighbours=3, min_distance_km=10)
    out["cutout_regular_default"] = sp.cutout_mask(lam_lat, lam_lon, g_lat, g_lon)
    out["thinning"] = sp.thinning_mask(lam_lat, lam_lon, o_lat, o_lon)
    out["thinning_crop6"] = sp.thinning_mask(lam_lat, lam_lon, g_lat, g_lon, cropping_distance=6.0)
    out["gol_none"] = sp.global_on_lam_mask(lam_lat, lam_lon, o_lat, o_lon)
    out["gol_150km"] = sp.global_on_lam_mask(lam_lat, lam_lon, o_lat, o_lon, distance_km=150.0)
    out["gol_1km_empty"] = sp.global_on_lam_mask(lam_lat, lam_lon, o_lat, o_lon, distance_km=1.0)
    out["ngp_k1"] = sp.nearest_grid_points(g_lat, g_lon, o_lat, o_lon)
    i4, d4 = sp.nearest_grid_points(g_lat, g_lon, lam_lat, lam_lon, num_neighbours_to_return=4, return_distances=True)
    out["ngp_k4_idx"], out["ngp_k4_dist"] = i4, d4
    iu, du = sp.nearest_grid_points(lam_lat, lam_lon, o_lat, o_lon, max_distance=0.01, return_distances=True)
    out["ngp_ub_idx"], out["ngp_ub_dist"] = iu, du
    out["crop_wrap"] = sp.cropping_mask(g_lat, g_lon, 70.0, -20.0, 40.0, 15.0)
    out["crop_plus360"] = sp.cropping_mask(g_lat, g_lon - 360.0, 10.0, 100.0, -10.0, 140.0)
    x, y, z = sp.latlon_to_xyz(o_lat, o_lon)
    out["o_x"], out["o_y"], out["o_z"] = x, y, z
    la, lo = sp.xyz_to_latlon(x, y, z)
    out["o_lat_back"], out["o_lon_back"] = la, lo
    # outline of a scattered patch (no exactly tied neighbour distances) and of the rotated LAM
    rng = np.random.default_rng(77)
    out["patch_lat"], out["patch_lon"] = rng.uniform(35, 60, 900), rng.uniform(-10, 30, 900)
    out["outline_patch"] = np.array(sp.outline(out["patch_lat"], out["patch_lon"]), dtype=np.int64)
    out["outline_patch_n7"] = np.array(sp.outline(out["patch_lat"], out["patch_lon"], neighbours=7), dtype=np.int64)
    out["outline_lam"] = np.array(sp.outline(lam_lat, lam_lon), dtype=np.int64)
    np.savez_compressed(GOLDEN / "spatial_small.npz", **out)
    print("spatial_small.npz:", {k: (v.shape, str(v.dtype)) for k, v in out.items() if k.startswith(("cutout", "thin", "gol", "ngp"))})


def _fieldlist(ekd, specs, lat, lon):
    return ekd.from_source(
        "list-of-dicts",
        [dict(param=p, levelist=lev, valid_datetime="2020-01-01T00:00:00", values=v, latitudes=lat, longitudes=lon) for p, lev, v in specs],
    )


def regrid_cases(mods, syn, ekd, tmp: Path):
    regrid = mods["regrid"]
    s_lat, s_lon = syn.regular_latlon(5.0)
    t_lat, t_lon = syn.octahedral(16)
    data, idx, ptr, shape = syn.bilinear_matrix(5.0, t_lat, t_lon)
    syn.save_regrid_npz(tmp / "m32.npz", data, idx, ptr, shape, s_lat, s_lon, t_lat, t_lon)
    # an irregular float64 matrix: empty rows, 1..7 entries, unsorted columns, explicit zeros
    rng = np.random.default_rng(7)
    n_t, n_s = 257, s_lat.size
    lens = rng.integers(0, 8, n_t)
    ptr64 = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    idx64 = rng.integers(0, n_s, ptr64[-1]).astype(np.int64)
    dat64 = rng.normal(size=ptr64[-1])
    dat64[rng.uniform(size=dat64.size) < 0.1] = 0.0
    irr_lat, irr_lon = rng.uniform(-90, 90, n_t), rng.uniform(0, 360, n_t)
    syn.save_regrid_npz(tmp / "m64.npz", dat64, idx64, ptr64, (n_t, n_s), s_lat, s_lon, irr_lat, irr_lon)

    fields32 = [syn.synthetic_field(p, n_s, seed, 0.01 if seed % 2 else 0.0) for seed, p in enumerate(["t", "u", "v", "q", "t", "z"])]
    fields32[1][5] = np.inf
    fields64 = [f.astype(np.float64) * 1.000000123 for f in fields32[:3]]
    specs32 = [(p, 500 + i, v) for i, (p, v) in enumerate(zip(["t", "u", "v", "q", "t", "z"], fields32))]
    specs64 = [(p, 500 + i, v) for i, (p, v) in enumerate(zip(["t", "u", "v"], fields64))]
    out = dict(
        s_lat=s_lat, s_lon=s_lon, t_lat=t_lat, t_lon=t_lon, m32_data=data, m32_indices=idx, m32_indptr=ptr, m32_shape=np.asarray(shape),
        m64_data=dat64, m64_indices=idx64, m64_indptr=ptr64, m64_shape=np.asarray((n_t, n_s)), irr_lat=irr_lat, irr_lon=irr_lon,
        fields32=np.stack(fields32), fields64=np.stack(fields64),
    )  # fmt: skip

    def run(filter_, specs):
        res = filter_.forward(_fieldlist(ekd, specs, s_lat, s_lon))
        vals = [f.to_numpy(flatten=True) for f in res]
        lat, lon = res[0].grid_points()
        return np.stack(vals), lat, lon, [f.metadata("param") for f in res]

    y, lat, lon, params = run(regrid.RegridFilter(matrix=str(tmp / "m32.npz")), specs32)
    out["y_m32_f32"], out["y_m32_lat"], out["y_m32_lon"] = y, lat, lon
    assert y.dtype == np.float32 and params == ["t", "u", "v", "q", "t", "z"]
    out["y_m32_f64"] = run(regrid.RegridFilter(matrix=str(tmp / "m32.npz")), specs64)[0]
    out["y_m64_f32"] = run(regrid.RegridFilter(matrix=str(tmp / "m64.npz")), specs32)[0]
    out["y_m64_f64"] = run(regrid.RegridFilter(matrix=str(tmp / "m64.npz")), specs64)[0]
    # nearest neighbours
    y, lat, lon, _ = run(
        regrid.RegridFilter(method="nearest", in_grid=dict(latitudes=s_lat, longitudes=s_lon), out_grid=dict(latitudes=t_lat, longitudes=t_lon)), specs32
    )
    out["y_nearest_f32"], out["y_nearest_lat"] = y, lat
    # index mask (as written by make-regrid-file global-on-lam-mask) and boolean mask
    sel = np.sort(rng.choice(n_s, 300, replace=False)).astype(np.int64)
    np.savez(tmp / "mask_idx.npz", mask=sel)
    y, lat, lon, _ = run(regrid.RegridFilter(mask=str(tmp / "mask_idx.npz")), specs32)
    out["mask_idx"], out["y_mask_f32"], out["y_mask_lat"], out["y_mask_lon"] = sel, y, lat, lon
    np.savez_compressed(GOLDEN / "regrid_small.npz", **out)
    print("regrid_small.npz:", {k: (v.shape, str(v.dtype)) for k, v in out.items() if k.startswith("y_")})


def filter_cases(mods, syn, ekd):
    rng = np.random.default_rng(11)
    lat = np.linspace(60, -60, 25)
    lon = np.linspace(0, 345, 24)
    n = lat.size * lon.size
    LAT, LON = (a.reshape(-1) for a in np.meshgrid(lat, lon, indexing="ij"))

    def fl(specs):
        return _fieldlist(ekd, specs, LAT, LON)

    out, order = {}, {}

    def record(name, result):
        order[name] = [[f.metadata("param"), int(f.metadata("levelist")), str(f.to_numpy().dtype)] for f in result]
        out[name] = np.stack([f.to_numpy(flatten=True).astype(np.float64) for f in result])

    u = {lev: rng.normal(0, 8, n).astype(np.float32) for lev in (500, 850)}
    v = {lev: rng.normal(0, 8, n).astype(np.float32) for lev in (500, 850)}
    specials = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-30, -1e-30, 3.0], dtype=np.float32)
    u[500][:8] = specials
    v[500][:8] = specials[::-1]
    u[850][:4] = [0.0, 0.0, -0.0, -0.0]
    v[850][:4] = [0.0, -0.0, 0.0, -0.0]
    t = {lev: rng.normal(265, 20, n).astype(np.float32) for lev in (500, 850)}
    q = {lev: rng.uniform(1e-6, 2e-2, n).astype(np.float32) for lev in (500, 850)}
    t[850][:3] = [250.16, 273.16, np.nan]
    z = rng.normal(5e4, 1e3, n).astype(np.float32)
    lsm = (rng.uniform(size=n) > 0.6).astype(np.float32)
    mixed = [("t", 850, t[850]), ("u", 850, u[850]), ("z", 500, z), ("v", 850, v[850]), ("u", 500, u[500]), ("q", 850, q[850]), ("v", 500, v[500]), ("t", 500, t[500]), ("q", 500, q[500]), ("lsm", 0, lsm)]
    out["in_values"] = np.stack([m[2] for m in mixed])
    order["in"] = [[m[0], m[1]] for m in mixed]
    out["lat"], out["lon"] = LAT, LON

    uv = mods["uv_to_ddff"].WindComponents()
    ddff = uv.forward(fl(mixed))
    record("uv_to_ddff", ddff)
    record("ddff_to_uv", uv.backward(ddff))
    qr = mods["q_to_r"].HumidityConversion()
    r_all = qr.forward(fl(mixed))
    record("q_to_r_all", r_all)
    record("q_to_r_none", mods["q_to_r"].HumidityConversion(return_inputs="none").forward(fl(mixed)))
    only_rt = [f for f in r_all if f.metadata("param") in ("r", "t")]
    record("r_to_q_all", qr.backward(ekd.SimpleFieldList(only_rt)))
    record("clip_t_both", mods["clipper"].Clipper(param="t", minimum=250.0, maximum=280.0).forward(fl(mixed)))
    record("clip_q_min", mods["clipper"].Clipper(param="q", minimum=0.005).forward(fl(mixed)))
    record("clip_u_max", mods["clipper"].Clipper(param="u", maximum=-1.5).forward(fl(mixed)))
    mv = mods["apply_mask"].MaskVariable
    record("mask_param_value", mv(mask_param="lsm", mask_value=0).forward(fl(mixed)))
    record("mask_param_thr_keep", mv(mask_param="lsm", threshold=0.5, threshold_operator="<=", return_mask=True, param=["t", "q"], rename="land").forward(fl(mixed)))
    record("mask_param_ne", mv(mask_param="z", threshold=5e4, threshold_operator="gt", param="u").forward(fl(mixed)))
    # float64 inputs keep float64
    mixed64 = [(p, lev, val.astype(np.float64)) for p, lev, val in mixed]
    record("uv_to_ddff_f64", uv.forward(fl(mixed64)))
    record("q_to_r_all_f64", qr.forward(fl(mixed64)))
    np.savez_compressed(GOLDEN / "filters.npz", order=json.dumps(order), **out)
    print("filters.npz:", {k: v.shape for k, v in out.items()})


def more_filter_cases(mods, syn, ekd):
    """SURVEY §8(f) rank 1 — rescale, lnsp_to_sp, impute_nans, remove_nans, cos_sin_*, dewpoint,
    sum — run through the reference's own classes (values of the dewpoint pair come from
    oracle/pointwise.py via the earthkit.meteo stub; pinned by test_dewpoint.py:23-27)."""
    rng = np.random.default_rng(23)
    lat = np.linspace(50, -50, 21)
    lon = np.linspace(0, 340, 18)
    n = lat.size * lon.size
    LAT, LON = (a.reshape(-1) for a in np.meshgrid(lat, lon, indexing="ij"))

    def fl(specs):
        # fresh arrays per call: the reference's DewPoint writes 1e-4 into the r == 0 points of the
        # array it is handed (dewpoint.py:63-64), which must not leak into the next case
        return _fieldlist(ekd, [(p, lev, v.copy()) for p, lev, v in specs], LAT, LON)

    out, order = {}, {}

    def record(name, result):
        order[name] = [[f.metadata("param"), None if f.metadata("levelist") is None else int(f.metadata("levelist")), str(f.to_numpy().dtype)] for f in result]
        out[name] = np.stack([f.to_numpy(flatten=True).astype(np.float64) for f in result])

    def nanspots(a, k):
        a = a.copy()
        a[rng.choice(a.size, k, replace=False)] = np.nan
        return a

    t = {lev: rng.normal(270, 20, n).astype(np.float32) for lev in (500, 850)}
    r = {lev: rng.uniform(0, 110, n).astype(np.float32) for lev in (500, 850)}
    r[850][:3] = [0.0, 100.0, np.nan]
    t[850][:6] = [280.0, 280.0, 280.0, np.nan, 273.16, 32.19]
    lnsp = rng.normal(11.5, 0.1, n).astype(np.float32)
    lnsp[:4] = [np.nan, np.inf, -np.inf, 0.0]
    mwd = rng.uniform(0, 360, n).astype(np.float32)
    mwd[:5] = [0.0, 360.0, 180.0, 90.0, np.nan]
    rad = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
    rad[:4] = [0.0, np.float32(np.pi), -np.float32(np.pi), np.nan]
    sst = nanspots(rng.normal(290, 5, n).astype(np.float32), 40)
    lsp, cp, sf = (np.abs(rng.normal(0, 1e-3, n)).astype(np.float32) for _ in range(3))
    cp = nanspots(cp, 3)
    mixed = [("t", 850, t[850]), ("r", 850, r[850]), ("lnsp", 1, lnsp), ("mwd", 0, mwd), ("rad", 0, rad), ("sst", 0, sst), ("r", 500, r[500]),
             ("lsp", 0, lsp), ("t", 500, t[500]), ("cp", 0, cp), ("sf", 0, sf)]  # fmt: skip
    out["in_values"] = np.stack([m[2] for m in mixed])
    order["in"] = [[m[0], m[1]] for m in mixed]
    out["lat"], out["lon"] = LAT, LON

    rs = mods["rescale"].Rescale(param="t", scale=1.8, offset=-459.67)
    fwd = rs.forward(fl(mixed))
    record("rescale_fwd", fwd)
    record("rescale_bwd", rs.backward(fwd))
    ls = mods["lnsp_to_sp"].LnspToSp()
    sp = ls.forward(fl(mixed))
    record("lnsp_to_sp", sp)
    record("sp_to_lnsp", ls.backward(sp))
    record("impute_sst", mods["impute_nans"].ImputeNaNs(param=["sst", "cp"], value=-1.5).forward(fl(mixed)))
    cs = mods["cos_sin_from_rad"].CosSinFromRad(param="rad")
    c = cs.forward(fl(mixed))
    record("cos_sin_from_rad", c)
    record("rad_from_cos_sin", cs.backward(c))
    cw = mods["cos_sin_mean_wave_direction"].CosSinWaveDirection()
    c = cw.forward(fl(mixed))
    record("cos_sin_mwd", c)
    record("mwd_from_cos_sin", cw.backward(c))
    dp = mods["dewpoint"].DewPoint()
    d = dp.forward(fl(mixed))
    record("r_to_d_all", d)
    record("r_to_d_none", mods["dewpoint"].DewPoint(return_inputs="none").forward(fl(mixed)))
    only_dt = [f for f in d if f.metadata("param") in ("d", "t")]
    record("d_to_r_all", dp.backward(ekd.SimpleFieldList(only_dt)))
    record("sum_tp", mods["sum"].Sum(params=["lsp", "cp", "sf"], output="tp").forward(fl(mixed)))
    rn = mods["remove_nans"].RemoveNaNs(param="sst")
    res = rn.forward(fl(mixed))
    record("remove_nans_sst", res)
    out["remove_nans_lat"], out["remove_nans_lon"] = res[0].grid_points()
    # float64 fields keep float64
    mixed64 = [(p, lev, val.astype(np.float64)) for p, lev, val in mixed]
    record("rescale_fwd_f64", rs.forward(fl(mixed64)))
    record("cos_sin_mwd_f64", cw.forward(fl(mixed64)))
    record("mwd_from_cos_sin_f64", cw.backward(cw.forward(fl(mixed64))))
    record("r_to_d_all_f64", dp.forward(fl(mixed64)))
    record("sum_tp_f64", mods["sum"].Sum(params=["lsp", "cp", "sf"], output="tp").forward(fl(mixed64)))
    np.savez_compressed(GOLDEN / "filters_more.npz", order=json.dumps(order), **out)
    print("filters_more.npz:", {k: v.shape for k, v in out.items()})


# ---- reference_checks.npz / patch_data_request.json: the inputs of the live comparisons -------
# (tests/test_oracle_vs_reference.py, tests/test_oracle_tabular.py), so those comparisons run
# without the reference.  Written from the reference by main().  The stored files were written by
# `python oracle/make_golden.py --checks-from-oracle`: the oracle (spatial, superob) and this
# package (patch_data_request) standing in for the reference, whose sources were not at hand.
# The live tests asserted exactly these outputs equal to the reference's (spatial at 1308bd5,
# superob at 19e11ba, patch_data_request at f615e80), and the code that produces them has not
# changed since.


def spatial_random_cases(syn):
    """(seed, lam, glob) of the three random LAM / global pairs."""
    for seed in range(3):
        rng = np.random.default_rng(seed)
        lam = syn.rotated_lam(12 + seed, 15, 0.7, float(rng.uniform(-60, 70)), float(rng.uniform(0, 360)))
        yield seed, lam, syn.octahedral(12 + 4 * seed)


def superob_case(syn):
    """(grid [lat, lon] in -180..180, observations with NaN latitudes) of the superob check."""
    from oracle import tabular as ot

    lat, lon = syn.octahedral(6)
    grid = np.column_stack([lat, np.where(lon > 180, lon - 360, lon)])
    obs = ot.synthetic_observations(5000, seed=3)
    obs.loc[::501, "latitude"] = np.nan
    return grid, obs


SUPEROB_ARGS = dict(timeslot_length=3600, columns_to_take_nearest=["date"], columns_to_groupby=["reporttype"])

PATCH_DATA_REQUEST_CASES = [
    ("orog_to_z_fields", {}, [{"param": ["z", "t"], "levtype": "pl"}, {"param": ["orog", "t"], "levelist": [500]}, {"param": ["z", "t"], "levtype": "sfc"}, {"param": "z", "levtype": "pl"}, {"param": ["q"]}, {}]),
    ("lnsp_to_sp", {}, [{"param": ["sp", "t"]}, {"param": ["lnsp"]}, {"param": ["q"]}, {}]),
    ("cos_sin_from_rad", {"param": "x"}, [{"param": ["cos_x", "t"]}, {"param": ["sin_x", "cos_x"]}, {"param": ["q"]}, {}]),
    ("cos_sin_mean_wave_direction", {}, [{"param": ["cos_mwd", "t"]}, {"param": ["mwd"]}, {}]),
]  # fmt: skip


def frame_arrays(prefix: str, df, skip=()) -> dict:
    """A DataFrame as npz entries: the column order and one array per column not in `skip`."""
    out = {f"{prefix}__columns": np.array(json.dumps(list(df.columns)))}
    for c in df.columns:
        if c not in skip:
            out[f"{prefix}__{c}"] = df[c].to_numpy()
    return out


def stored_frame(z, prefix: str, base=None):
    """The DataFrame `frame_arrays` stored; `base` supplies the skipped columns and the index."""
    import pandas as pd

    cols = json.loads(str(z[f"{prefix}__columns"]))
    data = {c: z[f"{prefix}__{c}"] if f"{prefix}__{c}" in z else base[c].to_numpy() for c in cols}
    return pd.DataFrame(data, columns=cols, index=None if base is None else base.index)


def reference_checks(spatial, assign_nearest_grid, superob, patch_filters, syn):
    """spatial: module with the reference's spatial functions; assign_nearest_grid(df, grid, slot);
    superob(obs, grid) → SuperOb(grid=<grid>, **SUPEROB_ARGS).forward(obs);
    patch_filters(name, kwargs) → filter with the reference's patch_data_request."""
    import copy

    out = {}
    for seed, lam, glob in spatial_random_cases(syn):
        out[f"spatial{seed}_cutout"] = spatial.cutout_mask(*lam, *glob)
        out[f"spatial{seed}_cutout_50_900"] = spatial.cutout_mask(*lam, *glob, min_distance_km=50, max_distance_km=900)
        out[f"spatial{seed}_thinning"] = spatial.thinning_mask(*lam, *glob)
        out[f"spatial{seed}_global_on_lam"] = spatial.global_on_lam_mask(*lam, *glob)
        out[f"spatial{seed}_ngp_k3"] = spatial.nearest_grid_points(*glob, *lam, num_neighbours_to_return=3)
    grid, obs = superob_case(syn)
    # the binned frame is the observations (index and columns kept) plus three columns: only those are stored
    out.update(frame_arrays("binned", assign_nearest_grid(obs.dropna(subset=["latitude"]), grid, 3600), skip=obs.columns))
    out.update(frame_arrays("superob", superob(obs.copy(), grid)))  # compared without its index
    np.savez_compressed(GOLDEN / "reference_checks.npz", **out)
    requests = [
        {"filter": name, "kwargs": kw, "request": req, "result": patch_filters(name, kw).patch_data_request(copy.deepcopy(req))}
        for name, kw, reqs in PATCH_DATA_REQUEST_CASES
        for req in reqs
    ]
    (GOLDEN / "patch_data_request.json").write_text(json.dumps(requests, indent=1) + "\n")
    print("reference_checks.npz:", len(out), "arrays; patch_data_request.json:", len(requests), "requests")


def reference_checks_from_reference(mods, syn):
    import importlib

    support = importlib.import_module("anemoi.transform.filters.tabular.support.superob")
    flt = importlib.import_module("anemoi.transform.filters.tabular.superob")

    def superob(obs, grid):
        flt.define_grid = lambda name: grid  # the named-grid download is not the arithmetic
        return flt.SuperOb(grid="o6", **SUPEROB_ARGS).forward(obs)

    classes = {
        "orog_to_z_fields": lambda: mods["orog_to_z"].Orography(),
        "lnsp_to_sp": lambda: mods["lnsp_to_sp"].LnspToSp(),
        "cos_sin_from_rad": lambda param: mods["cos_sin_from_rad"].CosSinFromRad(param=param),
        "cos_sin_mean_wave_direction": lambda: mods["cos_sin_mean_wave_direction"].CosSinWaveDirection(),
    }
    reference_checks(mods["spatial"], support.assign_nearest_grid, superob, lambda name, kw: classes[name](**kw), syn)


def reference_checks_from_oracle(syn):
    from anemoi_transform_b200.filters import create_filter_by_name
    from oracle import spatial as osp
    from oracle import tabular as ot

    def superob(obs, grid):
        return ot.superob(obs, grid, SUPEROB_ARGS["timeslot_length"], take_nearest=SUPEROB_ARGS["columns_to_take_nearest"], groupby=SUPEROB_ARGS["columns_to_groupby"])

    reference_checks(osp, ot.assign_nearest_grid, superob, lambda name, kw: create_filter_by_name(name, **kw), syn)


def main():
    import tempfile

    from anemoi_transform_b200 import synthetic as syn

    GOLDEN.mkdir(parents=True, exist_ok=True)
    if "--checks-from-oracle" in sys.argv:
        reference_checks_from_oracle(syn)
        return
    mods = reference_import.load()
    import earthkit.data as ekd  # the stub

    spatial_cases(mods["spatial"], syn)
    with tempfile.TemporaryDirectory() as tmp:
        regrid_cases(mods, syn, ekd, Path(tmp))
    filter_cases(mods, syn, ekd)
    more_filter_cases(mods, syn, ekd)
    reference_checks_from_reference(mods, syn)


if __name__ == "__main__":
    main()
