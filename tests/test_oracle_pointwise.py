"""The pointwise oracle against the reference's own golden vectors (the pin for the
earthkit-meteo formulas, which are not vendored in the reference)."""

import numpy as np

from oracle import pointwise as pw

# reference tests/field_filters/test_uv_to_ddff.py:24-42
U = {500: [[-3.26786804, -2.90458679], [-4.28153992, -10.75224304], [-6.29130554, -4.17704773]], 850: [[-6.72481718, -0.34174164], [-7.14725727, -2.02047454], [-4.93597360, -0.00018431]]}
V = {500: [[6.51824951, 4.7321167], [1.16961670, 1.73797607], [-2.93096924, 3.2399292]], 850: [[5.4374572, -0.00679462], [2.23226754, 6.78457592], [-1.79188286, -0.0093771]]}
WS = {500: [[7.29153881, 5.55243666], [4.43842171, 10.89179926], [6.94054076, 5.28629066]], 850: [[8.64806955, 0.34180918], [7.48774364, 7.07903862], [5.25115983, 0.00937891]]}
WDIR = {500: [[153.37349864, 148.45827835], [105.27908047, 99.18178736], [65.02031089, 127.79896253]], 850: [[128.95781905, 88.86097611], [107.34489249, 163.41625261], [70.04782648, 1.12603196]]}
# reference tests/field_filters/test_pressure_level_humidity.py:27-40
T = {850: [[293.32301331, 284.21559143], [260.53981018, 291.18824768], [279.88941956, 248.87574768]], 1000: [[291.22831726, 289.85136414], [271.29277039, 301.67362976], [287.53691101, 250.15409851]]}
Q = {850: [[0.00657578, 0.00769957], [0.00147607, 0.01088967], [0.00505508, 0.00044559]], 1000: [[0.01075057, 0.01080445], [0.00226020, 0.01525551], [0.00914679, 0.00047560]]}
R = {850: [[37.91091442, 79.51638317], [95.61794567, 71.53396130], [70.03982067, 89.69021130]], 1000: [[82.88058853, 90.86496353], [68.26144791, 62.40207291], [89.31613541, 99.25949478]]}


def test_wind_golden_vectors():
    for lev in (500, 850):
        ws, wdir = pw.xy_to_polar(np.array(U[lev]), np.array(V[lev]))
        assert np.allclose(ws, WS[lev]) and np.allclose(wdir, WDIR[lev])
        u, v = pw.polar_to_xy(np.array(WS[lev]), np.array(WDIR[lev]))
        assert np.allclose(u, U[lev]) and np.allclose(v, V[lev])


def test_humidity_golden_vectors():
    for lev in (850, 1000):
        r = pw.relative_humidity_from_specific_humidity(np.array(T[lev]), np.array(Q[lev]), 100.0 * lev)
        assert np.allclose(r, R[lev])
        q = pw.specific_humidity_from_relative_humidity(np.array(T[lev]), np.array(R[lev]), 100.0 * lev)
        assert np.allclose(q, Q[lev])


def test_float32_stays_float32_and_special_values():
    u = np.array([0.0, -0.0, 0.0, np.inf, np.nan, 3.0], dtype=np.float32)
    v = np.array([0.0, 0.0, -0.0, np.nan, 1.0, -4.0], dtype=np.float32)
    ws, wdir = pw.xy_to_polar(u, v)
    assert ws.dtype == np.float32 and wdir.dtype == np.float32
    assert wdir[0] == 270.0  # atan2(0, 0) = 0
    assert wdir[1] == 270.0 - 180.0  # atan2(0, -0) = pi
    assert ws[3] == np.inf and np.isnan(ws[4]) and ws[5] == 5.0
    t = np.array([250.16, 273.16, 260.0, np.nan], dtype=np.float32)
    q = np.full(4, 1e-3, dtype=np.float32)
    r = pw.relative_humidity_from_specific_humidity(t, q, 85000.0)
    assert r.dtype == np.float32 and np.isnan(r[3]) and np.all(r[:3] > 0)
    # clip passes NaN through; either bound may be absent
    x = np.array([np.nan, 1.0, 5.0], dtype=np.float32)
    assert np.array_equal(pw.clip(x, 2.0, 4.0), np.array([np.nan, 2.0, 4.0], dtype=np.float32), equal_nan=True)
    assert np.array_equal(pw.clip(x, None, 4.0), np.array([np.nan, 1.0, 4.0], dtype=np.float32), equal_nan=True)


def test_filter_level_golden_is_the_oracle(golden_filters):
    """tests/golden/filters.npz was produced by the reference's filters; its wind / humidity
    values must be what the oracle formulas give on the stored inputs."""
    g = golden_filters
    order = {tuple(o): i for i, o in enumerate(g["order"]["in"])}
    x = g["in_values"].astype(np.float32)
    u, v = x[order[("u", 850)]], x[order[("v", 850)]]
    ws, wdir = pw.xy_to_polar(u, v)
    names = [tuple(o[:2]) for o in g["order"]["uv_to_ddff"]]
    assert np.array_equal(g["uv_to_ddff"][names.index(("ws", 850))], ws.astype(np.float64), equal_nan=True)
    assert np.array_equal(g["uv_to_ddff"][names.index(("wdir", 850))], wdir.astype(np.float64), equal_nan=True)
    r = pw.relative_humidity_from_specific_humidity(x[order[("t", 500)]], x[order[("q", 500)]], 50000.0)
    names = [tuple(o[:2]) for o in g["order"]["q_to_r_all"]]
    assert np.array_equal(g["q_to_r_all"][names.index(("r", 500))], r.astype(np.float64), equal_nan=True)


# reference tests/field_filters/test_dewpoint.py:23-27
R_DEW = [[78.13834333, 71.28598853], [99.17328572, 44.52144788], [56.49667261, 86.10495618]]
T_DEW = [[298.42488098, 297.55574036], [278.68269348, 293.99324036], [300.61042786, 300.40144348]]
D_DEW = [[294.34245300, 292.02214050], [278.56315613, 281.47135925], [291.19792175, 297.87370300]]


def test_dewpoint_golden_vectors():
    td = pw.dewpoint_from_relative_humidity(np.array(T_DEW), np.array(R_DEW))
    assert np.allclose(td, D_DEW)
    r = pw.relative_humidity_from_dewpoint(np.array(T_DEW), np.array(D_DEW))
    assert np.allclose(r, R_DEW)
    t32 = np.array(T_DEW, dtype=np.float32)
    assert pw.dewpoint_from_relative_humidity(t32, np.array(R_DEW, dtype=np.float32)).dtype == np.float32


def test_more_filters_golden_is_numpy_and_the_oracle(golden_filters_more):
    """tests/golden/filters_more.npz (outputs of the reference's own filter classes) against
    the plain numpy statements of reference rescale.py:25-29, lnsp_to_sp.py:48,66,
    impute_nans.py:52-54, cos_sin_from_rad.py:78-79,100, cos_sin_mean_wave_direction.py:71-74,96-98,
    sum.py:109-115, remove_nans.py:103-117, and the oracle's dewpoint formulas."""
    g = golden_filters_more
    x = {tuple(o): v.astype(np.float32) for o, v in zip(g["order"]["in"], g["in_values"])}

    def got(name, param, lev):
        names = [tuple(o[:2]) for o in g["order"][name]]
        return g[name][names.index((param, lev))]

    def same(a, b):
        return np.array_equal(np.asarray(a, dtype=np.float64), b, equal_nan=True)

    t = x[("t", 850)]
    assert same(t * 1.8 + -459.67, got("rescale_fwd", "t", 850))
    assert same(((t * 1.8 + -459.67) - -459.67) / 1.8, got("rescale_bwd", "t", 850))
    with np.errstate(all="ignore"):
        assert same(np.exp(x[("lnsp", 1)]), got("lnsp_to_sp", "sp", None))
        assert same(np.log(np.exp(x[("lnsp", 1)])), got("sp_to_lnsp", "lnsp", None))
    sst = x[("sst", 0)].copy()
    sst[np.isnan(sst)] = -1.5
    assert same(sst, got("impute_sst", "sst", 0))
    rad, mwd = x[("rad", 0)], x[("mwd", 0)]
    assert same(np.cos(rad), got("cos_sin_from_rad", "cos_rad", 0)) and same(np.sin(rad), got("cos_sin_from_rad", "sin_rad", 0))
    assert same(np.arctan2(np.sin(rad), np.cos(rad)), got("rad_from_cos_sin", "rad", 0))
    assert same(np.cos(np.deg2rad(mwd)), got("cos_sin_mwd", "cos_mwd", 0))
    back = np.rad2deg(np.arctan2(np.sin(np.deg2rad(mwd)), np.cos(np.deg2rad(mwd))))
    back = np.where(back >= 360, back - 360, back)
    back = np.where(back < 0, back + 360, back)
    assert same(back, got("mwd_from_cos_sin", "mwd", 0))
    r = x[("r", 850)].copy()
    r[r == 0] = 1.0e-4
    assert same(pw.dewpoint_from_relative_humidity(t, r), got("r_to_d_all", "d", 850))
    assert same(pw.relative_humidity_from_dewpoint(t, pw.dewpoint_from_relative_humidity(t, r)), got("d_to_r_all", "r", 850))
    s = x[("lsp", 0)].copy()
    s += x[("cp", 0)]
    s += x[("sf", 0)]
    assert same(s, got("sum_tp", "tp", 0))
    keep = ~np.isnan(x[("sst", 0)])
    assert same(x[("t", 500)][keep], got("remove_nans_sst", "t", 500)) and np.array_equal(g["remove_nans_lat"], g["lat"][keep])


def test_es_table_restatement_meets_its_stated_bound():
    """epilogue.cuh:200-203 / DESIGN §3.3: the float32 cubics of es(T), Horner evaluation
    included, are within 2e-7 relative of the float64 formula.  Checked on the numpy
    restatement of fit_es_table and es_from_table at every interval's fit points, ends and
    midpoint, the float32 neighbours of both thresholds, and 200 000 random temperatures."""
    from oracle import es_table as et

    table = et.fit_es_table()
    assert table.shape == (400, 4) and table.dtype == np.float32
    assert et.T_TABLE + np.float32(23.0) == et.T_WATER  # node 246 is the water threshold exactly
    rng = np.random.default_rng(0)
    t = np.concatenate([et.table_sample_points(), rng.uniform(150.16, 350.15, 200_000).astype(np.float32)])
    t = t[et.covers(t)]
    rel = np.abs(et.es_from_table(t, table).astype(np.float64) / et.es_mixed_f64(t) - 1.0)
    assert rel.max() < 2e-7, (rel.max(), t[np.argmax(rel)])
    # and the bound is not vacuous: a coefficient off by one part in 1e-6 breaks it
    bad = table.copy()
    bad[10, 0] *= np.float32(1.000001)
    t10 = t[(t >= np.float32(155.16)) & (t < np.float32(155.66))]
    assert np.abs(et.es_from_table(t10, bad).astype(np.float64) / et.es_mixed_f64(t10) - 1.0).max() > 2e-7
