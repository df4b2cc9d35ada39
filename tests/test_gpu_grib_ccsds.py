"""CCSDS-packed GRIB2 fields (template 5.42) decoded on the device (ccsds_rsi_scan_kernel,
ccsds_decode_kernel, then grib_unpack_kernel) against the numpy oracle, against simple
packing of the same X, and through every regrid route.  Bit for bit throughout."""

import struct

import numpy as np
import pytest
from conftest import assert_same_values
from grib_ccsds_fields import CcsdsGribField as GribMessageField
from scipy.sparse import csr_array

from anemoi_transform_b200 import synthetic as syn
from oracle import grib as ogrib
from oracle import grib_ccsds as ogc

pytestmark = pytest.mark.gpu

WIDTHS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 24, 25, 31, 32]
BLOCKS = [8, 16, 32, 64]
RSIS = [1, 2, 3, 128, 4096]
FLAGS = [14, 8, 0, 46, 32, 40]


def _values(rng, k, n):
    kind = k % 3
    if kind == 0:  # smooth: mostly split-sample and zero blocks after preprocessing
        return np.cumsum(rng.normal(0.0, 0.05, n)) + 280.0
    if kind == 1:  # noise: uncompressed blocks
        return rng.normal(280.0, 15.0, n)
    v = np.full(n, 280.0)  # steps between the range ends: X pinned at 0 and at xmax, long zero runs
    v[n // 3 : 2 * n // 3] = 300.0
    v[rng.uniform(size=n) > 0.99] = 290.0
    return v


def _ccsds_messages(n_fields, n_points, seed, bitmaps=False):
    """(CCSDS message, simple message of the same X) pairs over the whole parameter grid: field k
    takes width k mod 13, block size k mod 4 and RSI k mod 5 (coprime: 260 fields see every
    combination), flags and end padding alternating."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n_fields):
        nb, J, rsi, fl = WIDTHS[k % 13], BLOCKS[k % 4], RSIS[k % 5], FLAGS[k % 6]
        bm = None
        count = n_points
        if bitmaps and k % 2:
            bm = rng.uniform(size=n_points) > (0.1 if k % 4 == 1 else 0.8)
            bm[0] = True
            count = int(bm.sum())
        v = _values(rng, k, count)
        if count > 1:
            v[0], v[-1] = v.min() - 1.0, v.max() + 1.0  # a non-constant field: n bits are used
        pad = "rsi" if k % 7 == 3 else "block"
        c = ogc.encode_grib2(v, nb, k % 2, bm, block_size=J, rsi=rsi, flags=fl, pad=pad)
        s = ogrib.encode_grib2(v, nb, k % 2, bm)
        out.append((c, s))
    return out


def _fields(messages, n_points, lat=None, lon=None, param="t"):
    return [GribMessageField(m, n_points, dict(param=param, levelist=850, step=k), latitudes=lat, longitudes=lon) for k, m in enumerate(messages)]


def _decode_both(packed, n):
    from anemoi_transform_b200 import grib

    b64 = grib.upload(packed).data[:, :n].cpu().numpy().T
    b32 = grib.upload(packed, np.float32).data[:, :n].cpu().numpy().T
    return b64, b32


@pytest.mark.parametrize("n_points,n_fields", [(1, 26), (7, 260), (255, 260), (256, 260), (1001, 260), (65160, 52)])
def test_device_decode_equals_the_oracle(cuda, n_points, n_fields):
    from anemoi_transform_b200 import grib

    pairs = _ccsds_messages(n_fields, n_points, seed=n_points)
    msgs = [c for c, _ in pairs]
    want = np.stack([ogc.decode(m, n_points=n_points) for m in msgs])
    packed = grib.packed_of(_fields(msgs, n_points))
    assert packed is not None and all(i.packing == 1 or i.bits_per_value == 0 for i in packed.infos)
    got64, got32 = _decode_both(packed, n_fields)
    assert_same_values(got64, want, "CCSDS float64 decode")
    assert_same_values(got32, want.astype(np.float32), "CCSDS float32 decode")


@pytest.mark.parametrize("n_points", [5, 256, 1001, 40320])
def test_device_decode_with_bitmaps(cuda, n_points):
    from anemoi_transform_b200 import grib

    pairs = _ccsds_messages(130, n_points, seed=7 * n_points, bitmaps=True)
    msgs = [c for c, _ in pairs]
    want = np.stack([ogc.decode(m, n_points=n_points) for m in msgs])
    assert np.isnan(want).any()
    got64, got32 = _decode_both(grib.packed_of(_fields(msgs, n_points)), len(msgs))
    assert_same_values(got64, want, "CCSDS bitmap float64")
    assert_same_values(got32, want.astype(np.float32), "CCSDS bitmap float32")


def test_ccsds_batch_equals_the_simple_batch_of_the_same_x(cuda):
    """Chunks that mix both packings: the CCSDS columns equal the simple-packing columns of the
    same X bit for bit (the unpack reads the decoded words through the same formula)."""
    from anemoi_transform_b200 import grib

    n_points = 40320
    pairs = _ccsds_messages(78, n_points, seed=5, bitmaps=True)
    mixed = [c if k % 3 else s for k, (c, s) in enumerate(pairs)]
    simple = [s for _, s in pairs]
    a64, a32 = _decode_both(grib.packed_of(_fields(mixed, n_points)), len(mixed))
    b64, b32 = _decode_both(grib.packed_of(_fields(simple, n_points)), len(simple))
    assert_same_values(a64, b64, "mixed vs simple float64")
    assert_same_values(a32, b32, "mixed vs simple float32")


def test_full_o1280_message(cuda):
    """6 599 680 points at ECMWF's defaults (J = 32, RSI = 128, flags 14), and a 24-bit field with
    PAD_RSI: 1 612 and 51 563 RSIs per field.  The oracle's CCSDS decode equals the simple decode of
    the same X (tests/test_oracle_ccsds.py); here the simple message is the reference, which
    numpy decodes in one pass."""
    from anemoi_transform_b200 import grib

    lat, _ = syn.octahedral(1280)
    n = lat.size
    assert n == 6_599_680
    rng = np.random.default_rng(1280)
    v = 250.0 + 40.0 * np.cos(np.deg2rad(lat)) + np.cumsum(rng.normal(0.0, 0.002, n))
    msgs = [
        (ogc.encode_grib2(v, 16, 0), ogrib.encode_grib2(v, 16, 0)),
        (ogc.encode_grib2(v, 24, 1, block_size=16, rsi=8, flags=8 | 32), ogrib.encode_grib2(v, 24, 1)),
    ]
    packed = grib.packed_of(_fields([c for c, _ in msgs], n))
    assert packed.packed_bytes < sum(len(s) for _, s in msgs)
    got64, got32 = _decode_both(packed, 2)
    want = np.stack([ogc.decode(s) for _, s in msgs])
    assert_same_values(got64, want, "O1280 float64")
    assert_same_values(got32, want.astype(np.float32), "O1280 float32")


@pytest.fixture(scope="module")
def small_matrix(tmp_path_factory):
    t_lat, t_lon = syn.octahedral(48)
    d, i, p, shape = syn.bilinear_matrix(2.0, t_lat, t_lon)
    s_lat, s_lon = syn.regular_latlon(2.0)
    path = str(tmp_path_factory.mktemp("ccsds") / "m.npz")
    syn.save_regrid_npz(path, d, i, p, shape, s_lat, s_lon, t_lat, t_lon)
    return path, csr_array((d, i, p), shape=shape), s_lat, s_lon


def test_regrid_routes_on_a_mixed_fieldlist(cuda, small_matrix):
    """Simple, CCSDS (one with a bitmap) and numpy fields in one FieldList: streamed, resident
    (regrid | rescale), fused (float32 decode, regrid | clip) — outputs in input order, equal to
    scipy on the oracle's host decode, nothing decoded on the host."""
    from anemoi_transform_b200 import ekd, grib
    from anemoi_transform_b200.filters import create_filter_by_name as F

    path, m, s_lat, s_lon = small_matrix
    n_src = s_lat.size
    pairs = _ccsds_messages(24, n_src, seed=17)
    rng = np.random.default_rng(17)
    bm = rng.uniform(size=n_src) > 0.2
    with_bitmap = ogc.encode_grib2(rng.normal(285.0, 5.0, int(bm.sum())), 16, 0, bm)
    msgs = [c if k % 2 else s for k, (c, s) in enumerate(pairs)] + [with_bitmap]
    fields = _fields(msgs, n_src, s_lat, s_lon)
    plain = ekd.ArrayField(rng.normal(0.0, 1.0, n_src), dict(param="z", step=0), latitudes=s_lat, longitudes=s_lon)
    mixed = fields[:10] + [plain] + fields[10:]
    host = [ogc.decode(f.message(), n_points=n_src) if isinstance(f, GribMessageField) else f.to_numpy() for f in mixed]

    out = F("regrid", matrix=path).forward(ekd.SimpleFieldList(mixed))
    assert [f.metadata("param") for f in out] == [f.metadata("param") for f in mixed]
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), m @ host[k], f"streamed field {k}")
    assert np.isnan(out[-1].to_numpy()).any()

    pipe = F("regrid", matrix=path) | F("rescale", param="t", scale=2.0, offset=1.0)
    out = pipe.forward(ekd.SimpleFieldList(fields))
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), (m @ ogc.decode(msgs[k], n_points=n_src)) * 2.0 + 1.0, f"resident field {k}")

    grib.set_decode_dtype(np.float32)
    try:
        pipe = F("regrid", matrix=path) | F("clip_fields", param="t", minimum=250.0, maximum=290.0)
        out = pipe.forward(ekd.SimpleFieldList(fields[:12]))
        for k, f in enumerate(out):
            x32 = ogc.decode(msgs[k], n_points=n_src).astype(np.float32)
            assert_same_values(f.to_numpy(), np.clip(m @ x32, np.float32(250.0), np.float32(290.0)), f"fused field {k}")
    finally:
        grib.set_decode_dtype(None)
    assert sum(f.decodes for f in fields) == 0


def _forward(monkeypatch, devices, filt, fields):
    if devices is None:
        monkeypatch.delenv("AT_B200_DEVICES", raising=False)
    else:
        monkeypatch.setenv("AT_B200_DEVICES", devices)
    return [f.to_numpy() for f in filt.forward(fields)]


@pytest.mark.parametrize("devices", ["twice", "all"])
def test_regrid_on_several_engines(cuda, monkeypatch, devices, tmp_path):
    """at_hostio_group_regrid_grib: two engines on one GPU, or every GPU (skipped below two)."""
    from anemoi_transform_b200.filters import create_filter_by_name as F

    if devices == "all":
        if cuda.cuda.device_count() < 2:
            pytest.skip(f"needs 2 GPUs, {cuda.cuda.device_count()} visible")
        spec = ",".join(str(d) for d in range(cuda.cuda.device_count()))
    else:
        d = cuda.cuda.current_device()
        spec = f"{d},{d}"
    s_lat, s_lon = syn.regular_latlon(0.25)
    t_lat, t_lon = syn.octahedral(32)
    d_, i_, p_, shape = syn.bilinear_matrix(0.25, t_lat, t_lon)
    d_ = d_.astype(np.float64)
    path = str(tmp_path / "m64.npz")
    syn.save_regrid_npz(path, d_, i_, p_, shape, s_lat, s_lon, t_lat, t_lon)
    m = csr_array((d_, i_, p_), shape=shape)
    rng = np.random.default_rng(9)
    msgs = []
    for k in range(24):
        v = np.cumsum(rng.normal(0.0, 0.05, s_lat.size)) + 280.0
        msgs.append(ogc.encode_grib2(v, 16, 1) if k % 3 else ogrib.encode_grib2(v, 16, 1))
    fields = _fields(msgs, s_lat.size, s_lat, s_lon)
    regrid = F("regrid", matrix=path)
    single = _forward(monkeypatch, None, regrid, fields)
    group = _forward(monkeypatch, spec, regrid, fields)
    assert all(f.decodes == 0 for f in fields)
    for k, msg in enumerate(msgs):
        want = m @ ogc.decode(msg, n_points=s_lat.size)
        assert_same_values(single[k], want, f"single engine, field {k}")
        assert_same_values(group[k], want, f"{spec}, field {k}")


# ------------------------------------------------------------------ malformed streams ------
def _with_section7(msg: bytes, data: bytes) -> bytes:
    """The message with section 7 replaced (and the total length fixed)."""
    info = ogc.scan(msg)
    start = info["data_offset"] - 5
    end = info["data_offset"] + info["data_length"]
    body = msg[16:start] + struct.pack(">IB", 5 + len(data), 7) + data + msg[end:]
    return msg[:8] + struct.pack(">Q", 16 + len(body)) + body


def test_malformed_streams_are_refused_and_the_engine_carries_on(cuda, small_matrix):
    from anemoi_transform_b200 import ekd, grib
    from anemoi_transform_b200.filters import create_filter_by_name as F

    path, m, s_lat, s_lon = small_matrix
    n_src = s_lat.size
    rng = np.random.default_rng(3)
    good = [ogc.encode_grib2(np.cumsum(rng.normal(0.0, 0.1, n_src)) + 280.0, 16, 0, rsi=4) for _ in range(6)]
    stream = good[3][ogc.scan(good[3])["data_offset"] :][: ogc.scan(good[3])["data_length"]]
    truncated = _with_section7(good[3], stream[: len(stream) // 2])
    # ID 0000, selector 0, then FS(195): a zero run of 195 blocks in an RSI of 4
    long_run = _with_section7(good[3], bytes(25) + b"\x80" + stream[26:])
    # 3 bits per value: option ID 110 is split-sample with k = 5 >= n
    tiny = ogc.encode_grib2(np.arange(float(n_src)) % 7, 3, 0, flags=0)
    s3 = tiny[ogc.scan(tiny)["data_offset"] :][: ogc.scan(tiny)["data_length"]]
    bad_option = _with_section7(tiny, b"\xc0" + s3[1:])
    for bad, what in ((truncated, "ends before"), (long_run, "zero-block run"), (bad_option, "k >= bits")):
        msgs = good[:3] + [bad] + good[4:]
        if bad is bad_option:
            msgs = [tiny, tiny, tiny, bad]
        fields = _fields(msgs, n_src, s_lat, s_lon)
        packed = grib.packed_of(fields)
        assert packed is not None  # the scan accepts it: only decoding the stream can tell
        with pytest.raises(ValueError, match=f"message 3: .*{what}"):
            grib.upload(packed)
        with pytest.raises(ValueError, match=f"message 3: .*{what}"):
            F("regrid", matrix=path).forward(ekd.SimpleFieldList(fields))
        # the engine serves the next call normally
        ok = F("regrid", matrix=path).forward(ekd.SimpleFieldList(_fields(good, n_src, s_lat, s_lon)))
        for k, f in enumerate(ok):
            assert_same_values(f.to_numpy(), m @ ogc.decode(good[k], n_points=n_src), f"after a refusal, field {k}")
        got = grib.upload(grib.packed_of(_fields(good, n_src))).data[:, :6].cpu().numpy().T
        assert_same_values(got, np.stack([ogc.decode(g) for g in good]), "upload after a refusal")
