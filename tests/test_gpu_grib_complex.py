"""Complex-packed GRIB2 fields (templates 5.2 and 5.3) decoded on the device (complex_groups_kernel,
complex_tile_sums_kernel, complex_carry_kernel, complex_values_kernel, then grib_unpack_kernel)
against the numpy oracle, against simple packing of the same X, and through every regrid
route.  Bit for bit throughout."""

import struct

import numpy as np
import pytest
from conftest import assert_same_values
from grib_complex_fields import ComplexGribField as GribMessageField
from scipy.sparse import csr_array

from anemoi_transform_b200 import synthetic as syn
from oracle import grib as ogrib
from oracle import grib_ccsds as ogc
from oracle import grib_complex as ogx

pytestmark = pytest.mark.gpu

WIDTHS = [1, 2, 3, 7, 8, 9, 12, 15, 16, 17, 24, 25]
ORDERS = [2, 0, 1]
GROUPS = [16, 1, 7, 1000, None]  # None: variable lengths 3 + 4k


def _values(rng, k, n):
    if k % 2 == 0:  # smooth: narrow second differences
        return 280.0 + np.cumsum(np.cumsum(rng.normal(0.0, 0.01, n)))
    return rng.normal(280.0, 15.0, n)


def _lengths(rng, n, size):
    if size is not None:
        return ogx.group_lengths(n, size)
    out = []
    while sum(out) < n:
        out.append(3 + 4 * int(rng.integers(0, 6)))
    out[-1] -= sum(out) - n
    if out[-1] <= 0:
        out.pop()
        out[-1] += n - sum(out)
    return out


def _complex_messages(n_fields, n_points, seed, bitmaps=False):
    """(complex message, simple message of the same X) pairs: field k takes width k mod 12,
    order k mod 3 and group layout k mod 5 (coprime: 180 fields see every combination)."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n_fields):
        nb, order, size = WIDTHS[k % 12], ORDERS[k % 3], GROUPS[k % 5]
        bm = None
        count = n_points
        if bitmaps and k % 2:
            bm = rng.uniform(size=n_points) > (0.1 if k % 4 == 1 else 0.8)
            bm[0] = True
            count = int(bm.sum())
        v = _values(rng, k, count)
        if count > 1:
            v[0], v[-1] = v.min() - 1.0, v.max() + 1.0
        s = ogrib.encode_grib2(v, nb, k % 2, bm)
        c = ogx.from_simple(s, order=order, lengths=_lengths(rng, count, size), increment=4 if size is None else 1)
        out.append((c, s))
    return out


def _fields(messages, n_points, lat=None, lon=None, param="t"):
    return [GribMessageField(m, n_points, dict(param=param, levelist=850, step=k), latitudes=lat, longitudes=lon) for k, m in enumerate(messages)]


def _decode_both(packed, n):
    from anemoi_transform_b200 import grib

    b64 = grib.upload(packed).data[:, :n].cpu().numpy().T
    b32 = grib.upload(packed, np.float32).data[:, :n].cpu().numpy().T
    return b64, b32


@pytest.mark.parametrize("n_points,n_fields", [(1, 15), (2, 60), (3, 60), (7, 180), (255, 180), (256, 180), (1001, 180), (65160, 45)])
def test_device_decode_equals_the_oracle(cuda, n_points, n_fields):
    from anemoi_transform_b200 import grib

    pairs = _complex_messages(n_fields, n_points, seed=n_points)
    msgs = [c for c, _ in pairs]
    want = np.stack([ogx.decode(m, n_points=n_points) for m in msgs])
    packed = grib.packed_of(_fields(msgs, n_points))
    assert packed is not None and all(i.packing == 2 for i in packed.infos)
    got64, got32 = _decode_both(packed, n_fields)
    assert_same_values(got64, want, "complex float64 decode")
    assert_same_values(got32, want.astype(np.float32), "complex float32 decode")


def test_chunks_of_many_fields(cuda):
    """More fields than one chunk holds: the upload splits them over several slots."""
    from anemoi_transform_b200 import grib

    n_points = 40320
    pairs = _complex_messages(600, n_points, seed=11)
    msgs = [c for c, _ in pairs]
    packed = grib.packed_of(_fields(msgs, n_points))
    got64, got32 = _decode_both(packed, len(msgs))
    want = np.stack([ogrib.decode(s) for _, s in pairs])
    assert_same_values(got64, want, "many fields float64")
    assert_same_values(got32, want.astype(np.float32), "many fields float32")


@pytest.mark.parametrize("n_points", [5, 256, 1001, 40320])
def test_device_decode_with_bitmaps(cuda, n_points):
    from anemoi_transform_b200 import grib

    pairs = _complex_messages(90, n_points, seed=7 * n_points, bitmaps=True)
    msgs = [c for c, _ in pairs]
    want = np.stack([ogx.decode(m, n_points=n_points) for m in msgs])
    assert np.isnan(want).any()
    got64, got32 = _decode_both(grib.packed_of(_fields(msgs, n_points)), len(msgs))
    assert_same_values(got64, want, "complex bitmap float64")
    assert_same_values(got32, want.astype(np.float32), "complex bitmap float32")


def test_complex_batch_equals_the_simple_batch_of_the_same_x(cuda):
    """Chunks that mix simple, CCSDS and complex packing: every column equals the simple-packing
    column of the same X bit for bit."""
    from anemoi_transform_b200 import grib

    n_points = 40320
    pairs = _complex_messages(78, n_points, seed=5, bitmaps=True)
    mixed = [(c if k % 3 == 1 else (ogc.from_simple(s) if k % 3 == 2 and ogrib.scan(s)["bits_per_value"] else s)) for k, (c, s) in enumerate(pairs)]
    complex_only = [c for c, _ in pairs]
    simple = [s for _, s in pairs]
    a64, a32 = _decode_both(grib.packed_of(_fields(mixed, n_points)), len(mixed))
    c64, c32 = _decode_both(grib.packed_of(_fields(complex_only, n_points)), len(mixed))
    b64, b32 = _decode_both(grib.packed_of(_fields(simple, n_points)), len(simple))
    assert_same_values(a64, b64, "mixed vs simple float64")
    assert_same_values(a32, b32, "mixed vs simple float32")
    assert_same_values(c64, b64, "complex vs simple float64")
    assert_same_values(c32, b32, "complex vs simple float32")


def test_full_o1280_message(cuda):
    """6 599 680 points as 5.3 order 2 (groups of 16) and as 5.2 with groups of one."""
    from anemoi_transform_b200 import grib

    lat, _ = syn.octahedral(1280)
    n = lat.size
    assert n == 6_599_680
    rng = np.random.default_rng(1280)
    v = 250.0 + 40.0 * np.cos(np.deg2rad(lat)) + np.cumsum(rng.normal(0.0, 0.002, n))
    s16, s24 = ogrib.encode_grib2(v, 16, 0), ogrib.encode_grib2(v, 24, 1)
    msgs = [(ogx.from_simple(s16, order=2), s16), (ogx.from_simple(s24, order=0, group_size=1), s24)]
    packed = grib.packed_of(_fields([c for c, _ in msgs], n))
    got64, got32 = _decode_both(packed, 2)
    want = np.stack([ogrib.decode(s) for _, s in msgs])
    assert_same_values(got64, want, "O1280 float64")
    assert_same_values(got32, want.astype(np.float32), "O1280 float32")


@pytest.fixture(scope="module")
def small_matrix(tmp_path_factory):
    t_lat, t_lon = syn.octahedral(48)
    d, i, p, shape = syn.bilinear_matrix(2.0, t_lat, t_lon)
    s_lat, s_lon = syn.regular_latlon(2.0)
    path = str(tmp_path_factory.mktemp("complex") / "m.npz")
    syn.save_regrid_npz(path, d, i, p, shape, s_lat, s_lon, t_lat, t_lon)
    return path, csr_array((d, i, p), shape=shape), s_lat, s_lon


def test_regrid_routes_on_a_mixed_fieldlist(cuda, small_matrix):
    """Simple, CCSDS, complex (one with a bitmap) and numpy fields in one FieldList: streamed,
    resident (regrid | rescale), fused (float32 decode, regrid | clip) — outputs in input order,
    equal to scipy on the oracle's host decode, nothing decoded on the host."""
    from anemoi_transform_b200 import ekd, grib
    from anemoi_transform_b200.filters import create_filter_by_name as F

    path, m, s_lat, s_lon = small_matrix
    n_src = s_lat.size
    pairs = _complex_messages(24, n_src, seed=17)
    rng = np.random.default_rng(17)
    bm = rng.uniform(size=n_src) > 0.2
    with_bitmap = ogx.encode_grib2(rng.normal(285.0, 5.0, int(bm.sum())), 16, 0, bm)
    msgs = [c if k % 3 == 0 else (s if k % 3 == 1 else ogc.from_simple(s)) for k, (c, s) in enumerate(pairs)] + [with_bitmap]
    assert {ogx.scan(x)["packing"] for x in msgs} == {0, 1, 2}
    fields = _fields(msgs, n_src, s_lat, s_lon)
    plain = ekd.ArrayField(rng.normal(0.0, 1.0, n_src), dict(param="z", step=0), latitudes=s_lat, longitudes=s_lon)
    mixed = fields[:10] + [plain] + fields[10:]
    host = [ogx.decode(f.message(), n_points=n_src) if isinstance(f, GribMessageField) else f.to_numpy() for f in mixed]

    out = F("regrid", matrix=path).forward(ekd.SimpleFieldList(mixed))
    assert [f.metadata("param") for f in out] == [f.metadata("param") for f in mixed]
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), m @ host[k], f"streamed field {k}")
    assert np.isnan(out[-1].to_numpy()).any()

    pipe = F("regrid", matrix=path) | F("rescale", param="t", scale=2.0, offset=1.0)
    out = pipe.forward(ekd.SimpleFieldList(fields))
    for k, f in enumerate(out):
        assert_same_values(f.to_numpy(), (m @ ogx.decode(msgs[k], n_points=n_src)) * 2.0 + 1.0, f"resident field {k}")

    grib.set_decode_dtype(np.float32)
    try:
        pipe = F("regrid", matrix=path) | F("clip_fields", param="t", minimum=250.0, maximum=290.0)
        out = pipe.forward(ekd.SimpleFieldList(fields[:12]))
        for k, f in enumerate(out):
            x32 = ogx.decode(msgs[k], n_points=n_src).astype(np.float32)
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
        msgs.append(ogx.encode_grib2(v, 16, 1, order=k % 3) if k % 4 else ogrib.encode_grib2(v, 16, 1))
    fields = _fields(msgs, s_lat.size, s_lat, s_lon)
    regrid = F("regrid", matrix=path)
    single = _forward(monkeypatch, None, regrid, fields)
    group = _forward(monkeypatch, spec, regrid, fields)
    assert all(f.decodes == 0 for f in fields)
    for k, msg in enumerate(msgs):
        want = m @ ogx.decode(msg, n_points=s_lat.size)
        assert_same_values(single[k], want, f"single engine, field {k}")
        assert_same_values(group[k], want, f"{spec}, field {k}")


# ------------------------------------------------------------------ malformed fields ------
def _with_section7(msg: bytes, data: bytes) -> bytes:
    return ogc._rebuild(msg, {7: data})


def _patch5(msg: bytes, octet: int, value: bytes) -> bytes:
    s5 = next(pos for pos, _, number in ogc._sections(msg) if number == 5)
    b = bytearray(msg)
    b[s5 + octet - 1 : s5 + octet - 1 + len(value)] = value
    return bytes(b)


def _refused(cuda, path, m, s_lat, s_lon, good, bad_msgs, index, what):
    from anemoi_transform_b200 import ekd, grib
    from anemoi_transform_b200.filters import create_filter_by_name as F

    n_src = s_lat.size
    fields = _fields(bad_msgs, n_src, s_lat, s_lon)
    packed = grib.packed_of(fields)
    assert packed is not None  # the scan accepts it: only decoding can tell
    with pytest.raises(ValueError, match=f"message {index}: .*{what}"):
        grib.upload(packed)
    with pytest.raises(ValueError, match=f"message {index}: .*{what}"):
        F("regrid", matrix=path).forward(ekd.SimpleFieldList(fields))
    # the engine serves the next call normally
    ok = F("regrid", matrix=path).forward(ekd.SimpleFieldList(_fields(good, n_src, s_lat, s_lon)))
    for k, f in enumerate(ok):
        assert_same_values(f.to_numpy(), m @ ogx.decode(good[k], n_points=n_src), f"after a refusal, field {k}")


def test_malformed_fields_are_refused_and_the_engine_carries_on(cuda, small_matrix):
    path, m, s_lat, s_lon = small_matrix
    n_src = s_lat.size
    rng = np.random.default_rng(3)
    good = [ogx.encode_grib2(np.cumsum(rng.normal(0.0, 0.1, n_src)) + 280.0, 16, 0, order=k % 3) for k in range(6)]
    base = good[3]  # order 0: section 7 is references, widths, lengths, values
    info = ogx.scan(base)
    s7 = base[info["data_offset"] : info["data_offset"] + info["data_length"]]
    ng = info["complex_groups"]
    # true last length one more than the values
    lengths = _patch5(base, 43, struct.pack(">I", info["complex_last_length"] + 1))
    # the values part cut to half
    overrun = _with_section7(base, s7[: info["complex_values_offset"] + (len(s7) - info["complex_values_offset"]) // 2])
    # width reference 40: every group is wider than 32 bits
    wide = _patch5(base, 36, bytes([40]))
    # order 1 with h1 = -1: the first X is negative
    o1 = ogx.encode_grib2(np.cumsum(rng.normal(0.0, 0.1, n_src)) + 280.0, 16, 0, order=1, ww=3)
    i1 = ogx.scan(o1)
    b = bytearray(o1)
    b[i1["data_offset"] : i1["data_offset"] + 3] = b"\x80\x00\x01"
    negative = bytes(b)
    assert ng > 1
    for bad, what in ((lengths, "group lengths"), (overrun, "run past section 7"), (wide, "width above 32"), (negative, r"outside \[0, 2\^32\)")):
        _refused(cuda, path, m, s_lat, s_lon, good, good[:3] + [bad] + good[4:], 3, what)


def test_bitmaps_with_too_many_set_bits_are_refused_on_every_packing(cuda, small_matrix):
    """A bitmap with more set bits than the message has values: simple, CCSDS and complex."""
    path, m, s_lat, s_lon = small_matrix
    n_src = s_lat.size
    rng = np.random.default_rng(4)
    good = [ogx.encode_grib2(np.cumsum(rng.normal(0.0, 0.1, n_src)) + 280.0, 16, 0, order=k % 3) for k in range(4)]
    bm = rng.uniform(size=n_src) > 0.5
    bm[0] = True
    v = rng.normal(280.0, 3.0, int(bm.sum()))
    for make in (ogrib.encode_grib2, ogc.encode_grib2, ogx.encode_grib2):
        msg = make(v, 16, 0, bm)
        info = ogx.scan(msg)
        b = bytearray(msg)
        off = info["bitmap_offset"]
        first_clear = int(np.flatnonzero(~bm)[0])
        b[off + first_clear // 8] |= 0x80 >> (first_clear % 8)  # one more set bit than values
        _refused(cuda, path, m, s_lat, s_lon, good, good[:2] + [bytes(b)] + good[2:], 2, "more set bits")
