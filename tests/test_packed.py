"""CF-packed int16 sources (``io.decode_packed``, ``ctb_pull_pack_decode`` and the ``_decode`` reduce-packs): raw
values decoded on the GPU while the referenced gridcells are packed.

The reference is numpy's ``raw.astype(D) * D(scale) + D(offset)`` with the fill values set to NaN.  Every GPU
result is compared bit for bit (as int64) with the same public call on that numpy-decoded float array of dtype D:
compact and full-grid plans sum in the same order (tests/test_ingest_matrix.py), so the two agree exactly.
CPU: the choice of D, attribute handling, every refusal, takes, raw int16 without ``decode_packed``, the C-ABI's
checks that need no plan and the ``ctb_decode`` layout."""
import ctypes

import numpy as np
import pandas as pd
import pytest

import oracle
from conftest import rel_err
from climate_toolbox_b200 import DataArray, Dataset
from climate_toolbox_b200 import _engine as E
from climate_toolbox_b200 import _native as N
from climate_toolbox_b200 import synthetic
from climate_toolbox_b200.aggregations.aggregations import (_GridView, _aggregate_core, _group_requests, _resolve,
                                                            weighted_aggregate_grid_to_regions,
                                                            weighted_aggregate_grid_to_regions_multi)
from climate_toolbox_b200.io import decode_packed
from climate_toolbox_b200.transformations.transformations import (snyder_edd, snyder_gdd, subdaily_bins,
                                                                  subdaily_edd, subdaily_gdd, tas_bins, tas_poly,
                                                                  tas_rcspline)
from climate_toolbox_b200.utils.utils import (convert_kelvin_to_celsius, convert_lons_split,
                                              get_daily_growing_season_mask, remove_leap_days, resample_daily)

F32, F64 = np.dtype("float32"), np.dtype("float64")
FILL, MISSING = -32767, -32768
START = "2003-12-20"        # a year end and 29 February 2004 within 80 days


def decode_ref(raw, scale, offset, fills, D):
    """numpy's CF decoding: ``raw.astype(D) * D(scale) + D(offset)``, NaN at the fill values."""
    D = np.dtype(D).type
    y = raw.astype(D) * D(scale) + D(offset)
    y[np.isin(raw, list(fills))] = np.nan
    return y


def encode(x, D):
    """(raw int16, attrs) of float data ``x``: ERA5-style packing with float64 attributes (D = float64) or float32
    attributes (D = float32); NaN becomes _FillValue, and a few values are set to missing_value."""
    lo, hi = float(np.nanmin(x)), float(np.nanmax(x))
    scale, offset = (hi - lo) / 65530.0, (hi + lo) / 2.0
    if np.dtype(D) == F32:
        scale, offset = np.float32(scale), np.float32(offset)
    with np.errstate(invalid="ignore"):
        raw = np.clip(np.round((x - offset) / scale), -32766, 32767)
    raw = np.where(np.isnan(raw), FILL, raw).astype(np.int16)
    raw.reshape(-1)[::997] = MISSING
    attrs = {"units": "K", "scale_factor": scale, "add_offset": offset, "_FillValue": np.int16(FILL),
             "missing_value": np.int16(MISSING), "long_name": "2 metre temperature"}
    return raw, attrs


def _bits(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a.view(np.int64)


def assert_bits(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.dtype == ref.dtype and got.shape == ref.shape, (got.dtype, ref.dtype, got.shape, ref.shape)
    np.testing.assert_array_equal(_bits(got), _bits(ref))


# ----------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------
def _var(attrs, dtype=np.int16, dims=("time", "lat", "lon")):
    return Dataset({"tas": (dims, np.zeros((2, 2, 4), dtype=dtype), attrs)},
                   coords={"time": pd.date_range("2000-01-01", periods=2).values, "lat": [0.0, 1.0],
                           "lon": [0.0, 1.0, 2.0, 3.0]})


@pytest.mark.parametrize("attrs, D", [
    ({"scale_factor": np.float32(0.5)}, F32),
    ({"scale_factor": np.float32(0.5), "add_offset": np.float32(2.0)}, F32),
    ({"_FillValue": np.int16(-1)}, F32),
    ({"missing_value": np.int16(-1)}, F32),
    ({"scale_factor": 0.5}, F64),                                          # a Python float is float64
    ({"scale_factor": np.float64(0.5), "add_offset": np.float64(2.0)}, F64),
    ({"scale_factor": np.float32(0.5), "add_offset": np.float64(2.0)}, F64),
    ({"add_offset": np.float32(2.0)}, F64),
    ({"add_offset": np.float64(2.0), "_FillValue": np.int16(-1)}, F64),
])
def test_decoded_dtype(attrs, D):
    v = decode_packed(_var(attrs))._vars["tas"]
    assert v.deferred.kind == "decode" and v.dtype == D and v.deferred.params[3] == D
    scale, offset, fills, _ = v.deferred.params
    assert scale == float(attrs.get("scale_factor", 1.0)) and offset == float(attrs.get("add_offset", 0.0))
    assert fills == tuple(sorted({int(attrs[k]) for k in ("_FillValue", "missing_value") if k in attrs}))


def test_attributes_and_pass_through():
    ds = _var({"units": "K", "scale_factor": 0.5, "add_offset": 1.0, "_FillValue": np.int16(-1),
               "missing_value": np.array([-2, -1], dtype=np.int16), "long_name": "t"})
    ds["f"] = (("time", "lat", "lon"), np.ones((2, 2, 4), dtype=np.float32), {"scale_factor": 2.0, "units": "K"})
    ds["raw"] = (("time", "lat", "lon"), np.ones((2, 2, 4), dtype=np.int16), {"units": "1"})
    ds["z"] = (("lat", "lon"), np.ones((2, 4)))
    out = decode_packed(ds)
    v = out._vars["tas"]
    assert v.attrs == {"units": "K", "long_name": "t"}
    assert v.deferred.params[2] == (-2, -1) and v.shape == (2, 2, 4) and v.dims == ("time", "lat", "lon")
    assert ds._vars["tas"].attrs["scale_factor"] == 0.5                    # the input is not changed
    for k in ("f", "raw", "z"):                  # float variables pass through whatever their attributes
        assert out._vars[k] is ds._vars[k]
    da = decode_packed(ds["tas"])
    assert isinstance(da, DataArray) and da.variable.deferred.kind == "decode" and da.name == "tas"


@pytest.mark.parametrize("dtype", [np.int8, np.uint8, np.int32, np.uint16])
def test_refuses_other_integer_packing(dtype):
    with pytest.raises(ValueError, match="int16"):
        decode_packed(_var({"scale_factor": 0.5}, dtype=dtype))


@pytest.mark.parametrize("attrs, match", [
    ({"scale_factor": 0.5, "_Unsigned": "true"}, "_Unsigned"),
    ({"_FillValue": -1.5}, "int16 integers"),
    ({"_FillValue": np.float32(-1.0)}, "int16 integers"),
    ({"missing_value": 40000}, "int16 integers"),
    ({"_FillValue": np.int16(1), "missing_value": np.array([2, 3, 4, 5], dtype=np.int16)}, "at most 4"),
    ({"scale_factor": np.nan}, "finite"),
    ({"add_offset": np.inf}, "finite"),
])
def test_refusals(attrs, match):
    with pytest.raises(ValueError, match=match):
        decode_packed(_var(attrs))


def test_dims():
    with pytest.raises(NotImplementedError):
        decode_packed(_var({"scale_factor": 0.5}, dims=("lat", "lon", "time")))
    with pytest.raises(ValueError):
        decode_packed(_var({"scale_factor": 0.5}, dims=("time", "y", "x")))
    # four fill values are fine; duplicates count once
    ok = decode_packed(_var({"_FillValue": np.int16(1), "missing_value": np.array([1, 2, 3, 4], dtype=np.int16)}))
    assert ok._vars["tas"].deferred.params[2] == (1, 2, 3, 4)


def test_takes_compose_onto_the_source():
    lat, lon = synthetic.grid_labels(30.0, lon_0_360=True)
    time = pd.date_range("2004-02-27", periods=4).values
    raw = np.arange(4 * len(lat) * len(lon), dtype=np.int16).reshape(4, len(lat), len(lon))
    ds = Dataset({"tas": (("time", "lat", "lon"), raw, {"scale_factor": 0.5, "units": "K"})},
                 coords={"time": time, "lat": lat, "lon": lon})
    d = convert_lons_split(remove_leap_days(decode_packed(ds)), "lon")
    v = d._vars["tas"]
    assert v.deferred.kind == "decode" and v.dtype == F64
    src = v.deferred.sources[0]
    assert src.physical is raw
    np.testing.assert_array_equal(src.takes["time"], [0, 1, 3])
    np.testing.assert_array_equal(src.takes["lon"], np.argsort((lon + 180) % 360 - 180, kind="stable"))
    assert v.shape == (3, len(lat), len(lon))
    # daily reductions read the raw source; a time take must be one run of steps
    h = Dataset({"tas": (("time", "lat", "lon"), np.zeros((48, 2, 4), dtype=np.int16), {"scale_factor": 0.5})},
                coords={"time": pd.date_range("2000-01-01", periods=48, freq="h").values, "lat": [0.0, 1.0],
                        "lon": [0.0, 1.0, 2.0, 3.0]})
    r = resample_daily(decode_packed(h).isel(time=np.arange(24, 48)), "max")
    dv = r._vars["tas"]
    assert dv.deferred.params[:3] == ("max", 24, 24) and dv.dtype == F64
    inner = dv.deferred.sources[0]
    assert inner.deferred.kind == "decode" and "time" not in inner.deferred.sources[0].takes


def test_raw_int16_without_decode_packed():
    """Without decode_packed an int16 variable is read as raw numbers: widened to float64, attributes ignored."""
    ds = _var({"scale_factor": 0.5, "add_offset": 100.0})
    ds._vars["tas"]._data[:] = np.arange(16, dtype=np.int16).reshape(2, 2, 4)
    v = _GridView(ds._vars["tas"])
    assert v.data2d.dtype == np.float64 and v.elem_bytes == 8
    np.testing.assert_array_equal(v.data2d.reshape(-1), np.arange(16))


def test_fusion_and_source_rules():
    x = np.zeros((4, 2, 4), dtype=np.int16)
    coords = {"time": pd.date_range("2001-01-01", periods=4).values, "lat": [0.0, 1.0], "lon": [0.0, 1.0, 2.0, 3.0]}
    ds = decode_packed(Dataset({"tas": (("time", "lat", "lon"), x, {"scale_factor": 0.5, "units": "K"}),
                                "t32": (("time", "lat", "lon"), x, {"scale_factor": np.float32(0.5), "units": "K"}),
                                "f": (("time", "lat", "lon"), x.astype(np.float64), {"units": "K"})}, coords=coords))
    p = tas_poly(ds, [1, 2, 3, 4], ["p1", "p2", "p3", "p4"])
    g = _group_requests([(n,) + _resolve(p._vars[n]) for n in ("p1", "p2", "p3", "p4")])
    assert len(g) == 1 and g[0]["srcs"][0].deferred.kind == "decode"
    c = convert_kelvin_to_celsius(ds, "tas")
    assert c._vars["tas"].deferred.sources[0].deferred.kind == "decode"
    df = pd.DataFrame({"lat": [0.0], "lon": [0.0], "popwt": [1.0], "areawt": [1.0], "hierid": ["a"]})
    # Snyder's two inputs: both decoded with the same D, or neither
    for a, b in (("tas", "f"), ("f", "tas"), ("tas", "t32")):
        e = snyder_edd(ds[a], ds[b], 300.0, check=False)
        with pytest.raises(ValueError, match="two-input"):
            _aggregate_core(Dataset({"e": e.variable}, coords=coords), ["e"], "popwt", "hierid", df, "areawt")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G
    G.build()
    return N.lib()


def test_decode_struct_layout(lib):
    assert ctypes.sizeof(N.Decode) == 8 + 8 + 4 + 4 + 4 * 2
    assert N.Decode.fill.offset == 24


def test_abi_refusals_without_a_plan(lib):
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    dec = N.Decode(1.0, 0.0, N.F32, 0)
    assert lib.ctb_pull_pack_decode(None, p, 1024, ctypes.byref(dec), None, 0, 4, p, None) == N.ERR_INVALID
    assert "ctb_pull_pack_decode" in N.last_error() and "compact plan" in N.last_error()
    assert lib.ctb_pull_pack_daily_decode(None, p, 1024, ctypes.byref(dec), 24, None, 0, 4, N.DAILY_MEAN, p, None,
                                          None, None) == N.ERR_INVALID
    assert "ctb_pull_pack_daily_decode" in N.last_error()
    prm = (ctypes.c_double * 1)(1.0)
    assert lib.ctb_pull_pack_daily_steps_decode(None, p, 1024, ctypes.byref(dec), 24, None, 0, 4, N.STEP_EDD, prm, 1,
                                                1, (ctypes.c_void_p * 1)(p), None) == N.ERR_INVALID
    assert "ctb_pull_pack_daily_steps_decode" in N.last_error()


# ----------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------
def _put(a, where):
    import torch
    if where == "device":
        return torch.from_numpy(a).cuda()
    if where == "pageable":
        return a
    host = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
    host.copy_(torch.from_numpy(a))
    return host.numpy()


def _pair(D, where="device", n_days=80, S=1, d=3.0, R=300, lon_0_360=False, seed=3):
    """(packed Dataset after decode_packed, the same Dataset on the numpy-decoded float array of D, weights, raw,
    attrs)."""
    lat, lon = synthetic.grid_labels(d, lon_0_360=lon_0_360)
    df = synthetic.weights_table(d, R, seed=5)
    x, _, _ = synthetic.tas_field(n_days * S, len(lat), len(lon), seed=seed, nan_frac=0.01)
    raw, attrs = encode(x, D)
    ref = decode_ref(raw, attrs["scale_factor"], attrs["add_offset"], (FILL, MISSING), D)
    if S == 1:
        time = pd.date_range(START, periods=n_days, freq="D").values
    else:
        time = pd.date_range(START, periods=n_days * S, freq="{}min".format(24 * 60 // S)).values
    coords = {"time": time, "lat": lat, "lon": lon}
    keep = {k: v for k, v in attrs.items() if k in ("units", "long_name")}
    packed = decode_packed(Dataset({"tas": (("time", "lat", "lon"), _put(raw, where), attrs)}, coords=coords))
    plain = Dataset({"tas": (("time", "lat", "lon"), _put(ref, where), keep)}, coords=coords)
    return packed, plain, df, raw, attrs


def _agg(ds, names, df, **kw):
    return weighted_aggregate_grid_to_regions(ds, names, "popwt", "hierid", weights=df, **kw)


def _same_result(got, ref, names):
    for n in names:
        assert got[n].dims == ref[n].dims
        assert_bits(got[n].values, ref[n].values)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [F32, F64])
def test_values_every_raw_value(D):
    """.values decodes all 65,536 int16 values, two of them fill values, through the full-grid plan."""
    raw = np.arange(-32768, 32768, dtype=np.int64).astype(np.int16).reshape(4, 128, 128)
    raw = np.concatenate([raw, raw[::-1, ::-1, ::-1]])        # 8 planes: the values in two orders
    scale, offset = (np.float32(0.0017), np.float32(261.3)) if D == F32 else (0.0017180, 261.30517)
    attrs = {"scale_factor": scale, "add_offset": offset, "_FillValue": np.int16(FILL),
             "missing_value": np.int16(MISSING)}
    for where in ("device", "pinned", "pageable"):
        ds = Dataset({"tas": (("time", "lat", "lon"), _put(raw, where), attrs)},
                     coords={"time": np.arange(8), "lat": np.arange(128.0), "lon": np.arange(128.0)})
        got = decode_packed(ds).tas.values
        ref = decode_ref(raw, scale, offset, (FILL, MISSING), D)
        assert got.dtype == D and np.isnan(got).sum() == 4
        np.testing.assert_array_equal(got.view(np.int32 if D == F32 else np.int64),
                                      ref.view(np.int32 if D == F32 else np.int64))
    # a negative scale and no fill values
    ds = Dataset({"tas": (("time", "lat", "lon"), _put(raw, "device"), {"scale_factor": -scale})},
                 coords={"time": np.arange(8), "lat": np.arange(128.0), "lon": np.arange(128.0)})
    got = decode_packed(ds).tas.values
    np.testing.assert_array_equal(got, decode_ref(raw, -scale, 0.0, (), D))


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned", "pageable"])
@pytest.mark.parametrize("D", [F32, F64])
def test_identity(D, where):
    packed, plain, df, _, _ = _pair(D, where)
    _same_result(_agg(packed, "tas", df), _agg(plain, "tas", df), ["tas"])


@pytest.mark.gpu
@pytest.mark.parametrize("D", [F32, F64])
def test_time_options(D):
    packed, plain, df, _, _ = _pair(D, "pinned", lon_0_360=True)
    lat = np.asarray(packed.coords["lat"].values)
    for f in (lambda ds: convert_lons_split(ds, "lon"), lambda ds: convert_lons_split(remove_leap_days(ds), "lon")):
        _same_result(_agg(f(packed), "tas", df), _agg(f(plain), "tas", df), ["tas"])
    p, q = convert_lons_split(packed, "lon"), convert_lons_split(plain, "lon")
    _same_result(_agg(p, "tas", df, time_groups="year"), _agg(q, "tas", df, time_groups="year"), ["tas"])
    lon = np.asarray(p.coords["lon"].values)
    z = np.random.default_rng(2).uniform(1, 366, (2, len(lat), len(lon)))
    gd = Dataset({"variable": (("z", "latitude", "longitude"), z)},
                 coords={"z": np.array([1, 2]), "latitude": lat, "longitude": lon + 180.0})
    mask = get_daily_growing_season_mask(lat, np.asarray(p.coords["lon"].values), p.coords["time"].values, gd)
    _same_result(_agg(p, "tas", df, season_mask=mask), _agg(q, "tas", df, season_mask=mask), ["tas"])
    m1 = weighted_aggregate_grid_to_regions_multi(p, "tas", ["popwt", "areawt"], "hierid", df)
    m2 = weighted_aggregate_grid_to_regions_multi(q, "tas", ["popwt", "areawt"], "hierid", df)
    _same_result(m1, m2, ["tas_popwt", "tas_areawt"])


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned"])
@pytest.mark.parametrize("D", [F32, F64])
def test_transforms_fuse(D, where):
    packed, plain, df, _, _ = _pair(D, where, n_days=300)
    _agg(packed, "tas", df)                      # builds the plan
    n0 = E.launch_count()
    _agg(packed, "tas", df)
    per_group = E.launch_count() - n0            # one decode-pack and the aggregation
    names = ["p1", "p2", "p3", "p4"]
    cases = [(lambda ds: tas_poly(ds, [1, 2, 3, 4], names), names),
             (lambda ds: tas_bins(ds, [-np.inf, -5, 0, 5, 10, 20, 30, np.inf], "b"), ["b_{}".format(k) for k in range(7)]),
             (lambda ds: tas_rcspline(ds, [-5, 5, 15, 25, 30], "r"), ["r_{}".format(k) for k in range(4)]),
             (lambda ds: convert_kelvin_to_celsius(ds, "tas"), ["tas"])]
    for make, ns in cases:
        n0 = E.launch_count()
        got = _agg(make(packed), ns, df)
        assert E.launch_count() - n0 == per_group * (-(-len(ns) // N.MAX_OUT))
        _same_result(got, _agg(make(plain), ns, df), ns)
    # Snyder: two decoded sources, one decode-pack each, one aggregation for two thresholds
    x2 = plain.tas.values + np.float64(5.0).astype(D)
    raw2, attrs2 = encode(x2, D)
    ref2 = decode_ref(raw2, attrs2["scale_factor"], attrs2["add_offset"], (FILL, MISSING), D)
    packed["tasmax"] = decode_packed(DataArray(_put(raw2, where), dims=("time", "lat", "lon"), attrs=attrs2))
    plain["tasmax"] = (("time", "lat", "lon"), _put(ref2, where), {"units": "K"})
    for ds in (packed, plain):
        ds["e1"] = snyder_edd(ds.tas, ds.tasmax, 290.0, check=False)
        ds["e2"] = snyder_edd(ds.tas, ds.tasmax, 300.0, check=False)
        ds["g"] = snyder_gdd(ds.tas, ds.tasmax, 280.0, 300.0, check=False)
    _agg(packed, ["g"], df)                      # builds the plan of two inputs
    n0 = E.launch_count()
    got = _agg(packed, ["e1", "e2", "g"], df)
    # per group and time chunk: two decode-packs and one aggregation, where identity has one of each
    assert E.launch_count() - n0 == 2 * (3 * per_group // 2)
    _same_result(got, _agg(plain, ["e1", "e2", "g"], df), ["e1", "e2", "g"])


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned", "pageable"])
@pytest.mark.parametrize("D", [F32, F64])
def test_subdaily(D, where):
    S, n_days = 24, 40
    packed, plain, df, _, _ = _pair(D, where, n_days=n_days, S=S, d=6.0, R=150)
    for how in ("mean", "min", "max"):
        a, b = resample_daily(packed, how), resample_daily(plain, how)
        assert a.tas.dtype == b.tas.dtype
        np.testing.assert_array_equal(a.tas.values, b.tas.values)
        _same_result(_agg(a, "tas", df), _agg(b, "tas", df), ["tas"])
    for make in (lambda ds: subdaily_edd(ds.tas, 295.0), lambda ds: subdaily_gdd(ds.tas, 283.0, 303.0)):
        a, b = make(packed), make(plain)
        np.testing.assert_array_equal(a.values, b.values)
        _same_result(_agg(Dataset({"e": a.variable}, coords=a._coords), "e", df),
                     _agg(Dataset({"e": b.variable}, coords=b._coords), "e", df), ["e"])
    edges = [-np.inf, 270.0, 280.0, 290.0, 300.0]
    a, b = subdaily_bins(packed.tas, edges, "h"), subdaily_bins(plain.tas, edges, "h")
    names = ["h_{}".format(k) for k in range(4)]
    _same_result(_agg(a, names, df, time_groups="year"), _agg(b, names, df, time_groups="year"), names)


@pytest.mark.gpu
def test_against_the_oracle():
    """One decoded case against the restated reference aggregation, at the kernel matrix's bound."""
    packed, plain, df, raw, attrs = _pair(F64, "pinned")
    got = _agg(tas_poly(packed, 2, "p"), "p", df)["p"].values
    x = plain.tas.values
    xt, _ = oracle.tas_poly(x, plain.coords["time"].values, 2)
    ref, dims, labels = oracle.weighted_aggregate_grid_to_regions(
        xt, ("time", "lat", "lon"), plain.coords["lat"].values, plain.coords["lon"].values, df, "popwt", "hierid")
    assert rel_err(got, ref) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 24])
def test_pcie_bytes(S):
    """A pinned int16 source: 8 bytes per referenced piece and step cross PCIe, once."""
    n_days = 30
    packed, _, df, _, _ = _pair(F64, "pinned", n_days=n_days, S=S)
    ds = resample_daily(packed) if S > 1 else packed
    before = E.TRANSFER_BYTES["h2d"]
    _agg(ds, "tas", df)
    moved = E.TRANSFER_BYTES["h2d"] - before
    lat, lon = packed.coords["lat"].values, packed.coords["lon"].values
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", stage_bytes=8, compact=True, elem_bytes=8)
    assert moved == n_days * S * plan.info["n_pieces_distinct"] * 8


@pytest.mark.gpu
def test_offsets_past_2_31_elements():
    """An hourly int16 source at 0.25 degrees: day 86 starts past 2^31 elements (4 GiB of bytes)."""
    import torch
    nlat, nlon, S, n_days = 721, 1440, 24, 87
    ncell = nlat * nlon
    need = n_days * S * ncell * 2
    free = torch.cuda.mem_get_info()[0]
    if free < need + (4 << 30):
        pytest.skip("needs {} bytes of free device memory, {} free".format(need + (4 << 30), free))
    assert 86 * S * ncell < 2 ** 31 <= (86 * S + S - 1) * ncell      # day 86's reads cross 2^31 elements
    x = torch.empty((n_days * S, nlat, nlon), dtype=torch.int16, device="cuda")
    cell = torch.arange(ncell, device="cuda", dtype=torch.int64).view(nlat, nlon)
    for t in range(n_days * S):
        x[t] = ((cell * 7919 + t * 104729) % 65536 - 32768).to(torch.int16)
    attrs = {"scale_factor": 0.0017, "add_offset": 261.3, "_FillValue": np.int16(FILL), "units": "K"}
    ds = Dataset({"tas": (("time", "lat", "lon"), x, attrs)},
                 coords={"time": pd.date_range("2001-01-01", periods=n_days * S, freq="h").values,
                         "lat": np.arange(nlat, dtype=np.float64), "lon": np.arange(nlon, dtype=np.float64)})
    p = decode_packed(ds)
    last = x[86 * S:].cpu().numpy()
    ref = decode_ref(last, 0.0017, 261.3, (FILL,), F64)
    got = p.isel(time=[86 * S + 23]).tas.values[0]                 # decode-pack with a time index
    assert_bits(got, ref[23])
    got = resample_daily(p, "mean").isel(time=[86]).tas.values[0]
    with np.errstate(invalid="ignore"):
        s = np.zeros(ref.shape[1:])
        c = np.zeros(ref.shape[1:])
        for h in range(S):
            ok = ~np.isnan(ref[h])
            s = np.where(ok, s + ref[h], s)
            c += ok
        assert_bits(got, s / c)
    got = resample_daily(p, "max").isel(time=[86]).tas.values[0]
    assert_bits(got, np.fmax.reduce(ref, axis=0))
    got = subdaily_edd(p.tas, 262.0).isel(time=[86]).values[0]
    with np.errstate(invalid="ignore"):
        s = np.zeros(ref.shape[1:])
        c = np.zeros(ref.shape[1:])
        for h in range(S):
            ok = ~np.isnan(ref[h])
            s = np.where(ok, s + np.where(ref[h] > 262.0, ref[h] - 262.0, 0.0), s)
            c += ok
        assert_bits(got, s / c)
    del x
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_abi_checks_with_a_plan(lib):
    import torch
    lat, lon = synthetic.grid_labels(3.0)
    df = synthetic.weights_table(3.0, 50, seed=5)
    g = E.GridSpec(lat, lon)
    p4 = E.get_plan(g, df, "popwt", "hierid", compact=True, elem_bytes=4, cache=False)
    p8 = E.get_plan(g, df, "popwt", "hierid", compact=True, elem_bytes=8, cache=False)
    ncell = len(lat) * len(lon)
    x = torch.zeros((4 * 24 + 1, ncell), dtype=torch.int16, device="cuda")
    d8 = torch.full((4, p8.info["n_packed_cells"]), 7.0, dtype=torch.float64, device="cuda")
    d4 = torch.full((4, p4.info["n_packed_cells"]), 7.0, dtype=torch.float32, device="cuda")
    L = lib
    good64, good32 = N.Decode(0.5, 1.0, N.F64, 1, (ctypes.c_int16 * 4)(-1)), N.Decode(0.5, 1.0, N.F32, 0)
    bad = [None, N.Decode(float("nan"), 0.0, N.F64, 0), N.Decode(1.0, float("inf"), N.F64, 0),
           N.Decode(1.0, 0.0, N.F64, 5), N.Decode(1.0, 0.0, N.F64, -1), N.Decode(1.0, 0.0, 7, 0)]
    prm = (ctypes.c_double * 1)(290.0)

    def calls(plan, dst, dec, xp):
        dp = None if dec is None else ctypes.byref(dec)
        return [L.ctb_pull_pack_decode(plan._h, xp, ncell, dp, None, 0, 4, dst.data_ptr(), None),
                L.ctb_pull_pack_daily_decode(plan._h, xp, ncell, dp, 24, None, 0, 4, N.DAILY_MEAN, dst.data_ptr(),
                                             None, None, None),
                L.ctb_pull_pack_daily_steps_decode(plan._h, xp, ncell, dp, 24, None, 0, 4, N.STEP_EDD, prm, 1, 1,
                                                   (ctypes.c_void_p * 1)(dst.data_ptr()), None)]

    for dec in bad:
        assert calls(p8, d8, dec, x.data_ptr()) == [N.ERR_INVALID] * 3
        assert "dec" in N.last_error()
    # an int16 plane 2 bytes off its 8-byte alignment
    assert calls(p8, d8, good64, x.data_ptr() + 2) == [N.ERR_UNSUPPORTED] * 3
    assert "8-byte aligned" in N.last_error()
    # plan element size against D (decoded planes) or float64 (mean and step planes)
    assert L.ctb_pull_pack_decode(p8._h, x.data_ptr(), ncell, ctypes.byref(good32), None, 0, 4, d8.data_ptr(),
                                  None) == N.ERR_INVALID
    assert L.ctb_pull_pack_decode(p4._h, x.data_ptr(), ncell, ctypes.byref(good64), None, 0, 4, d4.data_ptr(),
                                  None) == N.ERR_INVALID
    assert L.ctb_pull_pack_daily_decode(p4._h, x.data_ptr(), ncell, ctypes.byref(good32), 24, None, 0, 4,
                                        N.DAILY_MIN, None, d4.data_ptr(), None, None) == N.OK
    assert L.ctb_pull_pack_daily_decode(p8._h, x.data_ptr(), ncell, ctypes.byref(good32), 24, None, 0, 4,
                                        N.DAILY_MIN, None, d8.data_ptr(), None, None) == N.ERR_INVALID
    torch.cuda.synchronize()
    assert (d8 == 7.0).all()                                        # no refused call wrote anything
    assert not (d4 == 7.0).all()                                    # the accepted call did
    assert calls(p8, d8, good64, x.data_ptr()) == [N.OK] * 3
    torch.cuda.synchronize()
    for p in (p4, p8):
        p.close()
