"""Temperature bins (``tas_bins``, ``CTB_TR_BINS``): days per temperature bin, fused into the aggregation.

CPU: the reference membership rule (``bins_ref``; the parity tests feed it to the restated reference
aggregation of ``oracle``), ``tas_bins`` metadata and validation, the fusion of contiguous bins into launches,
and the C-ABI's parameter checks.  GPU: the fused aggregation and ``.values`` against the reference --
membership bit-exact, aggregates to the summation-order tolerance."""
import ctypes

import numpy as np
import pandas as pd
import pytest

import oracle
from conftest import rel_err
from climate_toolbox_b200 import Dataset
from climate_toolbox_b200._xr import Variable
from climate_toolbox_b200 import _engine as E
from climate_toolbox_b200 import _native as N
from climate_toolbox_b200 import synthetic
from climate_toolbox_b200.aggregations.aggregations import (_group_requests, _resolve,
                                                            weighted_aggregate_grid_to_regions)
from climate_toolbox_b200.transformations.transformations import tas_bins, tas_poly

OFF = 273.15
INF = np.inf


# ----------------------------------------------------------------------------
# the reference semantics of the bins (numpy), beside the restated reference in oracle/
# ----------------------------------------------------------------------------
def bins_ref(x, lo, hi, offset=OFF):
    """Temperature bin indicator: 1.0 where ``lo <= x - offset < hi``, 0.0 elsewhere, NaN where ``x`` is NaN.
    ``x`` is widened to float64 first and the subtraction and both comparisons are float64 (DESIGN.md
    "dtype policy"); +inf lies in no bin, -inf in a bin whose lower edge is -inf."""
    d = np.asarray(x).astype(np.float64) - offset
    with np.errstate(invalid="ignore"):
        out = ((d >= lo) & (d < hi)).astype(np.float64)
    return np.where(np.isnan(d), np.nan, out)


def tas_bins_ref(tas, times, lo, hi, time_axis=0):
    """The bins of ``tas`` (K) after leap-day removal, shaped like ``oracle.tas_poly``.  Returns
    ``(values, new_time_labels)``."""
    keep = oracle.leap_day_keep_mask(times)
    tas = np.compress(keep, np.asarray(tas), axis=time_axis)
    if tas.shape[time_axis] > 365:
        raise ValueError
    return bins_ref(tas, lo, hi), oracle.tas_poly_time_labels(np.asarray(times)[keep])


def _first_at_or_above(e, dtype):
    """The smallest ``x`` of ``dtype`` whose float64 ``x - 273.15`` is >= ``e``: the value on the edge."""
    x = dtype(e + OFF)
    while np.float64(x) - OFF >= e:
        x = np.nextafter(x, dtype(-INF))
    while np.float64(x) - OFF < e:
        x = np.nextafter(x, dtype(INF))
    return x


def _adjacent(e, dtype):
    """One ulp below, on, and one ulp above the edge ``e`` in ``dtype``."""
    x = _first_at_or_above(e, dtype)
    return np.array([np.nextafter(x, dtype(-INF)), x, np.nextafter(x, dtype(INF))], dtype=dtype)


def _f32_edge():
    """An edge that float32 data meets exactly: float64(float32(283.15)) - 273.15."""
    return np.float64(np.float32(283.15)) - OFF


# ----------------------------------------------------------------------------
# reference pins (CPU)
# ----------------------------------------------------------------------------
def test_reference_bins_hand_computed():
    x = np.array([273.15 + 10.0, 273.15 + 20.0, 273.15 + 15.0, 273.15 + 9.5, np.nan, 273.15 + 25.0])
    # float64: 273.15 + 10.0 and 273.15 + 20.0 are exact sums, so x - 273.15 lands on the edges
    np.testing.assert_array_equal(bins_ref(x, 10.0, 20.0), [1.0, 0.0, 1.0, 0.0, np.nan, 0.0])
    np.testing.assert_array_equal(bins_ref(x, 20.0, 30.0), [0.0, 1.0, 0.0, 0.0, np.nan, 1.0])
    assert np.isnan(bins_ref(np.float32(np.nan), -INF, INF))


def test_reference_bins_infinite_edges_and_data():
    x = np.array([-INF, INF, 0.0, 1e300, -1e300])
    np.testing.assert_array_equal(bins_ref(x, -INF, 0.0), [1.0, 0.0, 1.0, 0.0, 1.0])    # -inf in the first bin
    np.testing.assert_array_equal(bins_ref(x, 0.0, INF), [0.0, 0.0, 0.0, 1.0, 0.0])     # +inf in no bin
    np.testing.assert_array_equal(bins_ref(x, -INF, INF), [1.0, 0.0, 1.0, 1.0, 1.0])
    # bins covering (-inf, inf) sum to 1 for every value but NaN and +inf
    edges = [-INF, -5.0, 0.0, 12.5, INF]
    y = np.array([-INF, 260.0, 273.15, 280.0, 300.0, 1e10])
    total = sum(bins_ref(y, lo, hi) for lo, hi in zip(edges[:-1], edges[1:]))
    np.testing.assert_array_equal(total, np.ones_like(y))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_reference_bins_at_the_edges(dtype):
    """x on, one ulp below and one ulp above the value whose float64 x - 273.15 rounds onto an edge."""
    for e in (_f32_edge(), 20.0, 0.1, -40.0):
        below, on, above = _adjacent(e, dtype)
        assert np.float64(below) - OFF < e <= np.float64(on) - OFF < np.float64(above) - OFF
        np.testing.assert_array_equal(bins_ref(np.array([below, on, above]), e, e + 5.0), [0.0, 1.0, 1.0])
        np.testing.assert_array_equal(bins_ref(np.array([below, on, above]), e - 5.0, e), [1.0, 0.0, 0.0])
    # exactly on the edge
    assert np.float64(np.float32(283.15)) - OFF == _f32_edge()
    assert bins_ref(np.float32(283.15), _f32_edge(), 20.0) == 1.0
    assert np.float64(273.15 + 20.0) - OFF == 20.0
    # the order matters: float32(293.15) is below 293.15, so it lies under the edge 20 once widened and
    # subtracted, although it equals the edge shifted to Kelvin and rounded to float32
    x = np.float32(293.15)
    assert x == np.float32(20.0 + OFF)
    assert bins_ref(x, 20.0, 30.0) == 0.0 and bins_ref(x, 10.0, 20.0) == 1.0


def test_reference_tas_bins_drops_leap_days():
    t = pd.date_range("2000-02-27", periods=5)
    tas = np.array([270.0, 280.0, 290.0, 300.0, np.nan])[:, None]
    v, labels = tas_bins_ref(tas, t, 0.0, 20.0)
    np.testing.assert_array_equal(v[:, 0], [0.0, 1.0, 0.0, np.nan])
    np.testing.assert_array_equal(labels, oracle.tas_poly_time_labels(t[[0, 1, 3, 4]]))


# ----------------------------------------------------------------------------
# tas_bins metadata and validation (CPU)
# ----------------------------------------------------------------------------
def _small_ds(T=5, start="2000-02-27"):
    t = pd.date_range(start, periods=T)
    return Dataset({"tas": (("time", "lat", "lon"), np.full((T, 2, 2), 290.0, dtype=np.float32))},
                   coords={"time": t, "lat": [0.0, 1.0], "lon": [0.0, 1.0]}), t


def test_tas_bins_names_attrs_and_time():
    ds, t = _small_ds()
    ds1 = tas_bins(ds, [-INF, 0.0, 10.0, INF])
    assert list(ds1.data_vars) == ["tas_bin_0", "tas_bin_1", "tas_bin_2"]
    v = ds1["tas_bin_1"]
    assert v.shape == (4, 2, 2) and v.dims == ("time", "lat", "lon")           # Feb 29 dropped
    np.testing.assert_array_equal(ds1.time.values, oracle.tas_poly_time_labels(t[[0, 1, 3, 4]]))
    assert v.attrs["units"] == "days" and v.attrs["variable"] == "tas_bin_1"
    assert v.attrs["bin_lower"] == 0.0 and v.attrs["bin_upper"] == 10.0
    assert v.attrs["long_title"] == "Days with daily average temperature (degrees C) in [0, 10)"
    assert v.attrs["description"].startswith(v.attrs["long_title"])
    assert "365 day" in v.attrs["description"]
    assert ds1["tas_bin_0"].attrs["bin_lower"] == -INF and ds1["tas_bin_2"].attrs["bin_upper"] == INF
    d = v.variable.deferred
    assert d.kind == "bins" and d.params == (273.15, 0.0, 10.0)
    named = tas_bins(ds, [0.0, 10.0, 20.0], ["cool", "warm"])
    assert list(named.data_vars) == ["cool", "warm"] and named["warm"].attrs["variable"] == "warm"
    assert list(tas_bins(ds, [0, 1], "b").data_vars) == ["b_0"]


@pytest.mark.parametrize("edges,names", [
    ([0.0, 10.0, 10.0], "b"),            # not strictly increasing
    ([10.0, 0.0], "b"),                  # decreasing
    ([0.0, np.nan, 10.0], "b"),          # NaN edge
    ([0.0], "b"),                        # fewer than 2 edges
    ([], "b"),
    ([0.0, INF, 10.0], "b"),             # interior infinity
    ([-INF, -INF, 0.0], "b"),
    ([0.0, INF, INF], "b"),
    ([0.0, 10.0, 20.0], ["only_one"]),   # name count mismatch
    ([0.0, 10.0], ["a", "b"]),
])
def test_tas_bins_rejects_bad_edges_and_names(edges, names):
    ds, _ = _small_ds()
    with pytest.raises(ValueError):
        tas_bins(ds, edges, names)


def test_tas_bins_more_than_365_steps():
    big = Dataset({"tas": (("time", "lat"), np.zeros((400, 1)))},
                  coords={"time": pd.date_range("2001-01-01", periods=400), "lat": [0.0]})
    with pytest.raises(ValueError):
        tas_bins(big, [0.0, 10.0])


# ----------------------------------------------------------------------------
# fusion into launches (CPU)
# ----------------------------------------------------------------------------
def _reqs(ds1):
    return [(n,) + _resolve(ds1._vars[n]) for n in ds1.data_vars]


def test_nine_contiguous_bins_make_launches_of_4_4_1():
    ds, _ = _small_ds()
    edges = [-INF, 0.0, 5.0, 10.0, 15.0, 20.0, 25.0, 30.0, 35.0, INF]
    groups = _group_requests(_reqs(tas_bins(ds, edges)))
    assert [len(g["names"]) for g in groups] == [4, 4, 1]
    assert [g["kind"] for g in groups] == ["bins"] * 3
    assert groups[0]["params"] == (273.15, -INF, 0.0, 5.0, 10.0, 15.0)
    assert groups[1]["params"] == (273.15, 15.0, 20.0, 25.0, 30.0, 35.0)
    assert groups[2]["params"] == (273.15, 35.0, INF)
    assert groups[0]["names"] == ["tas_bin_0", "tas_bin_1", "tas_bin_2", "tas_bin_3"]
    assert groups[2]["names"] == ["tas_bin_8"]


def test_bins_that_do_not_fuse():
    a = Variable(("time", "lat", "lon"), np.zeros((2, 2, 2)))
    b = Variable(("time", "lat", "lon"), np.zeros((2, 2, 2)))

    def n_groups(reqs):
        return len(_group_requests(reqs))

    assert n_groups([("x", "bins", (OFF, 0.0, 5.0), [a]), ("y", "bins", (OFF, 5.0, 10.0), [a])]) == 1
    assert n_groups([("x", "bins", (OFF, 0.0, 5.0), [a]), ("y", "bins", (OFF, 10.0, 15.0), [a])]) == 2   # gap
    assert n_groups([("x", "bins", (OFF, 5.0, 10.0), [a]), ("y", "bins", (OFF, 0.0, 5.0), [a])]) == 2    # out of order
    assert n_groups([("x", "bins", (OFF, 0.0, 5.0), [a]), ("y", "bins", (273.0, 5.0, 10.0), [a])]) == 2  # offset
    assert n_groups([("x", "bins", (OFF, 0.0, 5.0), [a]), ("y", "bins", (OFF, 5.0, 10.0), [b])]) == 2    # source
    # next to a polynomial of the same source: separate launches, the polynomials still fuse
    ds, _ = _small_ds()
    mixed = _reqs(tas_poly(ds, [1, 2], ["p1", "p2"]))
    src = mixed[0][3]
    mixed.insert(1, ("bin", "bins", (OFF, 1.0, 2.0), src))
    groups = _group_requests(mixed)
    assert [(g["kind"], g["names"]) for g in groups] == [("poly", ["p1", "p2"]), ("bins", ["bin"])]
    assert groups[1]["params"] == (OFF, 1.0, 2.0)


# ----------------------------------------------------------------------------
# C-ABI parameter checks without a GPU
# ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G
    G.build()
    return N.lib()


def _transform_rc(L, params, n_out):
    p = np.ascontiguousarray(params, dtype=np.float64)
    dummy = ctypes.c_double(0.0)
    # n = 0: the call validates the parameters and returns before any CUDA call
    return L.ctb_transform(ctypes.addressof(dummy), None, N.F64, 0, N.TR_BINS,
                           p.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), int(p.size), n_out, None, None)


def test_abi_validates_bin_edges(lib):
    assert N.TR_BINS == 4
    assert _transform_rc(lib, [OFF, 0.0, 10.0], 1) == N.OK
    assert _transform_rc(lib, [OFF, -INF, 0.0, 10.0, INF], 3) == N.OK
    assert _transform_rc(lib, [OFF, -INF, 0.0, 5.0, 10.0, INF], 4) == N.OK
    assert _transform_rc(lib, [OFF, 10.0, 0.0], 1) == N.ERR_INVALID                  # decreasing
    assert _transform_rc(lib, [OFF, 0.0, 10.0, 10.0], 2) == N.ERR_INVALID            # not strictly
    assert _transform_rc(lib, [OFF, 0.0, np.nan, 10.0], 2) == N.ERR_INVALID          # NaN edge
    assert _transform_rc(lib, [OFF, 0.0, INF, 10.0], 2) == N.ERR_INVALID             # interior infinity
    assert _transform_rc(lib, [OFF, -INF, -INF, 10.0], 2) == N.ERR_INVALID
    assert _transform_rc(lib, [OFF, 0.0, 10.0, 20.0], 1) == N.ERR_INVALID            # n_params != n_out + 2
    assert _transform_rc(lib, [OFF, 0.0, 10.0], 2) == N.ERR_INVALID
    assert _transform_rc(lib, [OFF] + list(range(6)), 5) == N.ERR_INVALID            # n_out > CTB_MAX_OUT
    assert "BINS" in N.last_error() or "n_out" in N.last_error()


# ----------------------------------------------------------------------------
# GPU: fused aggregation and .values against the oracle
# ----------------------------------------------------------------------------
def _config(d, R, T, seed=1234, nan_frac=0.001, dtype=np.float32):
    lat, lon = synthetic.grid_labels(d)
    df = synthetic.weights_table(d, R, seed=seed)
    tas, _, _ = synthetic.tas_field(T, len(lat), len(lon), seed=7, nan_frac=nan_frac, dtype=dtype)
    return lat, lon, df, tas


def _oracle_agg(x, dims, lat, lon, df, aggwt, agglev):
    return oracle.weighted_aggregate_grid_to_regions(x, dims, lat, lon, df, aggwt, agglev)


def _check(got, ref, tol):
    err = rel_err(got, ref)
    assert err <= tol, err


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_edge_adjacent_values_fused_and_pointwise(dtype):
    """Every gridcell-day holds a value one ulp below, on or one ulp above an edge: the fused kernels
    (streaming: the integer widening of positive float32; direct) and .values agree with the oracle on
    every membership."""
    import torch
    inner = [_f32_edge(), 20.0, 20.1]
    edges = [-INF] + inner + [INF]
    values = np.concatenate([_adjacent(e, dtype) for e in inner])
    lat, lon = synthetic.grid_labels(2.0)
    df = synthetic.weights_table(2.0, 300, seed=11)
    T = 70
    x = np.random.default_rng(5).choice(values, size=(T, len(lat), len(lon))).astype(dtype)
    t = pd.date_range("2001-01-01", periods=T)
    ds = Dataset({"tas": (("time", "lat", "lon"), torch.from_numpy(x).cuda())},
                 coords={"time": t, "lat": lat, "lon": lon})
    ds1 = tas_bins(ds, edges, "b")
    names = list(ds1.data_vars)
    refs = [bins_ref(x, lo, hi) for lo, hi in zip(edges[:-1], edges[1:])]
    for name, ref in zip(names, refs):
        got = ds1[name].values
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got, ref)                   # membership bit-exact
        assert 0.0 < ref.mean() < 1.0                             # every bin populated
    for variant in (N.VARIANT_STAGED, N.VARIANT_DIRECT):
        weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df, variant=variant)
        n0 = E.launch_count()
        out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df, variant=variant)
        assert E.launch_count() - n0 == 1                         # 4 bins, one launch
        for name, ref in zip(names, refs):
            r, rd, labels = _oracle_agg(ref, ("time", "lat", "lon"), lat, lon, df, "popwt", "hierid")
            assert out[name].dims == rd and list(out.hierid.values) == list(labels)
            _check(out[name].values, r, 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("offset,edges", [(OFF, [-INF, -300.0, 0.0, _f32_edge(), INF]),
                                          (0.0, [-INF, -1e-40, 0.0, 1e-40, INF])])
def test_special_floats_one_gridcell_per_region(offset, edges):
    """Every region is one gridcell of weight 1, so each result is the membership itself (0 for NaN data):
    float32 NaN, infinities, signed zeros, denormals and negative values through the streaming kernel (which
    compares float data on the stored type) and the direct kernel, against the oracle exactly."""
    import torch
    nlat, nlon, T = 4, 8, 40
    lat, lon = np.arange(nlat) * 1.0, np.arange(nlon) * 1.0
    special = np.array([np.nan, INF, -INF, 0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.2e-38, -5.0, 3.4e38, -3.4e38,
                        273.15, 283.15, 293.15], dtype=np.float32)
    near = np.concatenate([_adjacent(e, np.float32) for e in edges[1:-1] if offset == OFF] or [special[:0]])
    pool = np.concatenate([special, np.nextafter(special, np.float32(INF)), near])
    x = np.random.default_rng(3).choice(pool, size=(T, nlat * nlon)).astype(np.float32)
    ii, jj = np.divmod(np.arange(nlat * nlon), nlon)
    df = pd.DataFrame({"lat": lat[ii], "lon": lon[jj], "hierid": np.arange(nlat * nlon),
                       "popwt": 1.0, "areawt": 1.0})
    dev = torch.device("cuda", 0)
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", device=dev, cache=False)
    xd = torch.from_numpy(x).to(dev)
    params = (offset,) + tuple(edges)
    exp = np.stack([np.nan_to_num(bins_ref(x, lo, hi, offset), nan=0.0).T
                    for lo, hi in zip(edges[:-1], edges[1:])])
    for variant in (N.VARIANT_STAGED, N.VARIANT_DIRECT):
        out = E.aggregate_device(plan, xd, None, N.LAYOUT_TIME_MAJOR, nlat * nlon, None, T, "bins", params, 4,
                                 variant=variant)
        np.testing.assert_array_equal(out.cpu().numpy(), exp)
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_values_nan_and_infinities_bit_exact(dtype):
    """.values (the pointwise kernel): NaN where tas is NaN, -inf in the first bin, +inf in none."""
    x = np.array([[250.0, np.nan, -INF, INF, 273.15, 293.15, 1e30, -1e30]], dtype=dtype)
    ds = Dataset({"tas": (("time", "x"), x)}, coords={"time": pd.date_range("2001-05-01", periods=1)})
    edges = [-INF, -20.0, 0.0, 20.0, INF]
    ds1 = tas_bins(ds, edges, "b")
    for k, (lo, hi) in enumerate(zip(edges[:-1], edges[1:])):
        got = ds1["b_{}".format(k)].values
        np.testing.assert_array_equal(got, bins_ref(x, lo, hi))
        assert np.isnan(got[0, 1]) and got[0, 2] == (k == 0) and got[0, 3] == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("aggwt,agglev", [("popwt", "ISO"), ("areawt", "hierid")])
def test_reference_fixture_cell_major(ref_fix, aggwt, agglev):
    """The reference fixture (lat, lon, time) float64: CELL_MAJOR, the direct kernel."""
    lat, lon, time, temp, df = ref_fix
    ds = Dataset({"tas": (["lat", "lon", "time"], temp)}, coords={"lon": lon, "lat": lat, "time": time})
    edges = [-INF, -250.0, -225.0, -200.0, INF]          # temp is 0..100 K: -273.15..-173.15 C
    ds1 = tas_bins(ds, edges, "b")
    names = list(ds1.data_vars)
    out = weighted_aggregate_grid_to_regions(ds1, names, aggwt, agglev, weights=df)
    total = 0.0
    for name, lo, hi in zip(names, edges[:-1], edges[1:]):
        xt, tl = tas_bins_ref(temp, time, lo, hi, time_axis=2)
        assert xt.mean() > 0.05                          # every bin populated
        np.testing.assert_array_equal(ds1[name].values, xt)
        ref, rd, labels = _oracle_agg(xt, ("lat", "lon", "time"), lat, lon, df, aggwt, agglev)
        assert out[name].dims == rd and list(out.coords[agglev].values) == list(labels)
        np.testing.assert_array_equal(out.coords["time"].values, tl)
        _check(out[name].values, ref, 1e-12)
        total = total + out[name].values
    np.testing.assert_allclose(total, 1.0, rtol=0, atol=1e-12)     # no NaN in the fixture


def _put(a, where):
    import torch
    if where == "device":
        return torch.from_numpy(a).cuda()
    host = torch.empty(a.shape, dtype=torch.float32 if a.dtype == np.float32 else torch.float64, pin_memory=True)
    host.copy_(torch.from_numpy(a))
    return host.numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "host_pinned"])
def test_quarter_degree_twelve_bins(where):
    """0.25-degree grid, 24,378 regions, 0.1 % NaN, 12 bins over (-inf, inf): three fused launches of 4
    bins (device: the streaming kernel; pinned host: the compact plan and the GPU pull)."""
    lat, lon, df, tas = _config(0.25, 24378, 5)
    t = pd.date_range("2001-06-01", periods=5)
    ds = Dataset({"tas": (("time", "lat", "lon"), _put(tas, where))}, coords={"time": t, "lat": lat, "lon": lon})
    edges = [-INF, -10.0, -5.0, 0.0, 5.0, 10.0, 15.0, 20.0, 25.0, 30.0, 35.0, 40.0, INF]
    ds1 = tas_bins(ds, edges, "b")
    names = list(ds1.data_vars)
    assert len(names) == 12
    out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df)
    if where == "device":
        n0 = E.launch_count()
        out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df)
        assert E.launch_count() - n0 == 3
    dims = ("time", "lat", "lon")
    total = 0.0
    for name, lo, hi in zip(names, edges[:-1], edges[1:]):
        ref, rd, labels = _oracle_agg(bins_ref(tas, lo, hi), dims, lat, lon, df, "popwt", "hierid")
        assert out[name].dims == rd
        _check(out[name].values, ref, 1e-9)
        total = total + out[name].values
    nan_share, _, _ = _oracle_agg(np.isnan(tas).astype(np.float64), dims, lat, lon, df, "popwt", "hierid")
    clean = nan_share == 0                      # region-days without a NaN gridcell (and with weights)
    assert clean.mean() > 0.5 and (nan_share > 0).any()
    np.testing.assert_allclose(total[clean], 1.0, rtol=0, atol=1e-12)
    assert (total[~clean & ~np.isnan(total)] < 1.0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "host"])
def test_time_groups_year_gives_days_per_year(where):
    """time_groups="year": the weighted days per year in each bin == the yearly sums of the daily oracle."""
    lat, lon, df, tas = _config(1.0, 3000, 365)
    t = pd.date_range("2001-07-01", periods=365)                 # two calendar years
    data = _put(tas, "device") if where == "device" else tas
    ds = Dataset({"tas": (("time", "lat", "lon"), data)}, coords={"time": t, "lat": lat, "lon": lon})
    edges = [-INF, 5.0, 10.0, 15.0, 20.0, 25.0, INF]            # 6 bins: launches of 4 and 2
    ds1 = tas_bins(ds, edges, "b")
    names = list(ds1.data_vars)
    out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df, time_groups="year")
    years = ds1.time.values // 1000
    total = 0.0
    for name, lo, hi in zip(names, edges[:-1], edges[1:]):
        xt, _ = tas_bins_ref(tas, t, lo, hi)
        ref, rd, _ = _oracle_agg(xt, ("time", "lat", "lon"), lat, lon, df, "popwt", "hierid")
        ref_y, yl = oracle.time_group_sum(ref, rd, years)
        assert out[name].dims == rd and list(out.time.values) == list(yl) == [2001, 2002]
        assert out[name].attrs["units"] == "days"
        _check(out[name].values, ref_y, 1e-9)
        total = total + out[name].values
    assert np.nanmax(total) <= 365 and np.nanmax(total) > 180     # days per year


@pytest.mark.gpu
def test_season_mask_gates_the_bins():
    """season_mask=: only gridcell-days inside their growing season count, == the oracle aggregate of
    bins x the dense growing-season mask."""
    from climate_toolbox_b200.utils.utils import get_daily_growing_season_mask
    rng = np.random.default_rng(21)
    T = 120
    lat, lon, df, tas = _config(1.0, 3000, T)
    t = pd.date_range("2003-01-01", periods=T)                  # YYYYDDD positions == days of year
    nlat, nlon = len(lat), len(lon)
    plant = rng.integers(1, 366, (nlat, nlon)).astype(np.float64)
    harv = rng.integers(1, 366, (nlat, nlon)).astype(np.float64)
    harv[rng.random((nlat, nlon)) < 0.05] = np.nan
    plant[rng.random((nlat, nlon)) < 0.05] = np.nan
    gd = Dataset({"variable": (("z", "latitude", "longitude"), np.stack([plant, harv]))},
                 coords={"z": np.array([1, 2]), "latitude": lat, "longitude": lon + 180})
    ds = Dataset({"tas": (("time", "lat", "lon"), _put(tas, "device"))}, coords={"time": t, "lat": lat, "lon": lon})
    edges = [-INF, 10.0, 20.0, INF]
    ds1 = tas_bins(ds, edges, "b")
    names = list(ds1.data_vars)
    m = get_daily_growing_season_mask(ds1["lat"], ds1["lon"], ds1["time"], gd)
    out = weighted_aggregate_grid_to_regions(ds1, names, "cropwt", "hierid", weights=df, season_mask=m)
    plain = weighted_aggregate_grid_to_regions(ds1, names, "cropwt", "hierid", weights=df)
    dense = oracle.growing_season_mask(plant, harv, t.dayofyear.values).transpose(2, 0, 1)
    for name, lo, hi in zip(names, edges[:-1], edges[1:]):
        ref, rd, _ = _oracle_agg(bins_ref(tas, lo, hi) * dense, ("time", "lat", "lon"), lat, lon, df,
                                 "cropwt", "hierid")
        assert out[name].dims == rd
        _check(out[name].values, ref, 1e-9)
        assert not np.allclose(np.nan_to_num(plain[name].values), np.nan_to_num(out[name].values))
