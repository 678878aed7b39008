"""Degree days and time per temperature bin from the steps of sub-daily data (``transformations.subdaily_edd`` /
``subdaily_gdd`` / ``subdaily_bins``, ``ctb_pull_pack_daily_steps``), computed while the referenced gridcells are
packed for aggregation.

``steps_ref`` restates the rules in numpy (an explicit float64 loop over the steps of a day, NaN steps skipped);
its daily arrays feed the restated reference aggregation of ``oracle``, which is unchanged.
CPU: known answers of the restatement, time-axis / threshold / edge validation, attributes, request fusion, and
the C-ABI's checks that need no plan.
GPU: ``.values`` bit-exact with the restatement; aggregates against the oracle and against the existing identity
path on the materialised daily planes; one reduce-pack for four thresholds; one read of a pinned source."""
import ctypes

import numpy as np
import pandas as pd
import pytest

import oracle
from climate_toolbox_b200 import Dataset
from climate_toolbox_b200 import _engine as E
from climate_toolbox_b200 import _native as N
from climate_toolbox_b200.aggregations.aggregations import (_group_requests, _resolve,
                                                            weighted_aggregate_grid_to_regions,
                                                            weighted_aggregate_grid_to_regions_multi)
from climate_toolbox_b200.transformations.transformations import subdaily_bins, subdaily_edd, subdaily_gdd
from climate_toolbox_b200.utils.utils import remove_leap_days, resample_daily
from test_subdaily import (DIMS, N_DAYS, _check_pair, _days, _dev, _ds, _oracle_agg, _same, _subdaily, _tiny,
                           _times, lib)  # noqa: F401  (lib: the build fixture)

EDD = (290.0, 295.5, 300.0, 283.15)
GDD = ((283.15, 303.15), (290.0, 300.0))
EDGES = (-np.inf, 280.0, 290.0, 295.5, 300.0, np.inf)


# ----------------------------------------------------------------------------
# the reference rules
# ----------------------------------------------------------------------------
def steps_ref(x, S, op, params):
    """Daily means of a per-step transform of ``x`` [days * S, ...] -> list of float64 arrays, one per output.
    Every step widened to float64; NaN steps skipped; f summed in step order, divided by the count of non-NaN
    steps (NaN without one).  ``op``: "edd" (params: thresholds), "gdd" (params: (lo, hi) pairs) or "bins"
    (params: edges)."""
    x = np.asarray(x)
    xs = x.reshape((x.shape[0] // S, S) + x.shape[1:])
    if op == "edd":
        fs = [lambda v, e=e: np.maximum(v - e, 0.0) for e in params]
    elif op == "gdd":
        fs = [lambda v, lo=lo, w=np.float64(hi) - np.float64(lo): np.minimum(np.maximum(v - lo, 0.0), w)
              for lo, hi in params]
    else:
        fs = [lambda v, lo=lo, hi=hi: ((v >= lo) & (v < hi)).astype(np.float64)
              for lo, hi in zip(params[:-1], params[1:])]
    out = []
    with np.errstate(invalid="ignore"):
        for f in fs:
            s = np.zeros(xs[:, 0].shape, dtype=np.float64)
            c = np.zeros(xs[:, 0].shape, dtype=np.int64)
            for h in range(S):
                v = xs[:, h].astype(np.float64)
                ok = ~np.isnan(v)
                s = np.where(ok, s + f(v), s)
                c += ok
            out.append(s / c)
    return out


def test_reference_known_answers():
    inf, nan = np.inf, np.nan
    # days of 3 steps: NaN steps, an all-NaN day, +-inf, values on the thresholds and edges
    x = np.array([[1.0], [nan], [4.0], [nan], [nan], [nan], [inf], [-inf], [2.0], [2.0], [3.0], [5.0]])
    e2, e3 = steps_ref(x, 3, "edd", (2.0, 3.0))
    np.testing.assert_array_equal(e2[:, 0], [1.0, nan, inf, 4.0 / 3.0])
    np.testing.assert_array_equal(e3[:, 0], [0.5, nan, inf, 2.0 / 3.0])
    g, = steps_ref(x, 3, "gdd", ((2.0, 4.0),))
    np.testing.assert_array_equal(g[:, 0], [1.0, nan, 2.0 / 3.0, 1.0])               # +inf gives hi - lo
    b = steps_ref(x, 3, "bins", (-inf, 2.0, 3.0, inf))
    np.testing.assert_array_equal(np.stack(b)[:, :, 0],
                                  [[0.5, nan, 1.0 / 3.0, 0.0],      # -inf lies in the first bin
                                   [0.0, nan, 1.0 / 3.0, 1.0 / 3.0],    # 2 lies in [2, 3)
                                   [0.5, nan, 0.0, 2.0 / 3.0]])     # +inf lies in no bin
    f = np.array([[16777216.0], [1.0], [1.0]], dtype=np.float32)          # widened before the subtraction
    assert steps_ref(f, 3, "edd", (0.5,))[0][0, 0] == (16777215.5 + 0.5 + 0.5) / 3


# ----------------------------------------------------------------------------
# CPU: validation, attributes, fusion
# ----------------------------------------------------------------------------
def _tas(time, units="K"):
    ds = _tiny(time)
    if units:
        ds._vars["tas"].attrs["units"] = units
    return ds.tas


@pytest.mark.parametrize("case", ["missing_hour", "ragged_day", "unordered_steps", "missing_day", "not_datetime"])
def test_time_axis_validation(case):
    t = _times(24, n_days=3)
    if case == "missing_hour":
        t = np.delete(t, 30)
    elif case == "ragged_day":
        t = np.sort(np.r_[t, t[30] + np.timedelta64(30, "m")])
    elif case == "unordered_steps":
        t = t.reshape(3, 24)[:, ::-1].ravel()
    elif case == "missing_day":
        t = np.r_[t[:24], t[48:]]
    else:
        t = np.arange(72)
    for f in (lambda a: subdaily_edd(a, 300.0), lambda a: subdaily_gdd(a, 280.0, 300.0),
              lambda a: subdaily_bins(a, [280.0, 300.0])):
        with pytest.raises(ValueError):
            f(_tas(t))


def test_threshold_and_edge_validation():
    a = _tas(_times(4, 2))
    for e in (np.inf, -np.inf, np.nan):
        with pytest.raises(ValueError):
            subdaily_edd(a, e)
    for lo, hi in ((300.0, 300.0), (301.0, 300.0), (-np.inf, 300.0), (280.0, np.inf), (np.nan, 300.0)):
        with pytest.raises(ValueError):
            subdaily_gdd(a, lo, hi)
    for edges in ([280.0], [290.0, 280.0], [280.0, np.nan], [280.0, -np.inf], [np.inf, 300.0],
                  [280.0, np.inf, 300.0]):
        with pytest.raises(ValueError):
            subdaily_bins(a, edges)
    with pytest.raises(ValueError):
        subdaily_bins(a, [280.0, 290.0, 300.0], ["one"])
    b = _tas(_times(4, 2), units=None)
    for f in (lambda: subdaily_edd(b, 300.0), lambda: subdaily_gdd(b, 280.0, 300.0),
              lambda: subdaily_bins(b, [280.0, 300.0])):
        with pytest.raises(AttributeError):
            f()
    with pytest.raises(NotImplementedError):
        ds = _tiny(_times(4, 2), ("lat", "lon", "time"))
        ds._vars["tas"].attrs["units"] = "K"
        subdaily_edd(ds.tas, 300.0)


def test_attributes():
    a = _tas(_times(24, 3))
    e = subdaily_edd(a, 300)
    assert e.dims == ("time", "lat", "lon") and e.shape == (3, 2, 2) and e.dtype == np.float64
    assert e.attrs == {"units": "degreedays_300K"} == {"units": oracle.snyder_edd_units(300, "K")}
    assert e.time.values.dtype == np.dtype("datetime64[D]")
    np.testing.assert_array_equal(e.time.values, _days(3))
    g = subdaily_gdd(a, 283.15, 303.15)
    assert g.attrs["units"] == "degreedays_283.15-303.15K" == oracle.snyder_gdd_units(283.15, 303.15, "K")
    assert g.dtype == np.float64 and g.shape == (3, 2, 2)
    b = subdaily_bins(a, [-np.inf, 280.0, np.inf], "b")
    assert list(b.data_vars) == ["b_0", "b_1"]
    assert b.b_0.attrs["units"] == "days" and b.b_0.attrs["bin_lower"] == -np.inf
    assert (b.b_1.attrs["bin_lower"], b.b_1.attrs["bin_upper"]) == (280.0, np.inf)
    assert b.b_1.dtype == np.float64 and b.b_1.shape == (3, 2, 2)
    np.testing.assert_array_equal(b.time.values, _days(3))
    assert list(subdaily_bins(a, [1.0, 2.0, 3.0], ["lo", "hi"]).data_vars) == ["lo", "hi"]
    assert remove_leap_days(Dataset({"e": subdaily_edd(_tas(_times(4, 5, "2004-02-27")), 1.0)},
                                    coords={"time": _days(5, "2004-02-27")})).e.shape == (4, 2, 2)


def _reqs(named):
    return [(n,) + _resolve(v.variable) for n, v in named]


def test_fusion_rules():
    t = _times(8, n_days=2)
    ds = _tiny(t)
    ds["tas2"] = (("time", "lat", "lon"), np.ones((16, 2, 2), dtype=np.float32))
    for v in ("tas", "tas2"):
        ds._vars[v].attrs["units"] = "K"
    edd = [("e{}".format(k), subdaily_edd(ds.tas, 280.0 + k)) for k in range(5)]
    g = _group_requests(_reqs(edd))
    assert [x["names"] for x in g] == [["e0", "e1", "e2", "e3"], ["e4"]]           # at most 4 per read
    gdd = [("g{}".format(k), subdaily_gdd(ds.tas, 280.0 + k, 300.0)) for k in range(2)]
    g = _group_requests(_reqs(edd[:2] + gdd + edd[2:3]))
    assert [x["names"] for x in g] == [["e0", "e1", "e2"], ["g0", "g1"]]           # families never mix
    bins = subdaily_bins(ds.tas, [270.0, 280.0, 290.0, 300.0], "b")
    g = _group_requests(_reqs([(n, bins[n]) for n in ("b_0", "b_1", "b_2")]))
    assert [x["names"] for x in g] == [["b_0", "b_1", "b_2"]]
    g = _group_requests(_reqs([(n, bins[n]) for n in ("b_0", "b_2", "b_1")]))     # b_2 does not continue b_0
    assert [x["names"] for x in g] == [["b_0", "b_1"], ["b_2"]]
    # the same read only: another variable, other days, another source start
    other = [("x", subdaily_edd(ds.tas2, 281.0)),
             ("y", subdaily_edd(ds.tas, 282.0).isel(time=[1, 0])),
             ("z", subdaily_edd(ds.isel(time=np.arange(8, 16)).tas, 283.0))]
    g = _group_requests(_reqs(edd[:1] + other))
    assert [x["names"] for x in g] == [["e0"], ["x"], ["y"], ["z"]]
    # daily means, minima and maxima keep their grouping: identity requests never fuse
    mean = resample_daily(ds, "mean")
    g = _group_requests(_reqs([("m", mean.tas), ("e0", edd[0][1]), ("m2", mean.tas)]))
    assert [x["names"] for x in g] == [["m"], ["e0"], ["m2"]]


def test_abi_rejects_null_plan(lib):
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    prm = (ctypes.c_double * 1)(300.0)
    dst = (ctypes.c_void_p * 1)(p)
    assert lib.ctb_pull_pack_daily_steps(None, p, N.F32, 1024, 24, None, 0, 4, N.STEP_EDD, prm, 1, 1, dst,
                                         None) == N.ERR_INVALID
    assert "compact plan" in N.last_error()
    assert lib.ctb_pull_pack_daily_steps(None, None, N.F32, 1024, 24, None, 0, 4, N.STEP_EDD, prm, 1, 1, dst,
                                         None) == N.ERR_INVALID


# ----------------------------------------------------------------------------
# GPU: values
# ----------------------------------------------------------------------------
def _on_thresholds(x, S, n_days, nlat, nlon):
    """Put steps exactly on thresholds and edges (all representable in float32)."""
    xs = x.reshape(n_days, S, nlat, nlon)
    rng = np.random.default_rng(7)
    for v in (290.0, 295.5, 300.0, 280.0):
        for _ in range(30):
            xs[rng.integers(n_days), rng.integers(S), rng.integers(nlat), rng.integers(nlon)] = v


def _results(src):
    """{op: [deferred daily DataArrays]} for the EDD thresholds, GDD pairs and bins."""
    b = subdaily_bins(src, EDGES, "b")
    return {"edd": [subdaily_edd(src, e) for e in EDD], "gdd": [subdaily_gdd(src, *p) for p in GDD],
            "bins": [b[n] for n in b.data_vars]}


PARAMS = {"edd": EDD, "gdd": GDD, "bins": EDGES}


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned", "pageable"])
@pytest.mark.parametrize("S", [24, 8, 4])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_values_bit_exact(dtype, S, where):
    lat, lon, _, x = _subdaily(S, dtype, n_days=12)
    _on_thresholds(x, S, 12, len(lat), len(lon))
    ds = _ds(x, lat, lon, S, where, n_days=12)
    ds._vars["tas"].attrs["units"] = "K"
    sub_ds = ds.isel(time=np.arange(2 * S, 7 * S))            # a source that starts within the physical steps
    for op, das in _results(ds.tas).items():
        refs = steps_ref(x, S, op, PARAMS[op])
        for da, ref in zip(das, refs):
            _same(da.values, ref)
            # lazy takes: lat / lon of the source, days of the result
            sub = da.isel(lat=np.arange(3, 17), lon=np.arange(40, 0, -3)).isel(time=[0, 5, 5, 11])
            _same(sub.values, ref[[0, 5, 5, 11]][:, 3:17][:, :, np.arange(40, 0, -3)])
        _same(_results(sub_ds.tas)[op][0].values, steps_ref(x[2 * S: 7 * S], S, op, PARAMS[op])[0])


# ----------------------------------------------------------------------------
# GPU: aggregates
# ----------------------------------------------------------------------------
CASES = ["plain", "year", "season", "leap", "multi"]
S_OF = {"plain": 24, "year": 8, "season": 4, "leap": 24, "multi": 8}


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("case", CASES)
def test_aggregates(case, dtype, where):
    S = S_OF[case]
    lat, lon, df, x = _subdaily(S, dtype)
    _on_thresholds(x, S, N_DAYS, len(lat), len(lon))
    ds = _ds(x, lat, lon, S, where)
    ds._vars["tas"].attrs["units"] = "K"
    days = _days()
    agg = weighted_aggregate_grid_to_regions
    for op, das in _results(ds.tas).items():
        refs = steps_ref(x, S, op, PARAMS[op])
        names = ["v{}".format(k) for k in range(len(das))]
        sub_ds = Dataset(dict(zip(names, das)), coords=das[0]._coords)
        mat = Dataset({n: (DIMS, _dev(r)) for n, r in zip(names, refs)}, coords={"time": days, "lat": lat, "lon": lon})
        if case == "plain":
            got, want = agg(sub_ds, names, "popwt", "hierid", weights=df), agg(mat, names, "popwt", "hierid", weights=df)
            for n, r in zip(names, refs):
                ref, _, labels = _oracle_agg(r, lat, lon, df)
                _check_pair(got[n].values, want[n].values, ref, _oracle_agg(np.abs(r), lat, lon, df)[0], df, "hierid",
                            labels)
        elif case == "year":
            got = agg(sub_ds, names, "popwt", "hierid", weights=df, time_groups="year")
            want = agg(mat, names, "popwt", "hierid", weights=df, time_groups="year")
            years = days.astype("datetime64[Y]").astype(np.int64) + 1970
            assert list(got.time.values) == [2003, 2004]
            for n, r in zip(names, refs):
                ref, rd, labels = _oracle_agg(r, lat, lon, df)
                scale = _oracle_agg(np.abs(r), lat, lon, df)[0]
                ref_y, _ = oracle.time_group_sum(ref, rd, years)
                scale_y, _ = oracle.time_group_sum(scale, rd, years)
                _check_pair(got[n].values, want[n].values, ref_y, scale_y, df, "hierid", labels, days=N_DAYS)
        elif case == "season":
            from climate_toolbox_b200.utils.utils import get_daily_growing_season_mask
            rng = np.random.default_rng(21)
            nlat, nlon = len(lat), len(lon)
            plant = rng.integers(1, 366, (nlat, nlon)).astype(np.float64)
            harv = rng.integers(1, 366, (nlat, nlon)).astype(np.float64)
            gd = Dataset({"variable": (("z", "latitude", "longitude"), np.stack([plant, harv]))},
                         coords={"z": np.array([1, 2]), "latitude": lat, "longitude": lon + 180})
            m = get_daily_growing_season_mask(lat, lon, days, gd)
            got = agg(sub_ds, names, "cropwt", "hierid", weights=df, season_mask=m)
            want = agg(mat, names, "cropwt", "hierid", weights=df, season_mask=m)
            dense = oracle.growing_season_mask(plant, harv, pd.DatetimeIndex(days).dayofyear.values).transpose(2, 0, 1)
            for n, r in zip(names, refs):
                with np.errstate(invalid="ignore"):          # inf x 0 outside the season: NaN, skipped
                    ref, _, labels = _oracle_agg(r * dense, lat, lon, df, "cropwt")
                    scale = _oracle_agg(np.abs(r) * dense, lat, lon, df, "cropwt")[0]
                _check_pair(got[n].values, want[n].values, ref, scale, df, "hierid", labels)
        elif case == "leap":
            keep = oracle.leap_day_keep_mask(days)
            got = agg(remove_leap_days(sub_ds), names, "popwt", "hierid", weights=df)
            want = agg(remove_leap_days(mat), names, "popwt", "hierid", weights=df)
            assert got.time.values.size == N_DAYS - 1
            np.testing.assert_array_equal(got.time.values, days[keep])
            for n, r in zip(names, refs):
                ref, _, labels = _oracle_agg(r[keep], lat, lon, df)
                scale = _oracle_agg(np.abs(r[keep]), lat, lon, df)[0]
                _check_pair(got[n].values, want[n].values, ref, scale, df, "hierid", labels)
        else:
            wts = ["popwt", "areawt"]
            got = weighted_aggregate_grid_to_regions_multi(sub_ds, names[1], wts, "hierid", df)
            want = weighted_aggregate_grid_to_regions_multi(mat, names[1], wts, "hierid", df)
            for wt in wts:
                ref, _, labels = _oracle_agg(refs[1], lat, lon, df, wt)
                scale = _oracle_agg(np.abs(refs[1]), lat, lon, df, wt)[0]
                name = "{}_{}".format(names[1], wt)
                _check_pair(got[name].values, want[name].values, ref, scale, df, "hierid", labels)


@pytest.mark.gpu
def test_four_thresholds_one_reduce_pack():
    """4 EDD thresholds of one device source: one reduce-pack, then one identity aggregation per plane."""
    S = 24
    lat, lon, df, x = _subdaily(S, np.float32, n_days=20)
    ds = _ds(x, lat, lon, S, "device", n_days=20)
    ds._vars["tas"].attrs["units"] = "K"
    names = ["e{}".format(k) for k in range(4)]
    das = [subdaily_edd(ds.tas, e) for e in EDD]
    d = Dataset(dict(zip(names, das)), coords=das[0]._coords)
    weighted_aggregate_grid_to_regions(d, names, "popwt", "hierid", weights=df)       # builds the plan
    n0 = E.launch_count()
    out = weighted_aggregate_grid_to_regions(d, names, "popwt", "hierid", weights=df)
    assert E.launch_count() - n0 == 1 + 4
    for n in names:                     # each plane in its own output, as one threshold at a time gives
        one = weighted_aggregate_grid_to_regions(Dataset({n: d[n]}, coords=d._coords), n, "popwt", "hierid",
                                                 weights=df)
        np.testing.assert_array_equal(out[n].values, one[n].values)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_pinned_source_read_once(dtype):
    """4 thresholds of one pinned source: one pass over the referenced pieces x steps crosses PCIe."""
    S, n_days = 24, 30
    lat, lon, df, x = _subdaily(S, dtype, n_days=n_days, specials=False)
    ds = _ds(x, lat, lon, S, "pinned", n_days=n_days)
    ds._vars["tas"].attrs["units"] = "K"
    b = subdaily_bins(ds.tas, EDGES[:5], "b")
    before = E.TRANSFER_BYTES["h2d"]
    weighted_aggregate_grid_to_regions(b, list(b.data_vars), "popwt", "hierid", weights=df)
    moved = E.TRANSFER_BYTES["h2d"] - before
    es = np.dtype(dtype).itemsize
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", stage_bytes=8, compact=True, elem_bytes=8)
    assert moved == n_days * S * plan.info["n_pieces_distinct"] * 4 * es


@pytest.mark.gpu
def test_abi_checks_with_a_plan(lib):
    import torch
    from climate_toolbox_b200 import synthetic
    lat, lon = synthetic.grid_labels(3.0)
    df = synthetic.weights_table(3.0, 50, seed=5)
    g = E.GridSpec(lat, lon)
    full = E.get_plan(g, df, "popwt", "hierid", cache=False)
    p4 = E.get_plan(g, df, "popwt", "hierid", compact=True, elem_bytes=4, cache=False)
    p8 = E.get_plan(g, df, "popwt", "hierid", compact=True, elem_bytes=8, cache=False)
    ncell = len(lat) * len(lon)
    x = torch.zeros((4 * 24, ncell), dtype=torch.float32, device="cuda")
    planes = [torch.zeros((4, p8.info["n_packed_cells"]), dtype=torch.float64, device="cuda") for _ in range(4)]
    L = lib

    def call(plan, op=N.STEP_EDD, params=(290.0,), n_out=1, n_params=None, dst="ok", S=24, xp=None):
        prm = (ctypes.c_double * max(1, len(params)))(*params)
        if dst == "ok":
            d = (ctypes.c_void_p * n_out)(*[p.data_ptr() for p in planes[:n_out]])
        elif dst == "hole":
            d = (ctypes.c_void_p * n_out)(*([planes[0].data_ptr()] + [None] * (n_out - 1)))
        elif dst == "odd":
            d = (ctypes.c_void_p * n_out)(planes[0].data_ptr() + 8)
        else:
            d = None
        return L.ctb_pull_pack_daily_steps(plan._h, xp or x.data_ptr(), N.F32, ncell, S, None, 0, 4, op, prm,
                                           len(params) if n_params is None else n_params, n_out, d, None)

    assert call(full) == N.ERR_INVALID and "compact" in N.last_error()
    assert call(p4) == N.ERR_INVALID and "float64" in N.last_error()
    assert call(p8, S=0) == N.ERR_INVALID and "steps_per_day" in N.last_error()
    for op in (0, 4):
        assert call(p8, op=op) == N.ERR_INVALID and "step_op" in N.last_error()
    assert call(p8, n_out=0, params=()) == N.ERR_INVALID
    assert call(p8, n_out=5, params=(1.0, 2.0, 3.0, 4.0, 5.0), dst=None) == N.ERR_INVALID
    assert call(p8, params=(290.0, 300.0)) == N.ERR_INVALID                       # n_params does not match n_out
    assert call(p8, op=N.STEP_GDD, params=(290.0,)) == N.ERR_INVALID
    assert call(p8, op=N.STEP_BINS, params=(290.0,)) == N.ERR_INVALID
    for bad in (np.nan, np.inf, -np.inf):
        assert call(p8, params=(bad,)) == N.ERR_INVALID
        assert call(p8, op=N.STEP_GDD, params=(bad, 300.0)) == N.ERR_INVALID
    assert call(p8, op=N.STEP_GDD, params=(300.0, 300.0)) == N.ERR_INVALID
    assert call(p8, op=N.STEP_GDD, params=(290.0, 300.0, 310.0, 305.0), n_out=2) == N.ERR_INVALID
    for edges in ((300.0, 290.0), (290.0, np.nan), (np.inf, 300.0), (290.0, -np.inf)):
        assert call(p8, op=N.STEP_BINS, params=edges) == N.ERR_INVALID
    assert call(p8, dst=None) == N.ERR_INVALID
    assert call(p8, op=N.STEP_EDD, params=(290.0, 300.0), n_out=2, dst="hole") == N.ERR_INVALID
    assert call(p8, dst="odd") == N.ERR_UNSUPPORTED
    assert call(p8, xp=x.data_ptr() + 4) == N.ERR_UNSUPPORTED
    assert call(p8, op=N.STEP_BINS, params=(-np.inf, 290.0, 300.0, np.inf, ), n_out=3) == N.OK
    assert call(p8, op=N.STEP_GDD, params=(280.0, 290.0, 290.0, 300.0), n_out=2) == N.OK
    assert call(p8, params=(1.0, 2.0, 3.0, 4.0), n_out=4) == N.OK
    torch.cuda.synchronize()
    for p in (full, p4, p8):
        p.close()
