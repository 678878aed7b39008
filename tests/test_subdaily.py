"""Daily mean / min / max of sub-daily data (``utils.resample_daily``, ``ctb_pull_pack_daily``), reduced while
the referenced gridcells are packed for aggregation.

``resample_daily_ref`` restates the reduction in numpy (an explicit float64 loop over the steps of a day, NaN
steps skipped); its daily arrays feed the restated reference aggregation of ``oracle``, which is unchanged.
CPU: time-axis and ``how`` validation, the C-ABI's argument checks that need no plan, and request grouping.
GPU: ``.values`` bit-exact with the reference; aggregates against the oracle on the restated daily arrays and
against the existing path on the materialised daily arrays; one read of the source for Snyder's min and max."""
import ctypes

import numpy as np
import pandas as pd
import pytest

import oracle
from conftest import rel_err
from climate_toolbox_b200 import Dataset
from climate_toolbox_b200 import _engine as E
from climate_toolbox_b200 import _native as N
from climate_toolbox_b200 import synthetic
from climate_toolbox_b200.aggregations.aggregations import (_group_requests, _resolve,
                                                            weighted_aggregate_grid_to_regions,
                                                            weighted_aggregate_grid_to_regions_multi)
from climate_toolbox_b200.transformations.transformations import (snyder_edd, snyder_gdd, tas_bins, tas_poly,
                                                                  tas_rcspline)
from climate_toolbox_b200.utils.utils import remove_leap_days, resample_daily
from test_bins import bins_ref
from test_rcspline import rcs_ref, rcs_scale

OFF = 273.15
TOL = 1e-9                 # tests/test_gpu_parity.py: |got - ref| <= 1e-9 max(|ref|, S)
START = "2003-12-15"       # 78 days: a year end and 29 February 2004
N_DAYS = 78


# ----------------------------------------------------------------------------
# the reference reduction
# ----------------------------------------------------------------------------
def resample_daily_ref(x, S, how):
    """Daily ``how`` of ``x`` [days * S, ...]: mean -- every step widened to float64 and added in step order,
    NaN steps skipped, divided by the count of non-NaN steps (NaN without one); min / max -- NaN steps
    skipped, NaN without a value, in the dtype of ``x``."""
    x = np.asarray(x)
    xs = x.reshape((x.shape[0] // S, S) + x.shape[1:])
    if how == "mean":
        s = np.zeros(xs[:, 0].shape, dtype=np.float64)
        c = np.zeros(xs[:, 0].shape, dtype=np.int64)
        with np.errstate(invalid="ignore"):
            for h in range(S):
                v = xs[:, h].astype(np.float64)
                ok = ~np.isnan(v)
                s = np.where(ok, s + v, s)
                c += ok
            return s / c
    f = np.fmin if how == "min" else np.fmax
    out = np.full(xs[:, 0].shape, np.nan, dtype=x.dtype)
    for h in range(S):
        out = f(out, xs[:, h])
    return out


def test_reference_reduction_known_answers():
    x = np.array([[1.0], [np.nan], [2.0], [np.nan], [np.nan], [np.nan], [np.inf], [-np.inf], [np.inf], [3.0],
                  [-1.0], [5.0]])
    np.testing.assert_array_equal(resample_daily_ref(x, 3, "mean")[:, 0], [1.5, np.nan, np.nan, 7.0 / 3.0])
    np.testing.assert_array_equal(resample_daily_ref(x, 3, "min")[:, 0], [1.0, np.nan, -np.inf, -1.0])
    np.testing.assert_array_equal(resample_daily_ref(x, 3, "max")[:, 0], [2.0, np.nan, np.inf, 5.0])
    f = np.array([[16777216.0], [1.0], [1.0]], dtype=np.float32)        # widened before the adds
    assert resample_daily_ref(f, 3, "mean")[0, 0] == (16777216.0 + 2.0) / 3


# ----------------------------------------------------------------------------
# fixtures
# ----------------------------------------------------------------------------
def _times(S, n_days=N_DAYS, start=START):
    return pd.date_range(start, periods=n_days * S, freq="{}min".format(24 * 60 // S)).values


def _subdaily(S, dtype, n_days=N_DAYS, d=3.0, R=400, specials=True, seed=3):
    """(lat, lon, weights, x [days * S, lat, lon]) with NaN hours, all-NaN days, +-inf and inf / -inf in one
    day at some gridcells."""
    lat, lon = synthetic.grid_labels(d)
    df = synthetic.weights_table(d, R, seed=5)
    x, _, _ = synthetic.tas_field(n_days * S, len(lat), len(lon), seed=seed, nan_frac=0.01, dtype=dtype)
    rng = np.random.default_rng(seed)
    nlat, nlon = len(lat), len(lon)
    xs = x.reshape(n_days, S, nlat, nlon)
    for _ in range(40):                                                  # all-NaN days
        xs[rng.integers(n_days), :, rng.integers(nlat), rng.integers(nlon)] = np.nan
    if specials:
        for v in (np.inf, -np.inf):
            for _ in range(10):
                xs[rng.integers(n_days), rng.integers(S), rng.integers(nlat), rng.integers(nlon)] = v
        for _ in range(10):                                              # inf and -inf in one day
            dd, i, j = rng.integers(n_days), rng.integers(nlat), rng.integers(nlon)
            xs[dd, 0, i, j], xs[dd, S - 1, i, j] = np.inf, -np.inf
    return lat, lon, df, x


def _put(a, where):
    import torch
    if where == "device":
        return torch.from_numpy(a).cuda()
    if where == "pageable":
        return a
    host = torch.empty(a.shape, dtype=torch.float32 if a.dtype == np.float32 else torch.float64, pin_memory=True)
    host.copy_(torch.from_numpy(a))
    return host.numpy()


def _ds(x, lat, lon, S, where, n_days=N_DAYS, start=START):
    return Dataset({"tas": (("time", "lat", "lon"), _put(x, where))},
                   coords={"time": _times(S, n_days, start), "lat": lat, "lon": lon})


def _days(n_days=N_DAYS, start=START):
    return pd.date_range(start, periods=n_days, freq="D").values.astype("datetime64[D]")


# ----------------------------------------------------------------------------
# CPU: validation
# ----------------------------------------------------------------------------
def _tiny(time, dims=("time", "lat", "lon")):
    shape = {"time": len(time), "lat": 2, "lon": 2}
    x = np.zeros([shape[d] for d in dims], dtype=np.float32)
    return Dataset({"tas": (dims, x)}, coords={"time": time, "lat": [0.0, 1.0], "lon": [0.0, 1.0]})


def test_resample_daily_metadata():
    t = _times(24, n_days=3)
    ds = _tiny(t)
    ds._vars["tas"].attrs["units"] = "K"
    for how in ("mean", "min", "max"):
        r = resample_daily(ds, how)
        assert r.tas.dims == ("time", "lat", "lon") and r.tas.shape == (3, 2, 2)
        assert r.tas.attrs == {"units": "K", "cell_methods": "time: {}".format(how)}
        assert r.time.values.dtype == np.dtype("datetime64[D]")
        np.testing.assert_array_equal(r.time.values, _days(3))
        assert r.tas.dtype == (np.float64 if how == "mean" else np.float32)
    da = resample_daily(ds.tas, "max")
    assert da.shape == (3, 2, 2) and da.attrs["cell_methods"] == "time: max"
    assert remove_leap_days(resample_daily(_tiny(_times(4, 5, "2004-02-27")), "mean")).tas.shape == (4, 2, 2)


@pytest.mark.parametrize("case", ["missing_hour", "ragged_day", "unordered_steps", "other_steps", "missing_day",
                                  "not_datetime"])
def test_time_axis_validation(case):
    t = _times(24, n_days=3)
    if case == "missing_hour":
        t = np.delete(t, 30)
    elif case == "ragged_day":
        t = np.sort(np.r_[t, t[30] + np.timedelta64(30, "m")])
    elif case == "unordered_steps":
        t = t.reshape(3, 24)[:, ::-1].ravel()
    elif case == "other_steps":
        t = t.copy()
        t[30] += np.timedelta64(30, "m")
    elif case == "missing_day":
        t = np.r_[t[:24], t[48:]]
    else:
        t = np.arange(72)
    with pytest.raises(ValueError):
        resample_daily(_tiny(t), "mean")


def test_cell_major_and_how():
    with pytest.raises(NotImplementedError):
        resample_daily(_tiny(_times(4, 2), ("lat", "lon", "time")), "mean")
    for how in ("sum", "median", None):
        with pytest.raises(ValueError):
            resample_daily(_tiny(_times(4, 2)), how)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as G
    G.build()
    return N.lib()


def _daily_call(L, plan=None, x=None, S=24, ops=N.DAILY_MEAN, mean=None, mn=None, mx=None, dtype=N.F32):
    return L.ctb_pull_pack_daily(plan, x, dtype, 1024, S, None, 0, 4, ops, mean, mn, mx, None)


def test_abi_rejects_null_plan_and_buffers(lib):
    buf = ctypes.create_string_buffer(64)
    p = ctypes.addressof(buf)
    assert _daily_call(lib, None, p, mean=p) == N.ERR_INVALID
    assert "compact plan" in N.last_error()
    assert _daily_call(lib, None, None, mean=p) == N.ERR_INVALID


def _snyder_reqs(pairs):
    reqs = []
    for k, (tn, tx, thr) in enumerate(pairs):
        da = snyder_edd(tn, tx, thr, check=False)
        reqs.append(("e{}".format(k),) + _resolve(da.variable))
    return reqs


def test_grouping_min_max_of_one_source():
    t = _times(8, n_days=2)
    ds = _tiny(t)
    ds["tasmax"] = (("time", "lat", "lon"), np.ones((16, 2, 2), dtype=np.float32))
    for v in ("tas", "tasmax"):
        ds._vars[v].attrs["units"] = "K"
    lo, hi, mean = resample_daily(ds, "min"), resample_daily(ds, "max"), resample_daily(ds, "mean")
    # the default check is skipped: a daily maximum is never below the minimum of the same steps
    e = snyder_edd(lo.tas, hi.tas, 300.0)
    assert [s.deferred.params[0] for s in e.variable.deferred.sources] == ["min", "max"]
    g = _group_requests(_snyder_reqs([(lo.tas, hi.tas, 290.0), (lo.tas, hi.tas, 300.0)]))
    assert len(g) == 1 and g[0]["names"] == ["e0", "e1"]
    for other in ((lo.tasmax, hi.tas), (lo.tas, hi.tasmax), (mean.tas, hi.tas),
                  (lo.isel(time=[1, 0]).tas, hi.tas)):
        g = _group_requests(_snyder_reqs([(lo.tas, hi.tas, 290.0), other + (300.0,)]))
        assert len(g) == 2
    # identity requests of daily reductions never fuse; poly orders of one daily mean do
    assert len(_group_requests([("a",) + _resolve(lo.tas.variable), ("b",) + _resolve(hi.tas.variable)])) == 2
    p = tas_poly(mean, [1, 2], ["p1", "p2"])
    assert len(_group_requests([(n,) + _resolve(p._vars[n]) for n in ("p1", "p2")])) == 1


# ----------------------------------------------------------------------------
# GPU: values
# ----------------------------------------------------------------------------
def _same(got, ref):
    """Bit-exact but for the sign of zero (+-0 ties of min / max compare equal)."""
    assert got.dtype == ref.dtype and got.shape == ref.shape
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan)
    assert (got[~nan] == ref[~nan]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned", "pageable"])
@pytest.mark.parametrize("S", [24, 8, 4])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_values_bit_exact(dtype, S, where):
    lat, lon, _, x = _subdaily(S, dtype, n_days=12)
    xs = x.reshape(12, S, len(lat), len(lon))
    xs[2, :, 0, :4] = [[0.0, -0.0, 1.0, np.nan]] * S                     # +-0 ties
    ds = _ds(x, lat, lon, S, where, n_days=12)
    for how in ("mean", "min", "max"):
        r = resample_daily(ds, how)
        ref = resample_daily_ref(x, S, how)
        _same(r.tas.values, ref)
        # lazy takes: lat / lon of the source, days of the result
        sub = r.isel(lat=np.arange(3, 17), lon=np.arange(40, 0, -3)).isel(time=[0, 5, 5, 11])
        _same(sub.tas.values, ref[[0, 5, 5, 11]][:, 3:17][:, :, np.arange(40, 0, -3)])
    # a source that starts within the physical steps
    r = resample_daily(ds.isel(time=np.arange(2 * S, 7 * S)), "mean")
    _same(r.tas.values, resample_daily_ref(x[2 * S: 7 * S], S, "mean"))


# ----------------------------------------------------------------------------
# GPU: aggregates
# ----------------------------------------------------------------------------
DIMS = ("time", "lat", "lon")
EDGES = (-np.inf, -5.0, 5.0, 15.0, np.inf)
KNOTS = (-5.0, 5.0, 12.0, 20.0, 28.0)


def _oracle_agg(x, lat, lon, df, aggwt="popwt", agglev="hierid"):
    return oracle.weighted_aggregate_grid_to_regions(x, DIMS, lat, lon, df, aggwt, agglev)


def _n_rows(df, agglev, labels):
    return df.groupby(agglev).size().reindex(labels).values.astype(np.float64)


def _check_pair(sub, mat, ref, scale, df, agglev, labels, tol=TOL, days=0):
    """``sub``: the sub-daily path; ``mat``: the existing path on the materialised daily arrays; ``ref``: the
    oracle on the restated daily arrays; all [time, region].  ``sub`` and ``ref`` agree to ``tol`` of the
    cancellation-aware scale, ``sub`` and ``mat`` to ``(n_r + 4) 2^-53 S_r`` (``+ days`` for sums of that many
    days)."""
    assert rel_err(sub, ref, scale) <= tol
    n_r = _n_rows(df, agglev, labels)
    bound = (n_r[None, :] + 4 + days) * 2.0 ** -53 * np.broadcast_to(scale, sub.shape)
    assert np.array_equal(np.isnan(sub), np.isnan(mat))
    fin = np.isfinite(sub)
    assert np.array_equal(sub[~fin & ~np.isnan(sub)], mat[~fin & ~np.isnan(sub)])
    assert (np.abs(sub[fin] - mat[fin]) <= bound[fin]).all(), np.max(np.abs(sub[fin] - mat[fin]) / bound[fin])


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


CASES = ["identity", "poly", "bins", "rcspline", "snyder", "year", "season", "multi"]
S_OF = {"identity": 24, "poly": 8, "bins": 4, "rcspline": 24, "snyder": 8, "year": 4, "season": 24, "multi": 8}


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "pinned"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("case", CASES)
def test_aggregates(case, dtype, where):
    S = S_OF[case]
    lat, lon, df, x = _subdaily(S, dtype, specials=case != "snyder")
    ds = _ds(x, lat, lon, S, where)
    days = _days()
    keep = oracle.leap_day_keep_mask(days)
    mean = resample_daily_ref(x, S, "mean")
    mat = Dataset({"tas": (DIMS, _dev(mean))}, coords={"time": days, "lat": lat, "lon": lon})
    agg = weighted_aggregate_grid_to_regions

    if case == "identity":
        sub = agg(resample_daily(ds, "mean"), "tas", "popwt", "hierid", weights=df)["tas"].values
        ref, _, labels = _oracle_agg(mean, lat, lon, df)
        scale = _oracle_agg(np.abs(mean), lat, lon, df)[0]
        _check_pair(sub, agg(mat, "tas", "popwt", "hierid", weights=df)["tas"].values, ref, scale, df, "hierid", labels)
    elif case in ("poly", "bins", "rcspline"):
        def build(src):
            if case == "poly":
                return tas_poly(src, [1, 2, 3, 4], ["p1", "p2", "p3", "p4"])
            if case == "bins":
                return tas_bins(src, EDGES, "b")
            return tas_rcspline(src, KNOTS, "s")
        d1 = build(resample_daily(ds, "mean"))
        names = list(d1.data_vars)
        agg(d1, names, "popwt", "hierid", weights=df)             # builds the plan
        n0 = E.launch_count()
        out = agg(d1, names, "popwt", "hierid", weights=df)
        if case == "poly" and where == "device":
            assert E.launch_count() - n0 == 2               # one reduce-pack, one aggregation of 4 orders
        ref_out = agg(build(mat), names, "popwt", "hierid", weights=df)
        xk = mean[keep]
        for i, name in enumerate(names):
            if case == "poly":
                v = oracle.tas_poly(mean, days, i + 1)[0]
                sc = np.abs(v)
            elif case == "bins":
                v = bins_ref(xk, EDGES[i], EDGES[i + 1])
                sc = np.abs(v)
            else:
                v, sc = rcs_ref(xk, KNOTS, i), rcs_scale(xk, KNOTS, i)
            ref, _, labels = _oracle_agg(v, lat, lon, df)
            scale = _oracle_agg(sc, lat, lon, df)[0]
            _check_pair(out[name].values, ref_out[name].values, ref, scale, df, "hierid", labels)
            np.testing.assert_array_equal(out.time.values, oracle.tas_poly_time_labels(days[keep]))
    elif case == "snyder":
        lo, hi = resample_daily(ds, "min"), resample_daily(ds, "max")
        tmin, tmax = resample_daily_ref(x, S, "min"), resample_daily_ref(x, S, "max")
        mat2 = Dataset({"mn": (DIMS, _dev(tmin)), "mx": (DIMS, _dev(tmax))},
                       coords={"time": days, "lat": lat, "lon": lon})
        for v in (lo.tas, hi.tas, mat2.mn, mat2.mx):
            v.attrs["units"] = "K"
        w = np.abs(tmin.astype(np.float64)) + np.abs(tmax.astype(np.float64))
        scale = _oracle_agg(w, lat, lon, df)[0]
        for thr in ((290.0,), (285.0, 295.0)):
            f = snyder_edd if len(thr) == 1 else snyder_gdd
            ofn = oracle.snyder_edd if len(thr) == 1 else oracle.snyder_gdd
            sub = agg(Dataset({"e": f(lo.tas, hi.tas, *thr)}, coords=lo._coords), "e", "popwt", "hierid", weights=df)
            mat_e = agg(Dataset({"e": f(mat2.mn, mat2.mx, *thr)}, coords=mat2._coords), "e", "popwt", "hierid",
                        weights=df)
            ref, _, labels = _oracle_agg(ofn(tmin, tmax, *thr), lat, lon, df)
            _check_pair(sub["e"].values, mat_e["e"].values, ref, scale, df, "hierid", labels)
    elif case == "year":
        d1 = tas_poly(resample_daily(ds, "mean"), 1, "p1")
        sub = agg(d1, "p1", "popwt", "hierid", weights=df, time_groups="year")
        mat_y = agg(tas_poly(mat, 1, "p1"), "p1", "popwt", "hierid", weights=df, time_groups="year")
        v = oracle.tas_poly(mean, days, 1)[0]
        ref, rd, labels = _oracle_agg(v, lat, lon, df)
        scale = _oracle_agg(np.abs(v), lat, lon, df)[0]
        years = d1.time.values // 1000
        ref_y, yl = oracle.time_group_sum(ref, rd, years)
        scale_y, _ = oracle.time_group_sum(scale, rd, years)
        assert list(sub.time.values) == list(yl) == [2003, 2004]
        _check_pair(sub["p1"].values, mat_y["p1"].values, ref_y, scale_y, df, "hierid", labels, days=N_DAYS)
    elif case == "season":
        from climate_toolbox_b200.utils.utils import get_daily_growing_season_mask
        rng = np.random.default_rng(21)
        nlat, nlon = len(lat), len(lon)
        plant = rng.integers(1, 366, (nlat, nlon)).astype(np.float64)
        harv = rng.integers(1, 366, (nlat, nlon)).astype(np.float64)
        plant[rng.random((nlat, nlon)) < 0.05] = np.nan
        gd = Dataset({"variable": (("z", "latitude", "longitude"), np.stack([plant, harv]))},
                     coords={"z": np.array([1, 2]), "latitude": lat, "longitude": lon + 180})
        d1 = resample_daily(ds, "mean")
        m = get_daily_growing_season_mask(lat, lon, days, gd)
        sub = agg(d1, "tas", "cropwt", "hierid", weights=df, season_mask=m)["tas"].values
        mat_s = agg(mat, "tas", "cropwt", "hierid", weights=df, season_mask=m)["tas"].values
        dense = oracle.growing_season_mask(plant, harv, pd.DatetimeIndex(days).dayofyear.values).transpose(2, 0, 1)
        with np.errstate(invalid="ignore"):                  # inf x 0 outside the season: NaN, skipped
            ref, _, labels = _oracle_agg(mean * dense, lat, lon, df, "cropwt")
            scale = _oracle_agg(np.abs(mean) * dense, lat, lon, df, "cropwt")[0]
        _check_pair(sub, mat_s, ref, scale, df, "hierid", labels)
        assert not np.allclose(np.nan_to_num(sub), np.nan_to_num(
            agg(d1, "tas", "cropwt", "hierid", weights=df)["tas"].values))
    else:
        wts = ["popwt", "areawt"]
        sub = weighted_aggregate_grid_to_regions_multi(resample_daily(ds, "mean"), "tas", wts, "hierid", df)
        mat_m = weighted_aggregate_grid_to_regions_multi(mat, "tas", wts, "hierid", df)
        for wt in wts:
            ref, _, labels = _oracle_agg(mean, lat, lon, df, wt)
            scale = _oracle_agg(np.abs(mean), lat, lon, df, wt)[0]
            name = "tas_{}".format(wt)
            _check_pair(sub[name].values, mat_m[name].values, ref, scale, df, "hierid", labels)


@pytest.mark.gpu
def test_pageable_host_source():
    """A pageable host source is staged in whole days and gives what the device source gives."""
    lat, lon, df, x = _subdaily(24, np.float32, n_days=20)
    res = [weighted_aggregate_grid_to_regions(resample_daily(_ds(x, lat, lon, 24, w, n_days=20), "mean"), "tas",
                                              "popwt", "hierid", weights=df)["tas"].values
           for w in ("pageable", "device")]
    np.testing.assert_array_equal(res[0], res[1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_snyder_reads_the_source_once(dtype):
    """min and max of one pinned source: one pass over the referenced pieces x steps crosses PCIe, not two."""
    S, n_days = 24, 30
    lat, lon, df, x = _subdaily(S, dtype, n_days=n_days, specials=False)
    ds = _ds(x, lat, lon, S, "pinned", n_days=n_days)
    lo, hi = resample_daily(ds, "min"), resample_daily(ds, "max")
    lo.tas.attrs["units"] = hi.tas.attrs["units"] = "K"
    e = Dataset({"e": snyder_edd(lo.tas, hi.tas, 290.0)}, coords=lo._coords)
    before = E.TRANSFER_BYTES["h2d"]
    weighted_aggregate_grid_to_regions(e, "e", "popwt", "hierid", weights=df)
    moved = E.TRANSFER_BYTES["h2d"] - before
    es = np.dtype(dtype).itemsize
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", stage_bytes=2 * es, compact=True, elem_bytes=es)
    assert moved == n_days * S * plan.info["n_pieces_distinct"] * 4 * es


@pytest.mark.gpu
def test_abi_checks_with_a_plan(lib):
    import torch
    lat, lon = synthetic.grid_labels(3.0)
    df = synthetic.weights_table(3.0, 50, seed=5)
    g = E.GridSpec(lat, lon)
    full = E.get_plan(g, df, "popwt", "hierid", cache=False)
    p4 = E.get_plan(g, df, "popwt", "hierid", compact=True, elem_bytes=4, cache=False)
    p8 = E.get_plan(g, df, "popwt", "hierid", compact=True, elem_bytes=8, cache=False)
    ncell = len(lat) * len(lon)
    x = torch.zeros((4 * 24, ncell), dtype=torch.float32, device="cuda")
    d8 = torch.zeros((4, p8.info["n_packed_cells"]), dtype=torch.float64, device="cuda")
    d4 = torch.zeros((4, p4.info["n_packed_cells"]), dtype=torch.float32, device="cuda")
    L = lib

    def call(plan, S=24, ops=N.DAILY_MEAN, mean=d8, mn=None, mx=None, xp=None):
        return L.ctb_pull_pack_daily(plan._h, xp or x.data_ptr(), N.F32, ncell, S, None, 0, 4, ops,
                                     None if mean is None else mean.data_ptr(), None if mn is None else mn.data_ptr(),
                                     None if mx is None else mx.data_ptr(), None)

    assert call(full) == N.ERR_INVALID and "compact" in N.last_error()
    assert call(p8, S=0) == N.ERR_INVALID and "steps_per_day" in N.last_error()
    assert call(p8, ops=0) == N.ERR_INVALID
    assert call(p8, ops=8) == N.ERR_INVALID
    assert call(p8, ops=N.DAILY_MIN, mn=None) == N.ERR_INVALID
    assert call(p4) == N.ERR_INVALID and "float64" in N.last_error()              # mean needs elem_bytes 8
    assert call(p8, ops=N.DAILY_MIN | N.DAILY_MAX, mean=None, mn=d8, mx=d8) == N.ERR_INVALID
    assert call(p8, xp=x.data_ptr() + 4) == N.ERR_UNSUPPORTED
    assert call(p4, ops=N.DAILY_MIN | N.DAILY_MAX, mean=None, mn=d4, mx=d4) == N.OK
    assert call(p8) == N.OK
    torch.cuda.synchronize()
    for p in (full, p4, p8):
        p.close()
