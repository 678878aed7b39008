"""Restricted cubic spline terms of daily temperature (``tas_rcspline``, ``CTB_TR_RCSPLINE``), fused into the
aggregation.

CPU: the reference rule (``rcs_ref``; the parity tests feed it to the restated reference aggregation of
``oracle``) against exact rational arithmetic, ``tas_rcspline`` metadata and validation, the fusion of
consecutive terms into launches, and the C-ABI's parameter checks.  GPU: ``.values`` and the fused aggregation
against the reference -- NaN, infinity and zero patterns exact, values within 1e-13 of the cancellation-aware
scale ``rcs_scale`` pointwise and within the summation-order tolerance aggregated."""
import ctypes
from fractions import Fraction

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
from climate_toolbox_b200.transformations.transformations import tas_poly, tas_rcspline

OFF = 273.15
INF = np.inf
KNOTS5 = (-5.0, 5.0, 12.0, 20.0, 28.0)
KNOTS7 = (-10.0, 0.0, 5.0, 10.0, 15.0, 20.0, 30.0)


# ----------------------------------------------------------------------------
# the reference rule (numpy), beside the restated reference in oracle/
# ----------------------------------------------------------------------------
def _pieces(x, knots, i, offset):
    """d, c(k_i), a_i, c(k_{n-1}), b_i, c(k_n) of term ``i >= 1`` in float64."""
    k = [float(v) for v in knots]
    n = len(k)
    d = np.asarray(x).astype(np.float64) - offset
    with np.errstate(invalid="ignore", over="ignore"):
        def c(kk):
            return np.maximum(d - kk, 0.0) ** 3
        ki, km, kn = k[i - 1], k[n - 2], k[n - 1]
        return d, c(ki), (kn - ki) / (kn - km), c(km), (km - ki) / (kn - km), c(kn)


def rcs_ref(x, knots, i, offset=OFF):
    """Term ``B_i`` of the restricted cubic spline basis of ``knots`` (Harrell, unnormalised) at
    ``d = float64(x) - offset``: ``B_0 = d``; for ``1 <= i <= n-2``
    ``B_i = c(k_i) - c(k_{n-1}) a_i + c(k_n) b_i`` with ``c(k) = max(d - k, 0)^3`` (NaN propagates),
    ``a_i = (k_n - k_i)/(k_n - k_{n-1})`` and ``b_i = (k_{n-1} - k_i)/(k_n - k_{n-1})``.  Every operation in
    float64 (DESIGN.md "dtype policy")."""
    if i == 0:
        return np.asarray(x).astype(np.float64) - offset
    _, ci, a, cm, b, cn = _pieces(x, knots, i, offset)
    with np.errstate(invalid="ignore", over="ignore"):
        return ci - cm * a + cn * b


def rcs_scale(x, knots, i, offset=OFF):
    """The cancellation-aware magnitude of ``B_i``: ``|c(k_i)| + |a_i c(k_{n-1})| + |b_i c(k_n)|`` (``|d|``
    for ``i = 0``).  Aggregated like the data, it is the scale of the aggregate's rounding too."""
    if i == 0:
        return np.abs(np.asarray(x).astype(np.float64) - offset)
    _, ci, a, cm, b, cn = _pieces(x, knots, i, offset)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.abs(ci) + np.abs(a * cm) + np.abs(b * cn)


def tas_rcspline_ref(tas, times, knots, i, time_axis=0):
    """Term ``i`` of ``tas`` (K) after leap-day removal, shaped like ``oracle.tas_poly``.  Returns
    ``(values, scale, new_time_labels)``."""
    keep = oracle.leap_day_keep_mask(times)
    tas = np.compress(keep, np.asarray(tas), axis=time_axis)
    if tas.shape[time_axis] > 365:
        raise ValueError
    return (rcs_ref(tas, knots, i), rcs_scale(tas, knots, i),
            oracle.tas_poly_time_labels(np.asarray(times)[keep]))


def rcs_exact(d, knots, i):
    """``B_i(d)`` in exact rational arithmetic from the definition."""
    k = knots
    n = len(k)

    def c(kk):
        return max(d - kk, Fraction(0)) ** 3
    ki, km, kn = k[i - 1], k[n - 2], k[n - 1]
    return c(ki) - c(km) * (kn - ki) / (kn - km) + c(kn) * (km - ki) / (kn - km)


# ----------------------------------------------------------------------------
# reference pins (CPU)
# ----------------------------------------------------------------------------
def test_reference_known_answers():
    k = (0.0, 1.0, 2.0)
    np.testing.assert_array_equal(rcs_ref(np.array([3.0, 4.0, 0.5, -1.0]), k, 1, 0.0), [12.0, 18.0, 0.125, 0.0])
    np.testing.assert_array_equal(rcs_ref(np.array([3.0, -1.0]), k, 0, 0.0), [3.0, -1.0])
    assert rcs_ref(np.float32(OFF), k, 0) == np.float64(np.float32(OFF)) - OFF     # widened, then subtracted


def test_reference_pieces_against_exact_rationals():
    """The three pieces of B_i and its linearity above k_n hold exactly for the definition, and the float64 rule
    is within 1e-13 of the scale of the exact value, on random dyadic knots and points (exact in float64)."""
    rng = np.random.default_rng(17)
    for _ in range(60):
        n = int(rng.integers(3, 8))
        kk = np.sort(rng.choice(np.arange(-400, 400), size=n, replace=False))
        knots = [Fraction(int(v), 8) for v in kk]
        pts = [Fraction(int(v), 16) for v in rng.integers(-1200, 1200, size=40)] + knots
        for i in range(1, n - 1):
            ki, km, kn = knots[i - 1], knots[n - 2], knots[n - 1]
            for d in pts:
                b = rcs_exact(d, knots, i)
                if d <= ki:
                    assert b == 0
                if ki <= d <= km:
                    assert b == (d - ki) ** 3
                if d >= kn:
                    assert b == (kn - ki) * (km - ki) * (3 * d - ki - km - kn)
                got = rcs_ref(np.float64(d), [float(v) for v in knots], i, 0.0)
                scale = rcs_scale(np.float64(d), [float(v) for v in knots], i, 0.0)
                assert abs(got - float(b)) <= 1e-13 * max(scale, 1e-300), (knots, i, d)
            # linear above k_n: equal steps give equal differences
            h = Fraction(3, 4)
            v = [rcs_exact(kn + j * h, knots, i) for j in range(4)]
            assert v[1] - v[0] == v[2] - v[1] == v[3] - v[2]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_reference_zero_exactly_at_or_below_the_knot(dtype):
    rng = np.random.default_rng(4)
    x = np.concatenate([(OFF + rng.uniform(-30, 40, 5000)).astype(dtype),
                        [dtype(v + OFF) for v in KNOTS5]])
    d = x.astype(np.float64) - OFF
    for i in range(1, len(KNOTS5) - 1):
        b = rcs_ref(x, KNOTS5, i)
        below = d <= KNOTS5[i - 1]
        assert below.any() and (~below).any()
        assert (b[below] == 0).all() and (b[~below] > 0).all()


def test_reference_nan_and_infinities():
    x = np.array([np.nan, INF, -INF])
    np.testing.assert_array_equal(rcs_ref(x, KNOTS5, 0), [np.nan, INF, -INF])
    for i in range(1, len(KNOTS5) - 1):
        np.testing.assert_array_equal(rcs_ref(x, KNOTS5, i), [np.nan, np.nan, 0.0])


def test_reference_tas_rcspline_drops_leap_days():
    t = pd.date_range("2000-02-27", periods=5)
    tas = np.array([270.0, 280.0, 290.0, 300.0, np.nan])[:, None]
    v, s, labels = tas_rcspline_ref(tas, t, KNOTS5, 1)
    np.testing.assert_array_equal(v[:, 0], rcs_ref(tas[[0, 1, 3, 4], 0], KNOTS5, 1))
    assert np.isnan(v[3, 0]) and np.isnan(s[3, 0])
    np.testing.assert_array_equal(labels, oracle.tas_poly_time_labels(t[[0, 1, 3, 4]]))


# ----------------------------------------------------------------------------
# tas_rcspline metadata and validation (CPU)
# ----------------------------------------------------------------------------
def _small_ds(T=5, start="2000-02-27"):
    t = pd.date_range(start, periods=T)
    return Dataset({"tas": (("time", "lat", "lon"), np.full((T, 2, 2), 290.0, dtype=np.float32))},
                   coords={"time": t, "lat": [0.0, 1.0], "lon": [0.0, 1.0]}), t


def test_tas_rcspline_names_attrs_and_time():
    ds, t = _small_ds()
    ds1 = tas_rcspline(ds, KNOTS5)
    names = ["tas_rcspline_{}".format(i) for i in range(4)]
    assert list(ds1.data_vars) == names
    v = ds1["tas_rcspline_2"]
    assert v.shape == (4, 2, 2) and v.dims == ("time", "lat", "lon")           # Feb 29 dropped
    np.testing.assert_array_equal(ds1.time.values, oracle.tas_poly_time_labels(t[[0, 1, 3, 4]]))
    assert ds1["tas_rcspline_0"].attrs["units"] == "C" and v.attrs["units"] == "C^3"
    assert v.attrs["knots"] == list(KNOTS5) and v.attrs["rcspline_term"] == 2
    assert v.attrs["variable"] == "tas_rcspline_2"
    assert v.attrs["long_title"] == "Restricted cubic spline term 2 of daily average temperature (degrees C)"
    assert ds1["tas_rcspline_0"].attrs["long_title"] == "Linear term of daily average temperature (degrees C)"
    assert v.attrs["description"].startswith(v.attrs["long_title"]) and "365 day" in v.attrs["description"]
    d = v.variable.deferred
    assert d.kind == "rcspline" and d.params == (273.15, 2.0) + KNOTS5
    named = tas_rcspline(ds, (0.0, 10.0, 20.0), ["lin", "cubic"])
    assert list(named.data_vars) == ["lin", "cubic"] and named["cubic"].attrs["variable"] == "cubic"
    assert list(tas_rcspline(ds, [0, 1, 2], "s").data_vars) == ["s_0", "s_1"]


@pytest.mark.parametrize("knots,names", [
    ([0.0, 10.0], "s"),                                   # 2 knots
    ([float(v) for v in range(8)], "s"),                  # 8 knots
    ([0.0, 20.0, 10.0], "s"),                             # unsorted
    ([0.0, 10.0, 10.0, 20.0], "s"),                       # duplicate
    ([0.0, np.nan, 20.0], "s"),                           # NaN
    ([0.0, 10.0, INF], "s"),                              # infinite
    ([-INF, 0.0, 10.0], "s"),
    ([[0.0, 10.0, 20.0]], "s"),                           # not 1-D
    ([0.0, 10.0, 20.0], ["only_one"]),                    # name count mismatch
    ([0.0, 10.0, 20.0, 30.0], ["a", "b", "c", "d"]),
])
def test_tas_rcspline_rejects_bad_knots_and_names(knots, names):
    ds, _ = _small_ds()
    with pytest.raises(ValueError):
        tas_rcspline(ds, knots, names)


def test_tas_rcspline_more_than_365_steps():
    big = Dataset({"tas": (("time", "lat"), np.zeros((400, 1)))},
                  coords={"time": pd.date_range("2001-01-01", periods=400), "lat": [0.0]})
    with pytest.raises(ValueError):
        tas_rcspline(big, KNOTS5)


# ----------------------------------------------------------------------------
# fusion into launches (CPU)
# ----------------------------------------------------------------------------
def _reqs(ds1):
    return [(n,) + _resolve(ds1._vars[n]) for n in ds1.data_vars]


def test_five_knots_one_launch_seven_knots_two():
    ds, _ = _small_ds()
    g5 = _group_requests(_reqs(tas_rcspline(ds, KNOTS5)))
    assert [len(g["names"]) for g in g5] == [4] and g5[0]["kind"] == "rcspline"
    assert g5[0]["params"] == (OFF, 0.0) + KNOTS5
    g7 = _group_requests(_reqs(tas_rcspline(ds, KNOTS7, "s")))
    assert [len(g["names"]) for g in g7] == [4, 2]
    assert g7[0]["params"] == (OFF, 0.0) + KNOTS7 and g7[1]["params"] == (OFF, 4.0) + KNOTS7
    assert g7[0]["names"] == ["s_0", "s_1", "s_2", "s_3"] and g7[1]["names"] == ["s_4", "s_5"]


def test_terms_that_do_not_fuse():
    a = Variable(("time", "lat", "lon"), np.zeros((2, 2, 2)))
    b = Variable(("time", "lat", "lon"), np.zeros((2, 2, 2)))
    k = (0.0, 10.0, 20.0, 30.0)

    def groups(*terms):
        return [len(g["names"]) for g in _group_requests(
            [("t{}".format(j), "rcspline", p, [s]) for j, (p, s) in enumerate(terms)])]

    assert groups(((OFF, 0.0) + k, a), ((OFF, 1.0) + k, a)) == [2]
    assert groups(((OFF, 0.0) + k, a), ((OFF, 2.0) + k, a)) == [1, 1]                       # gap
    assert groups(((OFF, 1.0) + k, a), ((OFF, 0.0) + k, a)) == [1, 1]                       # out of order
    assert groups(((OFF, 0.0) + k, a), ((OFF, 1.0, 0.0, 10.0, 20.0, 31.0), a)) == [1, 1]    # other knots
    assert groups(((OFF, 0.0) + k, a), ((273.0, 1.0) + k, a)) == [1, 1]                     # offset
    assert groups(((OFF, 0.0) + k, a), ((OFF, 1.0) + k, b)) == [1, 1]                       # source
    # next to a polynomial of the same source: separate launches, the polynomials still fuse
    ds, _ = _small_ds()
    mixed = _reqs(tas_poly(ds, [1, 2], ["p1", "p2"]))
    src = mixed[0][3]
    mixed.insert(1, ("s0", "rcspline", (OFF, 0.0) + k, src))
    mixed.append(("s1", "rcspline", (OFF, 1.0) + k, src))
    g = _group_requests(mixed)
    assert [(x["kind"], x["names"]) for x in g] == [("poly", ["p1", "p2"]), ("rcspline", ["s0", "s1"])]
    assert g[1]["params"] == (OFF, 0.0) + k


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
    return L.ctb_transform(ctypes.addressof(dummy), None, N.F64, 0, N.TR_RCSPLINE,
                           p.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), int(p.size), n_out, None, None)


def test_abi_validates_rcspline_params(lib):
    assert N.TR_RCSPLINE == 5
    k5 = list(KNOTS5)
    assert _transform_rc(lib, [OFF, 0.0] + k5, 4) == N.OK
    assert _transform_rc(lib, [OFF, 1.0] + k5, 3) == N.OK
    assert _transform_rc(lib, [OFF, 3.0] + k5, 1) == N.OK
    assert _transform_rc(lib, [OFF, 0.0, 0.0, 1.0, 2.0], 2) == N.OK                      # 3 knots
    assert _transform_rc(lib, [OFF, 4.0] + list(KNOTS7), 2) == N.OK                      # 7 knots, second launch
    assert _transform_rc(lib, [INF, 0.0] + k5, 4) == N.ERR_INVALID                       # offset
    assert _transform_rc(lib, [np.nan, 0.0] + k5, 4) == N.ERR_INVALID
    assert "offset" in N.last_error()
    assert _transform_rc(lib, [OFF, 0.0, 0.0, 1.0], 1) == N.ERR_INVALID                  # 2 knots
    assert _transform_rc(lib, [OFF, 0.0] + [float(v) for v in range(8)], 4) == N.ERR_INVALID   # 8 knots
    assert "knots" in N.last_error()
    assert _transform_rc(lib, [OFF, 0.0, 0.0, 2.0, 1.0], 1) == N.ERR_INVALID             # not increasing
    assert _transform_rc(lib, [OFF, 0.0, 0.0, 1.0, 1.0], 1) == N.ERR_INVALID             # duplicate
    assert _transform_rc(lib, [OFF, 0.0, 0.0, np.nan, 1.0], 1) == N.ERR_INVALID          # NaN knot
    assert _transform_rc(lib, [OFF, 0.0, 0.0, 1.0, INF], 1) == N.ERR_INVALID             # infinite knot
    assert "strictly increasing" in N.last_error()
    assert _transform_rc(lib, [OFF, 0.5] + k5, 1) == N.ERR_INVALID                       # first not an integer
    assert _transform_rc(lib, [OFF, np.nan] + k5, 1) == N.ERR_INVALID
    assert _transform_rc(lib, [OFF, -1.0] + k5, 1) == N.ERR_INVALID                      # first < 0
    assert _transform_rc(lib, [OFF, 1.0] + k5, 4) == N.ERR_INVALID                       # first + n_out > n - 1
    assert _transform_rc(lib, [OFF, 4.0] + k5, 1) == N.ERR_INVALID
    assert "first" in N.last_error()
    assert _transform_rc(lib, [OFF, 0.0] + k5, 5) == N.ERR_INVALID                       # n_out > CTB_MAX_OUT


# ----------------------------------------------------------------------------
# GPU: .values and the fused aggregation against the oracle
# ----------------------------------------------------------------------------
def _adjacent(k, dtype):
    """Around the knot ``k``: one ulp below, on and one ulp above ``k + 273.15`` in ``dtype``, and the least
    value whose float64 ``x - 273.15`` exceeds ``k`` with its lower neighbour."""
    x = dtype(k + OFF)
    y = x
    while np.float64(y) - OFF > k:
        y = np.nextafter(y, dtype(-INF))
    while not np.float64(y) - OFF > k:
        y = np.nextafter(y, dtype(INF))
    return np.array([np.nextafter(x, dtype(-INF)), x, np.nextafter(x, dtype(INF)), np.nextafter(y, dtype(-INF)), y],
                    dtype=dtype)


def _special(dtype):
    big = [1e30, -1e30, 3.4e38, -3.4e38] + ([1e100, -1e100, 1e300, -1e300] if dtype == np.float64 else [])
    return np.array([np.nan, INF, -INF, 0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.2e-38, 1e-310 if dtype == np.float64
                     else 1e-44, -5.0, 273.15, 283.15, 293.15] + big, dtype=dtype)


def _near_knots(knots, dtype):
    return np.concatenate([_adjacent(k, dtype) for k in knots])


def _check_terms(got, x, knots, i, offset=OFF, tol=1e-13):
    """``got`` = B_i(x): NaN / inf patterns equal, zeros exactly where the rule is zero (d <= k_i; d = -inf),
    and every other value within ``tol`` of the scale.  Far above the knots the definition cancels to rounding
    noise of the scale (d^3): there a zero and a tiny value are the same answer, so the zero pattern is
    compared where the value stands above that noise."""
    got, x = np.asarray(got), np.asarray(x)
    ref, scale = rcs_ref(x, knots, i, offset), rcs_scale(x, knots, i, offset)
    assert rel_err(got, ref, scale) <= tol
    if i > 0:
        d = np.asarray(x).astype(np.float64) - offset
        rule_zero = d <= knots[i - 1]
        assert (got[rule_zero] == 0).all() and (ref[rule_zero] == 0).all()
        above_noise = np.abs(ref) > tol * scale
        assert (got[above_noise] != 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_values_knot_adjacent_and_special(dtype):
    """.values (the pointwise kernel), every term of a 7-knot basis."""
    x = np.concatenate([_near_knots(KNOTS7, dtype), _special(dtype)])[None, :]
    ds = Dataset({"tas": (("time", "x"), x)}, coords={"time": pd.date_range("2001-05-01", periods=1)})
    ds1 = tas_rcspline(ds, KNOTS7, "s")
    for i in range(len(KNOTS7) - 1):
        got = ds1["s_{}".format(i)].values
        assert got.dtype == np.float64
        _check_terms(got, x, KNOTS7, i)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("pool", ["knot_adjacent", "special"])
def test_one_gridcell_per_region(dtype, pool):
    """Every region is one gridcell of weight 1, so each result is B_i(x) itself (0 where it is NaN), through
    the streaming kernel (knot-adjacent float32 only: the integer widening with the decisions on the stored
    type; with special values: the exact loops) and the direct kernel, both launches of a 7-knot basis."""
    import torch
    nlat, nlon, T = 4, 8, 70
    lat, lon = np.arange(nlat) * 1.0, np.arange(nlon) * 1.0
    pool_v = _near_knots(KNOTS7, dtype)
    if pool == "special":
        pool_v = np.concatenate([pool_v, _special(dtype)])
    x = np.random.default_rng(3).choice(pool_v, size=(T, nlat * nlon)).astype(dtype)
    ii, jj = np.divmod(np.arange(nlat * nlon), nlon)
    df = pd.DataFrame({"lat": lat[ii], "lon": lon[jj], "hierid": np.arange(nlat * nlon),
                       "popwt": 1.0, "areawt": 1.0})
    dev = torch.device("cuda", 0)
    es = np.dtype(dtype).itemsize
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", device=dev, cache=False, elem_bytes=es,
                      stage_bytes=es)
    xd = torch.from_numpy(x).to(dev)
    for first, n_out in ((0, 4), (4, 2)):
        params = (OFF, float(first)) + KNOTS7
        for variant in (N.VARIANT_STAGED, N.VARIANT_DIRECT):
            out = E.aggregate_device(plan, xd, None, N.LAYOUT_TIME_MAJOR, nlat * nlon, None, T, "rcspline", params,
                                     n_out, variant=variant).cpu().numpy()
            for j in range(n_out):
                got = out[j].T
                skipped = np.isnan(rcs_ref(x, KNOTS7, first + j))      # NaN products leave the sum
                assert (got[skipped] == 0).all()
                _check_terms(got[~skipped], x[~skipped], KNOTS7, first + j)
    plan.close()


def _config(d, R, T, seed=1234, nan_frac=0.001, dtype=np.float32):
    lat, lon = synthetic.grid_labels(d)
    df = synthetic.weights_table(d, R, seed=seed)
    tas, _, _ = synthetic.tas_field(T, len(lat), len(lon), seed=7, nan_frac=nan_frac, dtype=dtype)
    return lat, lon, df, tas


def _oracle_agg(x, dims, lat, lon, df, aggwt, agglev):
    return oracle.weighted_aggregate_grid_to_regions(x, dims, lat, lon, df, aggwt, agglev)


def _check_agg(got, x, scale_x, dims, lat, lon, df, aggwt, agglev, tol):
    ref, rd, labels = _oracle_agg(x, dims, lat, lon, df, aggwt, agglev)
    scale, _, _ = _oracle_agg(scale_x, dims, lat, lon, df, aggwt, agglev)
    err = rel_err(got, ref, scale)
    assert err <= tol, err
    return rd, labels


@pytest.mark.gpu
@pytest.mark.parametrize("aggwt,agglev", [("popwt", "ISO"), ("areawt", "hierid")])
def test_reference_fixture_cell_major(ref_fix, aggwt, agglev):
    """The reference fixture (lat, lon, time) float64: CELL_MAJOR, the direct kernel."""
    lat, lon, time, temp, df = ref_fix
    ds = Dataset({"tas": (["lat", "lon", "time"], temp)}, coords={"lon": lon, "lat": lat, "time": time})
    knots = (-260.0, -240.0, -220.0, -200.0, -180.0)          # temp is 0..100 K: -273.15..-173.15 C
    ds1 = tas_rcspline(ds, knots, "s")
    names = list(ds1.data_vars)
    out = weighted_aggregate_grid_to_regions(ds1, names, aggwt, agglev, weights=df)
    for i, name in enumerate(names):
        xt, st, tl = tas_rcspline_ref(temp, time, knots, i, time_axis=2)
        _check_terms(ds1[name].values, np.compress(oracle.leap_day_keep_mask(time), temp, axis=2), knots, i)
        rd, labels = _check_agg(out[name].values, xt, st, ("lat", "lon", "time"), lat, lon, df, aggwt, agglev, 1e-12)
        assert out[name].dims == rd and list(out.coords[agglev].values) == list(labels)
        np.testing.assert_array_equal(out.coords["time"].values, tl)
        assert out[name].attrs["units"] == ("C" if i == 0 else "C^3")


def _put(a, where):
    import torch
    if where == "device":
        return torch.from_numpy(a).cuda()
    host = torch.empty(a.shape, dtype=torch.float32 if a.dtype == np.float32 else torch.float64, pin_memory=True)
    host.copy_(torch.from_numpy(a))
    return host.numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "host_pinned"])
def test_quarter_degree_seven_knots(where):
    """0.25-degree grid, 24,378 regions, 0.1 % NaN, a 7-knot basis: two fused launches (4 + 2 terms; device: the
    streaming kernel; pinned host: the compact plan and the GPU pull)."""
    lat, lon, df, tas = _config(0.25, 24378, 5)
    t = pd.date_range("2001-06-01", periods=5)
    ds = Dataset({"tas": (("time", "lat", "lon"), _put(tas, where))}, coords={"time": t, "lat": lat, "lon": lon})
    ds1 = tas_rcspline(ds, KNOTS7, "s")
    names = list(ds1.data_vars)
    assert len(names) == 6
    out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df)
    if where == "device":
        n0 = E.launch_count()
        out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df)
        assert E.launch_count() - n0 == 2
    for i, name in enumerate(names):
        rd, _ = _check_agg(out[name].values, rcs_ref(tas, KNOTS7, i), rcs_scale(tas, KNOTS7, i),
                           ("time", "lat", "lon"), lat, lon, df, "popwt", "hierid", 1e-9)
        assert out[name].dims == rd
        assert np.isfinite(out[name].values).mean() > 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["device", "host"])
def test_time_groups_year_sums_the_days(where):
    """time_groups="year": the yearly sums of the daily oracle, for every term of a 5-knot basis."""
    lat, lon, df, tas = _config(1.0, 3000, 365)
    t = pd.date_range("2001-07-01", periods=365)                 # two calendar years
    data = _put(tas, "device") if where == "device" else tas
    ds = Dataset({"tas": (("time", "lat", "lon"), data)}, coords={"time": t, "lat": lat, "lon": lon})
    ds1 = tas_rcspline(ds, KNOTS5, "s")
    names = list(ds1.data_vars)
    out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df, time_groups="year")
    years = ds1.time.values // 1000
    dims = ("time", "lat", "lon")
    for i, name in enumerate(names):
        xt, st, _ = tas_rcspline_ref(tas, t, KNOTS5, i)
        ref, rd, _ = _oracle_agg(xt, dims, lat, lon, df, "popwt", "hierid")
        scale, _, _ = _oracle_agg(st, dims, lat, lon, df, "popwt", "hierid")
        ref_y, yl = oracle.time_group_sum(ref, rd, years)
        scale_y, _ = oracle.time_group_sum(scale, rd, years)
        assert out[name].dims == rd and list(out.time.values) == list(yl) == [2001, 2002]
        err = rel_err(out[name].values, ref_y, scale_y)
        assert err <= 1e-9, err


@pytest.mark.gpu
def test_season_mask_gates_the_terms():
    """season_mask=: only gridcell-days inside their growing season count, == the oracle aggregate of
    B_i x the dense growing-season mask."""
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
    ds1 = tas_rcspline(ds, KNOTS5, "s")
    names = list(ds1.data_vars)
    m = get_daily_growing_season_mask(ds1["lat"], ds1["lon"], ds1["time"], gd)
    out = weighted_aggregate_grid_to_regions(ds1, names, "cropwt", "hierid", weights=df, season_mask=m)
    plain = weighted_aggregate_grid_to_regions(ds1, names, "cropwt", "hierid", weights=df)
    dense = oracle.growing_season_mask(plant, harv, t.dayofyear.values).transpose(2, 0, 1)
    for i, name in enumerate(names):
        rd, _ = _check_agg(out[name].values, rcs_ref(tas, KNOTS5, i) * dense, rcs_scale(tas, KNOTS5, i) * dense,
                           ("time", "lat", "lon"), lat, lon, df, "cropwt", "hierid", 1e-9)
        assert out[name].dims == rd
        assert not np.allclose(np.nan_to_num(plain[name].values), np.nan_to_num(out[name].values))
