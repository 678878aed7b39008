"""Gridcell-level transforms (mirror of
``/root/reference/climate_toolbox/transformations/transformations.py:7-214``).

Each function returns variables holding a *deferred* transform: aggregating them
fuses the arithmetic into the gather kernel (no full-grid temporaries);
``.values`` evaluates them with the pointwise CUDA kernel.  Arithmetic is float64
from the first operation whatever the storage dtype (DESIGN.md, dtype policy).
"""
from __future__ import annotations

import numpy as np
import torch

from .._xr import DataArray, Dataset, Deferred, Variable, from_any, to_like
from ..utils.utils import remove_leap_days, convert_kelvin_to_celsius  # noqa: F401

__all__ = ["snyder_edd", "snyder_gdd", "validate_edd_snyder_agriculture", "tas_poly", "tas_bins", "tas_rcspline",
           "ordinal"]


def _source(da):
    """The stored data a transform reads: daily reductions of sub-daily data stay deferred (they are
    reduced while the aggregation packs its inputs), other deferred variables are evaluated."""
    v = da.variable
    return v if v.deferred is None or v.deferred.kind == "daily" else Variable(v.dims, v.values, v.attrs)


def _min_max_of_one_source(a, b):
    """``a`` and ``b`` are the daily minimum and maximum of the same sub-daily data and days."""
    da, db = a.deferred, b.deferred
    return (da is not None and db is not None and da.kind == db.kind == "daily" and
            (da.params[0], db.params[0]) == ("min", "max") and da.params[1:3] == db.params[1:3] and
            np.array_equal(da.params[3], db.params[3]) and da.sources[0].physical is db.sources[0].physical and
            da.sources[0].takes.keys() == db.sources[0].takes.keys() and
            all(np.array_equal(da.sources[0].takes[k], db.sources[0].takes[k]) for k in da.sources[0].takes))


def _any_less(a, b):
    """``(a < b).any()`` on the data's own device (precondition check only)."""
    if _min_max_of_one_source(b, a):
        return False          # a daily maximum is never below the minimum of the same steps
    pa, pb = a.physical, b.physical
    if isinstance(pa, torch.Tensor) and isinstance(pb, torch.Tensor) and not a.takes and not b.takes:
        return bool((pa < pb).any().item())
    return bool((a.values < b.values).any())


def snyder_edd(tasmin, tasmax, threshold, check=True):
    r"""
    Snyder exceedance degree days/cooling degree days (reference ``:7-93``).

    .. math::

        EDD_d = \begin{cases}
            ((M - e)(\pi/2 - \theta) + w\cos\theta)/\pi & tmin_d < e < tmax_d \\
            0 & tmax_d < e \\
            M - e & \text{otherwise} \end{cases}
        \quad M = (tmax_d + tmin_d)/2,\ w = (tmax_d - tmin_d)/2,\ \theta = \arcsin((e - M)/w)

    ``tasmin`` / ``tasmax`` : DataArray with a ``units`` attribute; ``threshold`` in
    the same units.  ``check=False`` skips the ``tasmax >= tasmin`` scan.
    """
    tasmin, tasmax = from_any(tasmin), from_any(tasmax)
    # Check for unit agreement (AttributeError if a `.units` attr is missing)
    assert tasmin.units == tasmax.units
    smin, smax = _source(tasmin), _source(tasmax)
    if check:
        assert not _any_less(smax, smin), "values encountered where tasmin > tasmax"
    attrs = {"units": "degreedays_{}{}".format(threshold, tasmax.attrs["units"])}
    var = Variable(smin.dims, None, attrs, None,
                   Deferred("edd", (float(threshold),), (smin, smax)))
    return DataArray._wrap(var, tasmax._coords, tasmax.name)


def snyder_gdd(tasmin, tasmax, threshold_low, threshold_high, check=True):
    r"""
    Snyder growing degree days (reference ``:96-147``):
    ``GDD = EDD(threshold_low) - EDD(threshold_high)`` per gridcell-day.
    """
    tasmin, tasmax = from_any(tasmin), from_any(tasmax)
    assert tasmin.units == tasmax.units
    smin, smax = _source(tasmin), _source(tasmax)
    if check:
        assert not _any_less(smax, smin), "values encountered where tasmin > tasmax"
    attrs = {"units": "degreedays_{}-{}{}".format(threshold_low, threshold_high,
                                                  tasmax.attrs["units"])}
    var = Variable(smin.dims, None, attrs, None,
                   Deferred("gdd", (float(threshold_low), float(threshold_high)), (smin, smax)))
    return DataArray._wrap(var, tasmax._coords, tasmax.name)


def validate_edd_snyder_agriculture(ds, thresholds):
    """reference ``:150-157``"""
    msg_null = "hierid dims do not match 24378"

    assert ds.hierid.shape == (24378,), msg_null

    for threshold in thresholds:
        assert threshold in list(ds.refTemp)
    return


def _daily_tas_365(ds):
    """The shared first steps of ``tas_poly`` / ``tas_bins`` / ``tas_rcspline``: ``ds["tas"]`` without leap
    days, and an empty Dataset with the coordinates of ``ds`` and ``time`` as ``YYYYDDD``.  Returns
    ``(ds1, tas)``; more than 365 steps raise ``ValueError``."""
    # remove leap years
    ds = remove_leap_days(ds)
    tas = _source(ds["tas"])

    # Replace datetime64[ns] 'time' with YYYYDDD int 'day'
    if ds.dims["time"] > 365:
        raise ValueError
    ds1 = Dataset()
    for k, c in ds._coords.items():
        if k != "time":
            ds1._coords[k] = c
    year = np.asarray(ds["time.year"].values, dtype=np.int64)
    ds1._coords["time"] = Variable(("time",), year * 1000 + np.arange(1, len(year) + 1))
    return ds1, tas


def tas_poly(ds, power, varname):
    """
    Daily average temperature (degrees C), raised to a power (reference ``:160-208``).

    Leap years are removed before counting days (uses a 365 day calendar).
    ``power`` / ``varname`` may also be equal-length lists: all orders are then
    produced from ONE read of ``tas`` when aggregated.
    """
    like = ds
    ds = from_any(ds)
    powers = [power] if np.isscalar(power) else list(power)
    names = [varname] if isinstance(varname, str) else list(varname)
    if len(powers) != len(names):
        raise ValueError("power and varname must have the same length")

    ds1, tas = _daily_tas_365(ds)

    for p, name in zip(powers, names):
        powername = ordinal(p)
        description = (
            """
            Daily average temperature (degrees C){raised}

            Leap years are removed before counting days (uses a 365 day
            calendar).
            """.format(
                raised="" if p == 1 else (" raised to the {powername} power".format(powername=powername))
            )
        ).strip()
        attrs = {"units": "C^{}".format(p) if p > 1 else "C",
                 "long_title": description.splitlines()[0], "description": description,
                 "variable": name}
        # do transformation: (tas - 273.15) ** power, deferred
        ds1._vars[name] = Variable(tas.dims, None, attrs, None,
                                   Deferred("poly", (273.15, float(p)), (tas,)))
    return to_like(ds1, like)


def _bin_edges(edges):
    """``edges`` as a float64 array of K+1 >= 2 strictly increasing, non-NaN values; only the first may
    be -inf and only the last +inf."""
    e = np.asarray(edges, dtype=np.float64)
    if e.ndim != 1 or e.size < 2:
        raise ValueError("edges must be a 1-D sequence of at least 2 values, got {!r}".format(edges))
    if np.isnan(e).any():
        raise ValueError("edges must not be NaN: {!r}".format(edges))
    # strictly increasing edges can be infinite only at the ends (inf - inf is NaN): -inf first, +inf last
    with np.errstate(invalid="ignore"):
        increasing = (np.diff(e) > 0).all()
    if not increasing:
        raise ValueError("edges must be strictly increasing, infinite only at the ends: {!r}".format(edges))
    return e


def tas_bins(ds, edges, varname="tas_bin"):
    """
    Daily average temperature (degrees C) binned: one variable per bin ``[lo, hi)``, 1.0 on the days the
    temperature lies in the bin, 0.0 otherwise and NaN where ``tas`` is NaN.  Aggregated with
    ``time_groups="year"`` it gives the (weighted) number of days per year each region spends in the bin.

    Same conventions as :func:`tas_poly` (reads ``ds["tas"]`` in K, leap years removed, at most 365
    steps, ``time`` as ``YYYYDDD``), so the two can be swapped in a pipeline.  A gridcell-day lies in a bin
    when ``lo <= tas - 273.15 < hi``, the value widened to float64 before the subtraction.  ``edges``:
    K+1 strictly increasing values in degrees C for K bins; the first may be ``-inf`` and the last
    ``+inf``.  ``varname``: a prefix (variables ``"{varname}_{k}"``) or a list of K names.  Contiguous
    bins of one ``tas`` are fused into one pass per 4 bins when aggregated.
    """
    e = _bin_edges(edges)
    K = e.size - 1
    names = ["{}_{}".format(varname, k) for k in range(K)] if isinstance(varname, str) else list(varname)
    if len(names) != K:
        raise ValueError("{} edges give {} bins, but {} names were given".format(e.size, K, len(names)))
    like = ds
    ds = from_any(ds)

    ds1, tas = _daily_tas_365(ds)

    for lo, hi, name in zip(e[:-1], e[1:], names):
        description = (
            """
            Days with daily average temperature (degrees C) in [{lo:g}, {hi:g})

            1 on a day whose average temperature lies in the bin, 0 otherwise;
            summed over a year, the number of days per year in the bin.

            Leap years are removed before counting days (uses a 365 day
            calendar).
            """.format(lo=lo, hi=hi)
        ).strip()
        attrs = {"units": "days", "bin_lower": float(lo), "bin_upper": float(hi),
                 "long_title": description.splitlines()[0], "description": description,
                 "variable": name}
        # do transformation: lo <= tas - 273.15 < hi, deferred
        ds1._vars[name] = Variable(tas.dims, None, attrs, None,
                                   Deferred("bins", (273.15, float(lo), float(hi)), (tas,)))
    return to_like(ds1, like)


def _rcspline_knots(knots):
    """``knots`` as a float64 array of 3 to 7 finite, strictly increasing values."""
    k = np.asarray(knots, dtype=np.float64)
    if k.ndim != 1 or not 3 <= k.size <= 7:
        raise ValueError("knots must be a 1-D sequence of 3 to 7 values, got {!r}".format(knots))
    if not np.isfinite(k).all() or not (np.diff(k) > 0).all():
        raise ValueError("knots must be finite and strictly increasing: {!r}".format(knots))
    return k


def tas_rcspline(ds, knots, varname="tas_rcspline"):
    """
    Restricted (natural) cubic spline terms of daily average temperature (degrees C): one variable per
    basis function of the knots ``k_1 < ... < k_n`` (3 <= n <= 7, degrees C), n - 1 in all.  With
    ``d = tas - 273.15`` (the value widened to float64 before the subtraction) and
    ``c(k) = max(d - k, 0)**3``::

        B_0 = d                                                               (units C)
        B_i = c(k_i) - c(k_{n-1}) (k_n - k_i) / (k_n - k_{n-1})
                     + c(k_n) (k_{n-1} - k_i) / (k_n - k_{n-1}),   1 <= i <= n-2   (units C^3)

    Each ``B_i`` is cubic between the knots and linear below ``k_1`` and above ``k_n``; NaN stays NaN, and
    ``tas = +inf`` gives NaN for ``i >= 1``.  This is Harrell's unnormalised form: his default
    normalisation divides ``B_i`` (i >= 1) by ``(k_n - k_1)**2``, and since aggregation is linear that
    scale can be applied to the aggregated values.

    Same conventions as :func:`tas_poly` (reads ``ds["tas"]`` in K, leap years removed, at most 365
    steps, ``time`` as ``YYYYDDD``).  ``varname``: a prefix (variables ``"{varname}_{i}"``, ``i = 0`` the
    linear term) or a list of n - 1 names.  The terms of one ``tas`` are fused into one pass per 4 terms
    when aggregated, sharing the cubes of the two last knots.
    """
    k = _rcspline_knots(knots)
    n = k.size
    names = ["{}_{}".format(varname, i) for i in range(n - 1)] if isinstance(varname, str) else list(varname)
    if len(names) != n - 1:
        raise ValueError("{} knots give {} terms, but {} names were given".format(n, n - 1, len(names)))
    like = ds
    ds1, tas = _daily_tas_365(from_any(ds))

    knot_list = ", ".join("{:g}".format(v) for v in k)
    for i, name in enumerate(names):
        description = (
            """
            {what} of daily average temperature (degrees C)

            Restricted cubic spline basis of the knots ({knots}) degrees C,
            unnormalised: cubic between the knots, linear outside them.

            Leap years are removed before counting days (uses a 365 day
            calendar).
            """.format(what="Linear term" if i == 0 else "Restricted cubic spline term {}".format(i),
                       knots=knot_list)
        ).strip()
        attrs = {"units": "C" if i == 0 else "C^3", "knots": [float(v) for v in k], "rcspline_term": i,
                 "long_title": description.splitlines()[0], "description": description,
                 "variable": name}
        # do transformation: B_i(tas - 273.15), deferred
        ds1._vars[name] = Variable(tas.dims, None, attrs, None,
                                   Deferred("rcspline", (273.15, float(i)) + tuple(float(v) for v in k), (tas,)))
    return to_like(ds1, like)


def ordinal(n):
    """Converts numbers into ordinal strings"""
    return "%d%s" % (n, "tsnrhtdd"[(n // 10 % 10 != 1) * (n % 10 < 4) * n % 10:: 4])
