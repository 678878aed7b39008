"""
Handy functions for standardizing the format of climate data
(mirror of ``/root/reference/climate_toolbox/utils/utils.py:10-80``).

The two functions on the aggregation path -- :func:`convert_lons_split`
(reference ``:33-40``) and :func:`remove_leap_days` (``:77-80``) -- copy the whole
dataset in the reference.  Here they only relabel / record positions (lazy takes
of ``_xr.Variable``); the plan builder folds the lon permutation into CSR column
indices and the kernel reads the time positions as an index list.
"""
from __future__ import annotations

import numpy as np

from .._xr import Dataset, DataArray, Deferred, Variable, from_any, to_like

__all__ = ["convert_kelvin_to_celsius", "convert_lons_mono", "convert_lons_split",
           "rename_coords_to_lon_and_lat", "rename_coords_to_longitude_and_latitude",
           "remove_leap_days", "resample_daily", "season_boundaries", "get_daily_growing_season_mask", "GrowingSeasonMask"]


def convert_kelvin_to_celsius(df, temp_name):
    """Convert Kelvin to Celsius (reference ``:10-20``).  The subtraction is
    deferred and fuses into the aggregation kernel as ``(x - 273.15)^1``."""
    like = df
    ds = from_any(df)
    var = ds._vars[temp_name]
    attrs = dict(var.attrs)
    attrs.update(units="C", valid_min=-108.78788, valid_max=62.02828)
    src = var if var.deferred is None else Variable(var.dims, var.values, var.attrs)
    out = ds.copy()
    out._vars[temp_name] = Variable(var.dims, None, attrs, None,
                                    Deferred("poly", (273.15, 1.0), (src,)))
    return to_like(out, like)


def _relabel_and_sort(ds, lon_name, fn):
    like = ds
    ds = from_any(ds)
    if lon_name not in ds._coords:
        raise KeyError(lon_name)
    new = fn(np.asarray(ds._coords[lon_name].values))
    out = ds.copy()
    c = out._coords[lon_name]
    out._coords[lon_name] = Variable(c.dims, new, c.attrs)
    # ds.sel(lon=np.sort(lon)): exact-label orthogonal selection -> lazy take
    return to_like(out.sel(**{lon_name: np.sort(new)}), like)


def convert_lons_mono(ds, lon_name="longitude"):
    """Convert longitude from -180-180 to 0-360 (reference ``:23-30``)"""
    return _relabel_and_sort(ds, lon_name, lambda lon: lon % 360)


def convert_lons_split(ds, lon_name="longitude"):
    """Convert longitude from 0-360 to -180-180 (reference ``:33-40``)"""
    return _relabel_and_sort(ds, lon_name, lambda lon: (lon + 180) % 360 - 180)


def _rename(ds, pairs):
    like = ds
    ds = from_any(ds)
    for old_names, new in pairs:
        for old in old_names:
            if old in ds.coords:
                ds = ds.rename({old: new})
                break
    if "z" in ds.coords:
        ds = ds.drop("z").squeeze()
    return to_like(ds, like)


def rename_coords_to_lon_and_lat(ds):
    """Rename Dataset spatial coord names to: lat, lon (reference ``:43-57``)"""
    return _rename(ds, ((("latitude",), "lat"), (("longitude", "long"), "lon")))


def rename_coords_to_longitude_and_latitude(ds):
    """Rename Dataset spatial coord names to: latitude, longitude (reference ``:60-74``)"""
    return _rename(ds, ((("lat",), "latitude"), (("lon", "long"), "longitude")))


def remove_leap_days(ds):
    """Drop Feb 29 steps (reference ``:77-80``) as a lazy time take."""
    like = ds
    ds = from_any(ds)
    keep = ~((ds["time.month"].values == 2) & (ds["time.day"].values == 29))
    return to_like(ds.loc[{"time": keep}], like)


_DAILY_HOW = ("mean", "min", "max")


def _steps_per_day(time):
    """Steps per day of a datetime64 time axis made of whole, consecutive calendar days that all hold the
    same steps in the same order; ``ValueError`` otherwise.  Returns ``(S, days)``."""
    t = np.asarray(time)
    if not np.issubdtype(t.dtype, np.datetime64):
        raise ValueError("resample_daily needs a datetime64 'time' coordinate, got {}".format(t.dtype))
    if t.size == 0:
        raise ValueError("resample_daily: the time axis is empty")
    if np.isnat(t).any():
        raise ValueError("resample_daily: the time axis holds NaT")
    days = t.astype("datetime64[D]")
    starts = np.flatnonzero(np.r_[True, days[1:] != days[:-1]])
    uniq = days[starts]
    if (np.diff(uniq) != np.timedelta64(1, "D")).any():
        raise ValueError("resample_daily: every calendar day from {} to {} must be present once, as one run of "
                         "steps".format(uniq.min(), uniq.max()))
    counts = np.diff(np.r_[starts, t.size])
    S = int(counts[0])
    if (counts != S).any():
        bad = int(np.flatnonzero(counts != S)[0])
        raise ValueError("resample_daily: day {} has {} steps, day {} has {}".format(uniq[0], S, uniq[bad], counts[bad]))
    offs = (t - days).reshape(-1, S)
    if S > 1 and (np.diff(offs[0]) <= np.timedelta64(0)).any():
        raise ValueError("resample_daily: the steps of day {} are not in increasing order".format(uniq[0]))
    if (offs != offs[0]).any():
        bad = int(np.flatnonzero((offs != offs[0]).any(axis=1))[0])
        raise ValueError("resample_daily: day {} holds other steps than day {}".format(uniq[bad], uniq[0]))
    return S, uniq


def resample_daily(ds, how="mean"):
    """Daily mean, minimum or maximum of sub-daily (hourly, 3- or 6-hourly) data, as xarray's
    ``ds.resample(time="1D").mean()`` / ``.min()`` / ``.max()`` with ``skipna=True``.

    ``ds``: a Dataset or DataArray whose ``time`` coordinate is datetime64 and consists of complete,
    consecutive calendar days that hold the same S steps in the same order (``ValueError`` otherwise).
    Variables over ``(time, lat, lon)`` become deferred daily variables over ``(time, lat, lon)`` with
    ``time`` as the day (``datetime64[D]``); other variables without ``time`` are kept.  The reduction runs
    on the GPU per gridcell while the referenced gridcells are packed for aggregation, so the daily grid is
    never built: the result feeds ``tas_poly``, ``tas_bins``, ``tas_rcspline``, ``snyder_edd`` /
    ``snyder_gdd``, ``remove_leap_days`` and ``weighted_aggregate_grid_to_regions`` directly, and
    ``.values`` computes it for the whole grid.

    * ``"mean"``: each step widened to float64 and summed in step order, NaN steps skipped, divided by the
      number of non-NaN steps (NaN for a day without one); float64.
    * ``"min"`` / ``"max"``: NaN steps skipped (NaN for a day without a value); exact, in the source dtype.

    Attributes carry over, plus ``cell_methods = "time: <how>"``.  Sources over ``(lat, lon, time)`` raise
    ``NotImplementedError``."""
    if how not in _DAILY_HOW:
        raise ValueError("how={!r}: expected one of {}".format(how, _DAILY_HOW))
    like = ds
    ds = from_any(ds)
    single = isinstance(ds, DataArray)
    if single:
        ds = Dataset({ds.name or "_da": ds.variable}, coords=ds._coords)
    if "time" not in ds._coords:
        raise ValueError("resample_daily needs a 'time' coordinate")
    S, days = _steps_per_day(ds._coords["time"].values)
    out = Dataset()
    for k, c in ds._coords.items():
        if "time" not in c.dims:
            out._coords[k] = c
    out._coords["time"] = Variable(("time",), days, ds._coords["time"].attrs)
    for name, var in ds._vars.items():
        if "time" not in var.dims:
            out._vars[name] = var
            continue
        if var.dims == ("lat", "lon", "time") or var.dims == ("lon", "lat", "time"):
            raise NotImplementedError("resample_daily: {!r} is over {}; sub-daily sources must be over "
                                      "(time, lat, lon)".format(name, var.dims))
        if var.dims != ("time", "lat", "lon"):
            raise ValueError("resample_daily: {!r} is over {}, expected (time, lat, lon)".format(name, var.dims))
        if var.deferred is not None:
            raise ValueError("resample_daily: {!r} is a deferred variable, not stored data".format(name))
        # the kernel reads whole days from the first step on: a time take must be one run of steps
        t0 = 0
        takes = dict(var.takes)
        pos = takes.pop("time", None)
        if pos is not None:
            if len(pos) and not np.array_equal(pos, np.arange(pos[0], pos[0] + len(pos))):
                raise NotImplementedError("resample_daily: {!r} selects time steps out of physical order".format(name))
            t0 = int(pos[0]) if len(pos) else 0
        src = Variable(var.dims, var.physical, var.attrs, takes)
        attrs = dict(var.attrs)
        attrs["cell_methods"] = "time: {}".format(how)
        out._vars[name] = Variable(var.dims, None, attrs, None,
                                   Deferred("daily", (how, S, t0, np.arange(len(days), dtype=np.int64)), (src,)))
    if single:
        name = next(iter(out._vars))
        res = DataArray._wrap(out._vars[name], out._coords_for(out._vars[name].dims), like.name)
        return res
    return to_like(out, like)


# ---------------------------------------------------------------------------
# growing-season mask (reference ``:83-153``), fused into the aggregation
# ---------------------------------------------------------------------------
def _growing_days_arrays(growing_days):
    """(planting [lat][lon], harvest [lat][lon], latitude, longitude) of a crop-calendar Dataset: data
    variable ``variable`` over (z, latitude, longitude) with z = 1 (planting day) and 2 (harvest day)."""
    gd = from_any(growing_days)
    v = gd["variable"]
    arr = np.asarray(v.transpose("z", "latitude", "longitude").values, dtype=np.float64)
    z = list(np.asarray(gd["z"].values).tolist())
    return (arr[z.index(1)], arr[z.index(2)], np.asarray(gd["latitude"].values, dtype=np.float64),
            np.asarray(gd["longitude"].values, dtype=np.float64))


def season_boundaries(growing_days):
    """Returns the sorted start and end date of growing season (reference ``:83-116``).

    The crop calendar's longitudes are on 0..360: they are shifted by -180 and the grid is sorted by
    longitude (the reference does the shift in place on the caller's Dataset; this does not).
    Returns ``(min_day, max_day)`` DataArrays over (latitude, longitude): the two ``z`` planes sorted
    per gridcell (NaN last, like ``np.sort``)."""
    plant, harv, lat, lon = _growing_days_arrays(growing_days)
    lon = lon - 180
    order = np.argsort(lon, kind="stable")
    lon = lon[order]
    both = np.sort(np.stack([plant[:, order], harv[:, order]], axis=2), axis=2)
    coords = {"latitude": lat, "longitude": lon}
    return (DataArray(both[:, :, 0], dims=("latitude", "longitude"), coords=coords),
            DataArray(both[:, :, 1], dims=("latitude", "longitude"), coords=coords))


class GrowingSeasonMask:
    """What :func:`get_daily_growing_season_mask` returns: the lat x lon x time mask of the reference
    in factored form -- a (first day, last day, wrap) triple per gridcell and the day of year of every
    time step.  Pass it as ``season_mask=`` to ``weighted_aggregate_grid_to_regions``: the gate is
    applied inside the kernel (a gridcell-day outside its season adds nothing to the weighted sum,
    exactly like multiplying the data by the mask, whose 0 and NaN both vanish in the skip-NaN sum).
    ``.values`` materialises the dense (lat, lon, time) array of 1 / 0 / NaN the reference returns."""

    dims = ("lat", "lon", "time")

    def __init__(self, lat, lon, time, first, last, wrap, missing):
        self.lat, self.lon, self.time = lat, lon, time
        self.first, self.last, self.wrap, self.missing = first, last, wrap, missing

    @property
    def day_of_year(self):
        return _day_of_year(self.time)

    @property
    def shape(self):
        return (len(self.lat), len(self.lon), len(self.time))

    def gate_words(self):
        """uint32 [lat][lon]: first | last << 9 | wrap << 18 (include/ctb.h)."""
        return (self.first.astype(np.uint32) | (self.last.astype(np.uint32) << np.uint32(9)) |
                (self.wrap.astype(np.uint32) << np.uint32(18)))

    @property
    def values(self):
        import torch
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        doy = torch.as_tensor(self.day_of_year.astype(np.int64), device=dev)[None, None, :]
        first = torch.as_tensor(self.first.astype(np.int64), device=dev)[:, :, None]
        last = torch.as_tensor(self.last.astype(np.int64), device=dev)[:, :, None]
        wrap = torch.as_tensor(self.wrap, device=dev)[:, :, None]
        on = ((doy >= first) & (doy <= last)) != wrap
        out = on.to(torch.float64)
        out[torch.as_tensor(self.missing, device=dev)] = float("nan")
        return out.cpu().numpy()


def _day_of_year(time):
    t = np.asarray(time)
    if np.issubdtype(t.dtype, np.datetime64):
        d = t.astype("datetime64[D]")
        return ((d - d.astype("datetime64[Y]").astype("datetime64[D]")).astype(np.int64) + 1).astype(np.int32)
    if np.issubdtype(t.dtype, np.integer):       # the YYYYDDD integers tas_poly writes
        return (t % 1000).astype(np.int32)
    import pandas as pd
    return pd.DatetimeIndex(t).dayofyear.values.astype(np.int32)


def get_daily_growing_season_mask(lat, lon, time, growing_days_path):
    """
    Constructs a mask for days in the within calendar growing season (reference ``:119-153``).

    Parameters
    ----------
    lat, lon, time : coordinate arrays (or DataArray coords) of the climate data
    growing_days_path : str or Dataset
        the crop calendar: variable ``variable`` over (z, latitude, longitude), z = 1 planting day,
        z = 2 harvest day, longitudes on 0..360 (a path needs a netCDF reader, which this image does
        not have; pass the Dataset)

    Returns
    -------
    GrowingSeasonMask
        over lat x lon x time: 1 inside the season, 0 outside; seasons that wrap around the new year
        (harvest < planting) are the complement of [min, max]; a missing harvest day gives 1 everywhere,
        a missing planting day NaN -- the reference's ``where / fillna(1 - mask) / where`` chain.
    """
    if isinstance(growing_days_path, str):
        raise NotImplementedError("reading netCDF needs xarray's backends; pass the crop-calendar Dataset")
    plant, harv, _, _ = _growing_days_arrays(growing_days_path)
    min_day, max_day = season_boundaries(growing_days_path)
    glat = np.asarray(min_day.coords["latitude"].values, dtype=np.float64)
    glon = np.asarray(min_day.coords["longitude"].values, dtype=np.float64)
    lon_src = np.asarray(from_any(growing_days_path)["longitude"].values, dtype=np.float64) - 180
    order = np.argsort(lon_src, kind="stable")
    plant, harv = plant[:, order], harv[:, order]
    mn, mx = np.asarray(min_day.values), np.asarray(max_day.values)
    with np.errstate(invalid="ignore"):
        # day-of-year comparisons against (possibly fractional) day numbers, as integers:
        # doy >= mn <=> doy >= ceil(mn);  doy <= mx <=> doy <= floor(mx);  a NaN bound is never met
        first = np.where(np.isnan(mn), 511, np.clip(np.ceil(mn), 0, 511)).astype(np.int32)
        last = np.where(np.isnan(mx), 0, np.clip(np.floor(mx), 0, 511)).astype(np.int32)
        empty = np.isnan(mn) | np.isnan(mx)
        first = np.where(empty, 511, first)
        last = np.where(empty, 0, last)
        wrap = ~(harv >= plant)                  # harvest < planting, or either missing: fillna(1 - mask)
    missing = np.isnan(plant)
    wrap = wrap & ~missing                       # planting missing: NaN, never counted
    # the data's grid: every (lat, lon) label must exist in the calendar (exact match, like xarray alignment)
    lat = np.asarray(getattr(lat, "values", lat), dtype=np.float64)
    lon = np.asarray(getattr(lon, "values", lon), dtype=np.float64)
    time = np.asarray(getattr(time, "values", time))
    ii = _match(glat, lat, "lat")
    jj = _match(glon, lon, "lon")
    sel = np.ix_(ii, jj)
    return GrowingSeasonMask(lat, lon, time, first[sel], last[sel], wrap[sel], missing[sel])


def _match(have, want, name):
    order = np.argsort(have, kind="stable")
    pos = np.searchsorted(have[order], want)
    pos = np.clip(pos, 0, len(have) - 1)
    idx = order[pos]
    if not np.array_equal(have[idx], want):
        raise KeyError("not all {} values of the data are in the crop calendar".format(name))
    return idx
