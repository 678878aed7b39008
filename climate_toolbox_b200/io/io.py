"""Loaders that put climate data into the form the aggregation path requires
(mirror of ``/root/reference/climate_toolbox/io/io.py:6-58``)."""
from __future__ import annotations

import numpy as np

from .._xr import DataArray, Dataset, Deferred, Variable, from_any, to_like
from ..utils.utils import rename_coords_to_lon_and_lat, convert_lons_split

__all__ = ["standardize_climate_data", "load_bcsd", "load_gmfd", "load_best", "decode_packed"]

_PACKING = ("scale_factor", "add_offset", "_FillValue", "missing_value")


def _decoded_dtype(attrs):
    """xarray's float type for a 16-bit integer source: float32 when ``scale_factor`` is float32 and
    ``add_offset`` is absent or float32, or when neither is present; float64 otherwise."""
    f32 = np.dtype("float32")
    if "scale_factor" not in attrs and "add_offset" not in attrs:
        return f32
    if ("scale_factor" in attrs and np.asarray(attrs["scale_factor"]).dtype == f32 and
            ("add_offset" not in attrs or np.asarray(attrs["add_offset"]).dtype == f32)):
        return f32
    return np.dtype("float64")


def _scalar_attr(name, attrs, default):
    v = np.asarray(attrs.get(name, default))
    if v.size != 1:
        raise ValueError("{} must be one value, got {!r}".format(name, attrs[name]))
    v = float(v.reshape(-1)[0])
    if not np.isfinite(v):
        raise ValueError("{} must be finite, got {!r}".format(name, attrs[name]))
    return v


def _fill_values(name, attrs):
    """The distinct raw fill values of ``_FillValue`` and ``missing_value``, as int16."""
    fills = []
    for key in ("_FillValue", "missing_value"):
        if key not in attrs:
            continue
        a = np.atleast_1d(np.asarray(attrs[key])).reshape(-1)
        if a.dtype.kind not in "iu" or (a.size and (a.min() < -32768 or a.max() > 32767)):
            raise ValueError("decode_packed: {}'s {} is {!r}, not int16 integers".format(name, key, attrs[key]))
        fills.extend(int(v) for v in a)
    fills = sorted(set(fills))
    if len(fills) > 4:
        raise ValueError("decode_packed: {} has {} fill values, at most 4 are supported".format(name, len(fills)))
    return tuple(fills)


def _decode_var(name, var):
    attrs = var.attrs
    if not any(k in attrs for k in _PACKING) or var.dtype.kind == "f":
        return var
    if var.deferred is not None:
        raise ValueError("decode_packed: {!r} is a deferred variable, not stored data".format(name))
    if var.dtype != np.dtype("int16"):
        raise ValueError("decode_packed: {!r} is packed as {}; only int16 (netCDF short) is supported".format(
            name, var.dtype))
    if "_Unsigned" in attrs:
        raise ValueError("decode_packed: {!r} has _Unsigned; unsigned packing is not supported".format(name))
    if "time" in var.dims and set(var.dims) == {"time", "lat", "lon"} and var.dims != ("time", "lat", "lon"):
        raise NotImplementedError("decode_packed: {!r} is over {}; packed sources must be over (time, lat, lon)".format(
            name, var.dims))
    if var.dims != ("time", "lat", "lon"):
        raise ValueError("decode_packed: {!r} is over {}, expected (time, lat, lon)".format(name, var.dims))
    scale = _scalar_attr("scale_factor", attrs, 1.0)
    offset = _scalar_attr("add_offset", attrs, 0.0)
    fills = _fill_values(name, attrs)
    D = _decoded_dtype(attrs)
    keep = {k: v for k, v in attrs.items() if k not in _PACKING}
    return Variable(var.dims, None, keep, None, Deferred("decode", (scale, offset, fills, D), (var,)))


def decode_packed(ds):
    """CF-packed 16-bit sources decoded on the GPU, the way ``xr.open_dataset`` decodes them by default.

    ``ds``: a Dataset or DataArray (with real xarray: opened with ``mask_and_scale=False``).  Every ``(time, lat,
    lon)`` int16 variable that carries ``scale_factor``, ``add_offset``, ``_FillValue`` or ``missing_value``
    becomes a deferred variable: the raw values stay where they are (host, pinned or device memory), and the
    aggregation's GPU pack decodes only the referenced gridcells -- a quarter of the bytes of a float64 source
    cross PCIe.  A raw value ``r`` decodes to NaN when it is a fill value, else to
    ``r.astype(D) * D(scale_factor) + D(add_offset)`` (two rounded operations), with a missing ``scale_factor`` 1
    and a missing ``add_offset`` 0.  ``D`` is xarray's choice for 16-bit integers: float32 when ``scale_factor`` is
    float32 and ``add_offset`` absent or float32, or when neither is present; float64 otherwise (ERA5's float64
    attributes).  Downstream everything sees exactly what a float source of dtype ``D`` holding the decoded values
    gives: ``tas_poly`` / ``tas_bins`` / ``tas_rcspline`` / ``snyder_edd`` / ``snyder_gdd``,
    ``convert_kelvin_to_celsius``, ``resample_daily`` and ``subdaily_*`` (reduced while decoding), lazy
    ``remove_leap_days`` and longitude rolls, ``time_groups=``, ``season_mask=``, the multi-weight entry and
    ``.values`` (the whole grid).

    The packing attributes leave ``attrs`` (xarray moves them to ``.encoding``); other attributes stay.  Float and
    unpacked variables pass through unchanged; int16 variables that are not passed through here keep being read
    as raw numbers.  ``ValueError`` for a packed variable that is not int16, ``_Unsigned``, fill values that are
    not int16 integers, or more than 4 of them; sources over ``(lat, lon, time)`` raise ``NotImplementedError``."""
    like = ds
    ds = from_any(ds)
    if isinstance(ds, DataArray):
        return DataArray._wrap(_decode_var(ds.name, ds.variable), ds._coords, ds.name)
    out = ds.copy()
    for name, var in ds._vars.items():
        out._vars[name] = _decode_var(name, var)
    return to_like(out, like)


def standardize_climate_data(ds):
    """
    Read climate data and standardize units to lon and lat, lon to -180 to 180
    (reference ``io.py:6-24``).  No data is moved: coordinates are relabelled and
    the lon sort is recorded as a lazy permutation.
    """
    ds = rename_coords_to_lon_and_lat(ds)
    ds = convert_lons_split(ds, lon_name="lon")
    return ds


def load_bcsd(fp, varname, lon_name="lon", broadcast_dims=("time",)):
    """
    Read and prepare climate data (reference ``io.py:27-58``).

    ``fp`` may be a Dataset (this package's, holding numpy arrays or CUDA tensors, or
    ``xarray``'s) -- passed through like the reference's ``hasattr(fp, "sel_points")``
    branch -- or a netCDF path, which needs ``xarray`` (not part of this image; netCDF
    decode is outside the hot path).  ``varname``, ``lon_name`` and ``broadcast_dims``
    are accepted and ignored, as in the reference.
    """
    if isinstance(fp, Dataset) or hasattr(fp, "data_vars"):
        ds = fp
    else:
        try:
            import xarray as xr
        except ImportError as e:  # pragma: no cover
            raise ImportError("reading netCDF paths needs xarray; pass an in-memory Dataset") from e
        with xr.open_dataset(fp) as ds:  # pragma: no cover
            ds.load()
    return standardize_climate_data(ds)


def load_gmfd(fp, varname, lon_name="lon", broadcast_dims=("time",)):
    pass  # stub in the reference too (io.py:61-62)


def load_best(fp, varname, lon_name="lon", broadcast_dims=("time",)):
    pass  # stub in the reference too (io.py:65-66)
