"""Minimal named-array containers (``Dataset`` / ``DataArray``) for the hot path.

The reference API takes and returns ``xarray`` objects
(``/root/reference/climate_toolbox/aggregations/aggregations.py:87-124``), but
``xarray`` is not installed in this image (nor on the GPU box).  This module is
the small subset of that interface which the reference's hot path and its tests
touch, with two additions that let host-side "data movement" in the reference
become index metadata here:

* **lazy takes** -- an orthogonal ``sel`` / ``isel`` / boolean ``loc`` along a
  dim (``utils.convert_lons_split``'s lon sort, ``utils.remove_leap_days``'s
  time mask) does not move data; it records ``positions`` for that dim.  The
  aggregation planner folds those into CSR column indices / the time-index
  list (SURVEY.md section 3.2).
* **deferred transforms** -- ``tas_poly`` / ``tas_bins`` / ``tas_rcspline`` / ``snyder_edd`` / ``snyder_gdd`` return
  variables that remember (kind, params, sources); aggregation fuses them into
  the gather kernel, ``.values`` materialises them with the pointwise CUDA
  kernel.

Data may be ``numpy`` (host) or ``torch`` CUDA tensors (device-resident).
When real ``xarray`` is importable, :func:`from_any` / :func:`to_like` convert
at the boundary so real Datasets work too.
"""
from __future__ import annotations

import numpy as np
import pandas as pd

try:  # torch is plumbing: device memory + streams
    import torch
except Exception:  # pragma: no cover
    torch = None

__all__ = ["Dataset", "DataArray", "Variable", "Deferred", "from_any", "to_like", "where"]


def _is_torch(a):
    return torch is not None and isinstance(a, torch.Tensor)


def _as_data(a):
    if _is_torch(a):
        return a
    if isinstance(a, (DataArray, Variable)):
        return a.values
    return np.asarray(a)


class Deferred:
    """A pointwise gridcell transform that has not been evaluated yet.

    kind   : "poly" | "bins" | "rcspline" | "edd" | "gdd" | "reindex" (pointwise lat/lon gather,
             params = (materialise closure, origin Dataset)) | "daily" (daily reduction of a sub-daily
             (time, lat, lon) source, params = (how, steps per day, first step, physical day of every day);
             how = "mean" | "min" | "max", or the daily mean of a per-step transform: ("edd", e) |
             ("gdd", lo, hi) | ("bins", lo, hi)) | "decode" (a CF-packed int16 (time, lat, lon) source decoded on
             the GPU, ``io.decode_packed``; params = (scale, offset, fill values, D), D the decoded numpy dtype;
             takes compose onto the raw source)
    params : tuple of floats (poly: (offset, power); bins: (offset, lo, hi); rcspline: (offset, term,
             k_1, ..., k_n); edd: (threshold,); gdd: (threshold_low, threshold_high))
    sources: tuple of :class:`Variable` (poly / bins / rcspline: (tas,); edd/gdd: (tasmin, tasmax))
    """

    __slots__ = ("kind", "params", "sources", "shape")

    def __init__(self, kind, params, sources, shape=None):
        self.kind, self.params, self.sources = kind, tuple(params), tuple(sources)
        self.shape = None if shape is None else tuple(shape)


class Variable:
    """dims + physical data + attrs + lazy per-dim takes (+ optional deferred op)."""

    __slots__ = ("dims", "_data", "attrs", "takes", "deferred")

    def __init__(self, dims, data, attrs=None, takes=None, deferred=None):
        if isinstance(dims, str):
            dims = (dims,)
        self.dims = tuple(dims)
        self._data = data
        self.attrs = dict(attrs or {})
        self.takes = dict(takes or {})
        self.deferred = deferred
        if deferred is None and data is not None and len(self.dims) != data.ndim:
            raise ValueError("dims {} do not match data of rank {}".format(self.dims, data.ndim))

    # -- structure -------------------------------------------------------
    @property
    def physical(self):
        """Underlying buffer, BEFORE lazy takes are applied (None if deferred)."""
        return self._data

    @property
    def shape(self):
        if self.deferred is not None:
            d = self.deferred
            if d.kind == "daily":
                return (len(d.params[3]),) + d.sources[0].shape[1:]
            return d.shape or d.sources[0].shape
        phys = tuple(self._data.shape)
        return tuple(len(self.takes[d]) if d in self.takes else phys[i]
                     for i, d in enumerate(self.dims))

    @property
    def ndim(self):
        return len(self.dims)

    @property
    def dtype(self):
        if self.deferred is not None:
            d = self.deferred
            if d.kind == "decode":
                return np.dtype(d.params[3])
            return d.sources[0].dtype if d.kind == "daily" and d.params[0] in ("min", "max") else np.dtype("float64")
        d = self._data.dtype
        return np.dtype(str(d).replace("torch.", "")) if _is_torch(self._data) else d

    def positions(self, dim):
        """Physical positions along ``dim`` (None = identity)."""
        return self.takes.get(dim)

    def with_take(self, dim, pos):
        """Compose an orthogonal take along ``dim`` (no data movement)."""
        pos = np.asarray(pos)
        if pos.dtype == bool:
            pos = np.flatnonzero(pos)
        pos = pos.astype(np.int64)
        if self.deferred is not None and self.deferred.kind == "reindex":
            return Variable(self.dims, self.values, self.attrs).with_take(dim, pos)
        if self.deferred is not None and self.deferred.kind == "daily":
            d = self.deferred
            if dim == self.dims[0]:     # a take of days: the physical day of every kept day
                new = Deferred(d.kind, d.params[:3] + (d.params[3][pos],), d.sources)
            else:
                new = Deferred(d.kind, d.params, tuple(s.with_take(dim, pos) for s in d.sources))
            return Variable(self.dims, None, self.attrs, None, new)
        if self.deferred is not None:
            d = self.deferred
            new = Deferred(d.kind, d.params, tuple(s.with_take(dim, pos) for s in d.sources))
            return Variable(self.dims, None, self.attrs, None, new)
        takes = dict(self.takes)
        takes[dim] = takes[dim][pos] if dim in takes else pos
        return Variable(self.dims, self._data, self.attrs, takes)

    # -- materialisation -------------------------------------------------
    @property
    def values(self):
        if self.deferred is not None:
            from . import _engine  # pointwise CUDA kernel; no CPU fallback
            return _engine.materialize_deferred(self)
        a = self._data
        if _is_torch(a):
            for ax, d in enumerate(self.dims):
                if d in self.takes:
                    a = a.index_select(ax, torch.as_tensor(self.takes[d], device=a.device))
            return a.detach().cpu().numpy()
        for ax, d in enumerate(self.dims):
            if d in self.takes:
                a = np.take(a, self.takes[d], axis=ax)
        return a

    def copy(self):
        return Variable(self.dims, self._data, self.attrs, self.takes, self.deferred)


def _coord_var(name, value):
    if isinstance(value, DataArray):
        return value.variable
    if isinstance(value, Variable):
        return value
    if isinstance(value, tuple):
        return Variable(*value)
    arr = np.asarray(value)
    if arr.ndim == 0:
        return Variable((), arr)
    return Variable((name,), arr)


class _Coords:
    """Mapping view over a container's coordinate variables."""

    def __init__(self, owner):
        self._o = owner

    def __contains__(self, k):
        return k in self._o._coords

    def __iter__(self):
        return iter(self._o._coords)

    def __len__(self):
        return len(self._o._coords)

    def keys(self):
        return self._o._coords.keys()

    def __getitem__(self, k):
        return DataArray._wrap(self._o._coords[k], self._o._coords_for(self._o._coords[k].dims), k)

    def __setitem__(self, k, v):
        self._o._coords[k] = _coord_var(k, v)

    def __repr__(self):
        return "Coordinates({})".format(list(self._o._coords))


class _Loc:
    def __init__(self, owner):
        self._o = owner

    def __getitem__(self, key):
        if not isinstance(key, dict):
            raise TypeError("only dict-style .loc is supported")
        out = self._o
        for dim, k in key.items():
            k = _as_data(k)
            if getattr(k, "dtype", None) == bool:
                out = out.isel(**{dim: np.flatnonzero(k)})
            else:
                out = out.sel(**{dim: k})
        return out


class _Base:
    """Shared indexing logic of Dataset and DataArray."""

    def _coords_for(self, dims):
        return {k: v for k, v in self._coords.items() if set(v.dims) <= set(dims)}

    @property
    def coords(self):
        return _Coords(self)

    @property
    def loc(self):
        return _Loc(self)

    def _label_positions(self, dim, labels):
        if dim not in self._coords:
            raise KeyError(dim)
        index = pd.Index(self._coords[dim].values)
        labels = np.asarray(_as_data(labels))
        scalar = labels.ndim == 0
        pos = index.get_indexer(np.atleast_1d(labels))
        if (pos < 0).any():
            raise KeyError("not all values found in index {!r}".format(dim))
        return (pos[0] if scalar else pos), scalar

    def sel(self, **indexers):
        """Exact-label selection (no ``method=``): orthogonal for plain arrays,
        pointwise when indexers are DataArrays sharing a new dim."""
        das = [v for v in indexers.values() if isinstance(v, DataArray) and v.ndim == 1]
        if das and len(das) == len(indexers) and len({d.dims for d in das}) == 1 \
                and das[0].dims[0] not in indexers:
            return self._sel_pointwise(indexers, das[0].dims[0])
        pos = {}
        for dim, lab in indexers.items():
            pos[dim], _ = self._label_positions(dim, lab)
        return self.isel(**pos)


class DataArray(_Base):
    def __init__(self, data=None, coords=None, dims=None, name=None, attrs=None):
        if isinstance(data, Variable):
            self.variable = data
        else:
            data = data if _is_torch(data) else np.asarray(data)
            if dims is None and isinstance(coords, (list, tuple)) and coords \
                    and isinstance(coords[0], tuple):
                dims = tuple(c[0] for c in coords)            # [("time", idx), ...]
                coords = {c[0]: c[1] for c in coords}
            elif dims is None and isinstance(coords, (list, tuple)):
                raise ValueError("dims required")
            if dims is None:
                dims = tuple("dim_{}".format(i) for i in range(data.ndim))
            if isinstance(dims, dict):                         # aggregations.py:65 passes a dict
                dims = tuple(dims)
            if isinstance(coords, (list, tuple)):              # coords=[lat, lon, time] + dims
                coords = dict(zip(dims, coords))
            self.variable = Variable(dims, data, attrs)
        self._coords = {}
        for k, v in (coords or {}).items():
            cv = _coord_var(k, v)
            if set(cv.dims) <= set(self.variable.dims):
                self._coords[k] = cv
        self.name = name

    @classmethod
    def _wrap(cls, variable, coords, name=None):
        out = cls.__new__(cls)
        out.variable, out._coords, out.name = variable, dict(coords), name
        return out

    # -- basics -----------------------------------------------------------
    dims = property(lambda s: s.variable.dims)
    shape = property(lambda s: s.variable.shape)
    ndim = property(lambda s: s.variable.ndim)
    dtype = property(lambda s: s.variable.dtype)
    attrs = property(lambda s: s.variable.attrs)
    values = property(lambda s: s.variable.values)
    data = property(lambda s: s.variable.physical)

    def __len__(self):
        return self.shape[0]

    def __array__(self, dtype=None, copy=None):
        v = self.values
        return v.astype(dtype) if dtype is not None else v

    def __getattr__(self, name):
        if name.startswith("_") or name in ("variable", "name"):
            raise AttributeError(name)
        if name in self._coords:
            return self.coords[name]
        if name in self.variable.attrs:
            return self.variable.attrs[name]
        raise AttributeError(name)

    def __getitem__(self, key):
        if isinstance(key, str):
            if key in self._coords:
                return self.coords[key]
            if "." in key:
                base, comp = key.split(".", 1)
                idx = pd.DatetimeIndex(self._coords[base].values)
                return DataArray(np.asarray(getattr(idx, comp)), dims=self._coords[base].dims,
                                 coords={base: self._coords[base]}, name=comp)
            raise KeyError(key)
        return DataArray(self.values[key])

    def __repr__(self):
        return "<DataArray {} {} {}>".format(self.name or "", dict(zip(self.dims, self.shape)),
                                              "deferred" if self.variable.deferred else self.dtype)

    def item(self, *a):
        return self.values.item(*a)

    def copy(self):
        return DataArray._wrap(self.variable.copy(), self._coords, self.name)

    # -- indexing ---------------------------------------------------------
    def isel(self, **indexers):
        var, coords = self.variable, dict(self._coords)
        for dim, pos in indexers.items():
            pos = np.asarray(_as_data(pos))
            if pos.ndim == 0:
                sub = np.take(self.values, int(pos), axis=self.dims.index(dim))
                rest = tuple(d for d in self.dims if d != dim)
                cs = {k: v for k, v in coords.items() if dim not in v.dims}
                return DataArray(sub, dims=rest, coords=cs, name=self.name,
                                 attrs=self.attrs).isel(
                    **{k: v for k, v in indexers.items() if k != dim})
            var = var.with_take(dim, pos)
            for k, v in list(coords.items()):
                if dim in v.dims:
                    coords[k] = v.with_take(dim, pos)
        return DataArray._wrap(var, coords, self.name)

    def _sel_pointwise(self, indexers, new_dim):
        from .aggregations.aggregations import _pointwise_reindex
        return _pointwise_reindex(self, indexers, new_dim)

    def transpose(self, *dims):
        perm = [self.dims.index(d) for d in dims]
        return DataArray(np.transpose(self.values, perm), dims=dims,
                         coords=self._coords, name=self.name, attrs=self.attrs)

    T = property(lambda s: s.transpose(*reversed(s.dims)))

    # -- reductions / predicates (host numpy; not the hot path) ----------
    def isnull(self):
        return self._like(np.isnan(self.values))

    def notnull(self):
        return self._like(~np.isnan(self.values))

    def any(self):
        return self._scalar(np.any(self.values))

    def all(self):
        return self._scalar(np.all(self.values))

    def sum(self, dim=None, skipna=True):
        v = self.values
        f = np.nansum if (skipna and v.dtype.kind == "f") else np.sum
        if dim is None:
            return self._scalar(f(v))
        ax = self.dims.index(dim)
        rest = tuple(d for d in self.dims if d != dim)
        return DataArray(f(v, axis=ax), dims=rest,
                         coords={k: c for k, c in self._coords.items() if dim not in c.dims})

    def where(self, cond, other=np.nan):
        return self._like(np.where(_as_data(cond), self.values, _as_data(other)))

    def fillna(self, value):
        v = self.values
        return self._like(np.where(np.isnan(v), _as_data(value), v))

    def _like(self, arr):
        return DataArray(arr, dims=self.dims, coords=self._coords, name=self.name)

    @staticmethod
    def _scalar(x):
        return DataArray(np.asarray(x), dims=())

    def __bool__(self):
        return bool(self.values)

    def _binop(self, other, op):
        if isinstance(other, DataArray) and other.dims != self.dims:
            a, b, dims = _broadcast_by_name(self, other)
            return DataArray(op(a, b), dims=dims, coords={**other._coords, **self._coords})
        return self._like(op(self.values, _as_data(other)))

    __add__ = lambda s, o: s._binop(o, np.add)
    __radd__ = lambda s, o: s._binop(o, lambda a, b: b + a)
    __sub__ = lambda s, o: s._binop(o, np.subtract)
    __rsub__ = lambda s, o: s._binop(o, lambda a, b: b - a)
    __mul__ = lambda s, o: s._binop(o, np.multiply)
    __rmul__ = lambda s, o: s._binop(o, lambda a, b: b * a)
    __truediv__ = lambda s, o: s._binop(o, np.divide)
    __pow__ = lambda s, o: s._binop(o, np.power)
    __lt__ = lambda s, o: s._binop(o, np.less)
    __le__ = lambda s, o: s._binop(o, np.less_equal)
    __gt__ = lambda s, o: s._binop(o, np.greater)
    __ge__ = lambda s, o: s._binop(o, np.greater_equal)
    __and__ = lambda s, o: s._binop(o, np.logical_and)
    __or__ = lambda s, o: s._binop(o, np.logical_or)
    __invert__ = lambda s: s._like(~s.values)
    __neg__ = lambda s: s._like(-s.values)
    __hash__ = None


def _broadcast_by_name(a, b):
    dims = tuple(a.dims) + tuple(d for d in b.dims if d not in a.dims)

    def expand(x):
        v = x.values
        src = [d for d in dims if d in x.dims]
        v = np.transpose(v, [x.dims.index(d) for d in src])
        return v.reshape([v.shape[src.index(d)] if d in src else 1 for d in dims])

    return expand(a), expand(b), dims


def where(cond, x, y):
    """``xr.where`` for same-shaped operands."""
    ref = next(o for o in (cond, x, y) if isinstance(o, DataArray))
    return ref._like(np.where(_as_data(cond), _as_data(x), _as_data(y)))


class _DataVars:
    def __init__(self, ds):
        self._ds = ds

    def __contains__(self, k):
        return k in self._ds._vars

    def __iter__(self):
        return iter(self._ds._vars)

    def __len__(self):
        return len(self._ds._vars)

    def keys(self):
        return self._ds._vars.keys()

    def __getitem__(self, k):
        if k not in self._ds._vars:
            raise KeyError(k)
        return self._ds[k]


class Dataset(_Base):
    def __init__(self, data_vars=None, coords=None, attrs=None):
        self._vars, self._coords, self.attrs = {}, {}, dict(attrs or {})
        for k, v in (coords or {}).items():
            self._coords[k] = _coord_var(k, v)
        for k, v in (data_vars or {}).items():
            self[k] = v

    # -- structure --------------------------------------------------------
    @property
    def dims(self):
        out = {}
        for v in list(self._coords.values()) + list(self._vars.values()):
            for d, n in zip(v.dims, v.shape):
                out.setdefault(d, n)
        return out

    sizes = dims

    @property
    def data_vars(self):
        return _DataVars(self)

    @property
    def variables(self):
        return {**self._coords, **self._vars}

    def __contains__(self, k):
        return k in self._vars or k in self._coords

    def __iter__(self):
        return iter(self._vars)

    def __getitem__(self, key):
        if key in self._vars:
            v = self._vars[key]
            return DataArray._wrap(v, self._coords_for(v.dims), key)
        if key in self._coords:
            return self.coords[key]
        if isinstance(key, str) and "." in key:
            base, comp = key.split(".", 1)
            idx = pd.DatetimeIndex(self._coords[base].values)
            return DataArray(np.asarray(getattr(idx, comp)), dims=self._coords[base].dims,
                             coords={base: self._coords[base]}, name=comp)
        raise KeyError(key)

    def __setitem__(self, key, value):
        if isinstance(value, DataArray):
            var = value.variable
            for k, c in value._coords.items():
                self._coords.setdefault(k, c)
        elif isinstance(value, Variable):
            var = value
        elif isinstance(value, tuple):
            dims, data = value[0], value[1]
            data = data if _is_torch(data) else np.asarray(data)
            var = Variable(dims, data, value[2] if len(value) > 2 else None)
        else:
            raise TypeError("cannot assign {!r}".format(type(value)))
        if key in self._coords:
            self._coords[key] = var
        else:
            self._vars[key] = var

    def __getattr__(self, name):
        if name.startswith("_") or name == "attrs":
            raise AttributeError(name)
        if name in self._vars or name in self._coords:
            return self[name]
        raise AttributeError(name)

    def __repr__(self):
        return "<Dataset dims={} vars={} coords={}>".format(
            self.dims, list(self._vars), list(self._coords))

    def _new(self, variables, coords):
        out = Dataset.__new__(Dataset)
        out._vars, out._coords, out.attrs = variables, coords, dict(self.attrs)
        return out

    def copy(self):
        return self._new({k: v.copy() for k, v in self._vars.items()},
                         {k: v.copy() for k, v in self._coords.items()})

    def load(self):
        return self

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    # -- indexing ---------------------------------------------------------
    def isel(self, **indexers):
        vs, cs = dict(self._vars), dict(self._coords)
        for dim, pos in indexers.items():
            pos = np.asarray(_as_data(pos))
            if pos.ndim == 0:
                pos = pos.reshape(1)  # keep rank; squeeze() drops it
            for store in (vs, cs):
                for k, v in list(store.items()):
                    if dim in v.dims:
                        store[k] = v.with_take(dim, pos)
        return self._new(vs, cs)

    def _sel_pointwise(self, indexers, new_dim):
        from .aggregations.aggregations import _pointwise_reindex
        return _pointwise_reindex(self, indexers, new_dim)

    def rename(self, mapping):
        def ren(v):
            out = v.copy()
            out.dims = tuple(mapping.get(d, d) for d in v.dims)
            out.takes = {mapping.get(d, d): p for d, p in v.takes.items()}
            if v.deferred is not None:
                out.deferred = Deferred(v.deferred.kind, v.deferred.params,
                                        tuple(ren(s) for s in v.deferred.sources))
            return out

        return self._new({mapping.get(k, k): ren(v) for k, v in self._vars.items()},
                         {mapping.get(k, k): ren(v) for k, v in self._coords.items()})

    def drop(self, name):
        names = [name] if isinstance(name, str) else list(name)
        return self._new({k: v for k, v in self._vars.items() if k not in names},
                         {k: v for k, v in self._coords.items() if k not in names})

    drop_vars = drop

    def squeeze(self):
        def sq(v):
            keep = [i for i, n in enumerate(v.shape) if n != 1]
            if len(keep) == v.ndim:
                return v
            return Variable(tuple(v.dims[i] for i in keep), v.values.reshape(
                [v.shape[i] for i in keep]), v.attrs)

        return self._new({k: sq(v) for k, v in self._vars.items()},
                         {k: sq(v) for k, v in self._coords.items()})


# ---------------------------------------------------------------------------
# real-xarray interop (only exercised where xarray is installed)
# ---------------------------------------------------------------------------
def _is_real_xarray(obj):
    return type(obj).__module__.split(".")[0] == "xarray"


def from_any(obj):
    """Accept shim objects as-is; convert real xarray objects by protocol."""
    if isinstance(obj, (Dataset, DataArray)) or not _is_real_xarray(obj):
        return obj
    if hasattr(obj, "data_vars"):
        return Dataset(
            {k: (v.dims, v.values, dict(v.attrs)) for k, v in obj.data_vars.items()},
            coords={k: (v.dims, v.values, dict(v.attrs)) for k, v in obj.coords.items()},
            attrs=dict(obj.attrs))
    return DataArray(obj.values, dims=obj.dims, name=obj.name, attrs=dict(obj.attrs),
                     coords={k: (v.dims, v.values) for k, v in obj.coords.items()})


def to_like(result, like):
    """Return ``result`` (a shim Dataset) as the same family ``like`` came from."""
    if not _is_real_xarray(like):
        return result
    import xarray as xr  # pragma: no cover

    return xr.Dataset(
        {k: (result[k].dims, result[k].values, dict(result[k].attrs)) for k in result.data_vars},
        coords={k: (result.coords[k].dims, result.coords[k].values) for k in result.coords})
