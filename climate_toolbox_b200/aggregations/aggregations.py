"""Weighted grid -> region aggregation on B200 (drop-in for the reference module).

Same names, argument meaning and error behaviour as
``/root/reference/climate_toolbox/aggregations/aggregations.py``:

* :func:`weighted_aggregate_grid_to_regions`    (reference ``:87-124``)
* :func:`_reindex_spatial_data_to_regions`      (reference ``:8-32``)
* :func:`_aggregate_reindexed_data_to_regions`  (reference ``:35-84``)
* :func:`prepare_spatial_weights_data`          (reference ``:127-152``)

What changes underneath: the label lookup + per-row weights + region grouping are
compiled ONCE into a device plan (``ctb_plan_build``), and the gather, the
gridcell transform and ``sum(w*x)/sum(w)`` run as one fused CUDA kernel
(``ctb_aggregate``).  Nothing here computes on the CPU.
"""
from __future__ import annotations

import functools
import os

import numpy as np
import pandas as pd
import torch

from .. import _engine as E
from .. import _native as N
from .._xr import DataArray, Dataset, Deferred, Variable, from_any, to_like

__all__ = ["weighted_aggregate_grid_to_regions", "prepare_spatial_weights_data"]


# ---------------------------------------------------------------------------
# layout analysis: a Variable -> (2-D device/host view, layout, stride, tix, T)
# ---------------------------------------------------------------------------
class _GridView:
    """How one source variable's buffer is seen by the kernels."""

    def __init__(self, var):
        dims = var.dims
        if "lat" not in dims or "lon" not in dims:
            raise KeyError("variable must have 'lat' and 'lon' dimensions, got {}".format(dims))
        a_lat, a_lon = dims.index("lat"), dims.index("lon")
        data = var.physical
        if not isinstance(data, (np.ndarray, torch.Tensor)):
            data = np.asarray(data)
        if isinstance(data, torch.Tensor) and not data.is_cuda:
            data = data.numpy()
        fl = (np.float32, np.float64) if isinstance(data, np.ndarray) else (torch.float32, torch.float64)
        if data.dtype not in fl:
            data = data.astype(np.float64) if isinstance(data, np.ndarray) else data.to(torch.float64)
        n = len(dims)
        if not ((a_lat, a_lon) == (n - 2, n - 1) or (a_lat, a_lon) == (0, 1)):
            # bring (lat, lon) to the back -> TIME_MAJOR
            perm = [i for i in range(n) if i not in (a_lat, a_lon)] + [a_lat, a_lon]
            data = data.permute(*perm) if isinstance(data, torch.Tensor) else np.transpose(data, perm)
            dims = tuple(dims[i] for i in perm)
            a_lat, a_lon = n - 2, n - 1
        if isinstance(data, torch.Tensor):
            data = data.contiguous()
        else:
            data = np.ascontiguousarray(data)
        self.dims = dims
        self.other_dims = tuple(d for d in dims if d not in ("lat", "lon"))
        self.first_spatial_axis = min(var.dims.index("lat"), var.dims.index("lon"))
        self.out_dims_template = var.dims
        shape = tuple(data.shape)
        self.nlat_phys, self.nlon_phys = shape[a_lat], shape[a_lon]
        ncell = self.nlat_phys * self.nlon_phys
        oshape = tuple(s for i, s in enumerate(shape) if i not in (a_lat, a_lon))
        t_phys = int(np.prod(oshape)) if oshape else 1
        if (a_lat, a_lon) == (0, 1) and n > 2:
            self.layout, self.stride = N.LAYOUT_CELL_MAJOR, t_phys
            self.data2d = data.reshape(ncell, t_phys)
        else:
            self.layout, self.stride = N.LAYOUT_TIME_MAJOR, ncell
            self.data2d = data.reshape(t_phys, ncell)
        self.lat_phys = var.takes.get("lat")
        self.lon_phys = var.takes.get("lon")
        # flattened physical time positions of the logical (taken) other-dims
        pos = [var.takes.get(d) for d in self.other_dims]
        self.other_shape = tuple(len(p) if p is not None else s for p, s in zip(pos, oshape))
        self.T = int(np.prod(self.other_shape)) if self.other_shape else 1
        if any(p is not None for p in pos):
            full = [p if p is not None else np.arange(s) for p, s in zip(pos, oshape)]
            mesh = np.meshgrid(*full, indexing="ij")
            self.tix = np.ravel_multi_index([m.ravel() for m in mesh], oshape).astype(np.int64)
            if len(self.tix) == t_phys and np.array_equal(self.tix, np.arange(t_phys)):
                self.tix = None      # a take that keeps every step in place: the kernel without a time index
        else:
            self.tix = None
        self.on_device = isinstance(data, torch.Tensor)
        self.elem_bytes = 4 if str(data.dtype).endswith("float32") else 8

    def same_geometry(self, other):
        return (self.layout == other.layout and self.stride == other.stride and self.T == other.T
                and self.data2d.shape == other.data2d.shape
                and _eq(self.tix, other.tix) and _eq(self.lat_phys, other.lat_phys)
                and _eq(self.lon_phys, other.lon_phys) and self.elem_bytes == other.elem_bytes
                and self.on_device == other.on_device)


class _DailyView:
    """A deferred daily reduction of sub-daily data (``utils.resample_daily``) or a decoded packed source
    (``io.decode_packed``) as the kernels see it: packed planes of days, written by the reduce-pack or decode-pack
    kernel for a compact plan of the planes' element size."""

    layout = N.LAYOUT_TIME_MAJOR
    tix = None

    def __init__(self, var):
        self.src = E.DailySource(var)
        self.kind = var.deferred.kind
        self.how = self.src.how
        self.dims = self.out_dims_template = var.dims
        self.other_dims = (var.dims[0],)
        self.T = self.src.T
        self.other_shape = (self.T,)
        self.lat_phys, self.lon_phys = self.src.lat_phys, self.src.lon_phys
        self.nlat_phys, self.nlon_phys = self.src.nlat_phys, self.src.nlon_phys
        self.stride = self.src.stride
        self.data2d = self.src.x
        self.on_device = self.src.on_device
        self.elem_bytes = self.src.out_bytes

    def same_geometry(self, other):
        return (isinstance(other, _DailyView) and self.T == other.T and self.elem_bytes == other.elem_bytes
                and (self.nlat_phys, self.nlon_phys) == (other.nlat_phys, other.nlon_phys)
                and _eq(self.lat_phys, other.lat_phys) and _eq(self.lon_phys, other.lon_phys)
                and self.on_device == other.on_device)


def _is_daily(var):
    """A deferred variable that the GPU pack evaluates: a daily reduction or a decoded packed source."""
    return var.deferred is not None and var.deferred.kind in ("daily", "decode")


def _view(var):
    return _DailyView(var) if _is_daily(var) else _GridView(var)


def _step_family(var):
    """"edd" / "gdd" / "bins" for the daily mean of a per-step transform of sub-daily data
    (``transformations.subdaily_*``), else None."""
    d = var.deferred
    return d.params[0][0] if _is_daily(var) and d.kind == "daily" and isinstance(d.params[0], tuple) else None


def _same_steps(a, b):
    """Two deferred daily variables read the same steps of the same buffer."""
    pa, pb = a.deferred.params, b.deferred.params
    return (pa[1:3] == pb[1:3] and np.array_equal(pa[3], pb[3]) and
            _same_source(a.deferred.sources[0], b.deferred.sources[0]))


def _same_source(a, b):
    """Two transform sources read the same data: the same buffer and takes, for daily reductions also the same
    ``how``, steps and days, and for decoded sources the same decoding."""
    if _is_daily(a) or _is_daily(b):
        if not (_is_daily(a) and _is_daily(b) and a.deferred.kind == b.deferred.kind):
            return False
        if a.deferred.kind == "decode":
            return _same_decode(a.deferred.params, b.deferred.params) and \
                _same_source(a.deferred.sources[0], b.deferred.sources[0])
        return a.deferred.params[0] == b.deferred.params[0] and _same_steps(a, b)
    return (a.physical is b.physical and a.dims == b.dims and
            all(_eq(a.takes.get(d), b.takes.get(d)) for d in a.dims))


def _same_decode(pa, pb):
    return pa[:3] == pb[:3] and np.dtype(pa[3]) == np.dtype(pb[3])


def _eq(a, b):
    if a is None or b is None:
        return a is None and b is None
    return np.array_equal(a, b)


def _resolve(var):
    """Variable -> (kind, params, [source Variables])."""
    if var.deferred is None or _is_daily(var):
        return "identity", (), [var]
    d = var.deferred
    if d.kind == "reindex":
        raise ValueError("variable is already reindexed to regions")
    return d.kind, tuple(d.params), list(d.sources)


def _coord_labels(ds, name):
    if name not in ds._coords:
        raise KeyError(name)
    return np.asarray(ds._coords[name].values, dtype=np.float64)


def _run_group(plan, views, kind, params, n_out, variant, groups=None, ingest=None, host_out=None, doy=None):
    """One fused launch for `n_out` outputs sharing the same sources."""
    v0 = views[0]
    if isinstance(v0, _DailyView):
        out = E.aggregate_daily(plan, [(v.src, v.how) for v in views], kind, params, n_out, variant, groups,
                                host_out, doy)
    elif v0.on_device:
        out = E.aggregate_device(plan, views[0].data2d, views[1].data2d if len(views) > 1 else None,
                                 v0.layout, v0.stride, v0.tix, v0.T, kind, params, n_out, variant,
                                 groups=groups, doy=doy)
    else:
        out = E.aggregate_host(plan, [v.data2d for v in views], v0.layout, v0.stride, v0.tix, v0.T,
                               kind, params, n_out, variant, groups=groups, ingest=ingest, host_out=host_out,
                               doy=doy)
    return out


def _season_gate(mask, ds, lat, lon, view, time_dim):
    """GrowingSeasonMask -> (gate word of every PHYSICAL gridcell, day of year of every logical step)."""
    from ..utils.utils import _day_of_year, _match
    words = mask.gate_words()
    never = np.uint32(N.GATE_NEVER)
    words = np.where(mask.missing, never, words)
    ii = _match(np.asarray(mask.lat, dtype=np.float64), lat, "lat")       # data labels -> mask rows
    jj = _match(np.asarray(mask.lon, dtype=np.float64), lon, "lon")
    logical = words[np.ix_(ii, jj)]
    pi = view.lat_phys if view.lat_phys is not None else np.arange(len(lat))
    pj = view.lon_phys if view.lon_phys is not None else np.arange(len(lon))
    phys = np.full((view.nlat_phys, view.nlon_phys), never, dtype=np.uint32)
    phys[np.ix_(np.asarray(pi), np.asarray(pj))] = logical
    if time_dim not in ds._coords:
        raise KeyError(time_dim)
    doy = _day_of_year(ds._coords[time_dim].values)
    if len(doy) != view.T:
        raise ValueError("time coordinate has {} steps, the variable {}".format(len(doy), view.T))
    if len(mask.time) == view.T and not np.array_equal(_day_of_year(mask.time), doy):
        raise ValueError("season_mask was built for another time axis")
    return phys, doy.astype(np.int32)


def _time_group_ids(ds, dim, n, spec):
    """``time_groups=`` of :func:`weighted_aggregate_grid_to_regions` -> (group id of every step,
    group labels).  ``"year"``: the calendar year of a datetime coordinate, or ``YYYYDDD // 1000`` of
    the integer time ``tas_poly`` writes; an int ``p``: blocks of ``p`` consecutive steps; an array:
    one label per step.  Groups must be runs of consecutive steps."""
    if isinstance(spec, str):
        if spec != "year":
            raise ValueError("time_groups={!r}: expected 'year', a block length or one label per step".format(spec))
        if dim not in ds._coords:
            raise KeyError(dim)
        c = np.asarray(ds._coords[dim].values)
        if np.issubdtype(c.dtype, np.datetime64):
            lab = c.astype("datetime64[Y]").astype(np.int64) + 1970
        elif np.issubdtype(c.dtype, np.integer):
            lab = c.astype(np.int64) // 1000
        else:
            lab = pd.DatetimeIndex(c).year.values.astype(np.int64)
    elif np.isscalar(spec):
        p = int(spec)
        if p <= 0:
            raise ValueError("time_groups block length must be positive")
        lab = np.arange(n, dtype=np.int64) // p
    else:
        lab = np.asarray(spec)
    if len(lab) != n:
        raise ValueError("time_groups gives {} labels for {} steps".format(len(lab), n))
    change = np.ones(n, dtype=bool)
    if n:
        change[1:] = lab[1:] != lab[:-1]
    gid = np.cumsum(change) - 1
    labels = lab[change]
    if len(set(labels.tolist())) != len(labels):
        raise ValueError("time_groups: every group must be one run of consecutive steps")
    return gid.astype(np.int32), labels


def _group_requests(reqs):
    """Fuse requests that read the same sources: poly orders / EDD thresholds /
    GDD pairs / contiguous temperature bins become extra outputs of ONE pass over
    the data (config 3/4).  A bin (offset, lo, hi) joins a group of bins whose
    last edge is lo: the group's params are (offset, e_0, ..., e_n).  A spline term
    (offset, i, k_1, ..., k_n) joins a group of the same offset and knots whose
    terms run first .. i - 1: the group keeps the params (offset, first, k_1, ..., k_n).
    Per-step transforms of sub-daily data (identity requests of one ``_step_family``) that read the same steps
    fuse too, bins when contiguous: up to MAX_OUT planes from one reduce-pack call, each aggregated on its own
    (the group's "step" names the family, its "srcs" hold every member)."""
    groups = []
    for name, kind, params, srcs in reqs:
        placed = False
        step = _step_family(srcs[0]) if kind == "identity" else None
        for g in groups:
            if step is not None or g["step"] is not None:
                last = g["srcs"][-1]
                if (step == g["step"] and len(g["names"]) < N.MAX_OUT and _same_steps(last, srcs[0]) and
                        (step != "bins" or last.deferred.params[0][2] == srcs[0].deferred.params[0][1])):
                    g["names"].append(name)
                    g["srcs"].append(srcs[0])
                    placed = True
                    break
                continue
            same_src = len(g["srcs"]) == len(srcs) and all(_same_source(a, b) for a, b in zip(g["srcs"], srcs))
            if not same_src or g["kind"] != kind or len(g["names"]) >= N.MAX_OUT:
                continue
            if kind == "identity" or (kind in ("poly", "bins") and g["params"][0] != params[0]):
                continue
            if kind == "bins" and g["params"][-1] != params[1]:
                continue
            if kind == "rcspline" and (g["params"][:1] + g["params"][2:] != params[:1] + params[2:] or
                                       g["params"][1] + len(g["names"]) != params[1]):
                continue
            g["names"].append(name)
            if kind != "rcspline":
                g["params"] = g["params"] + (params[1:] if kind == "poly" else params[2:] if kind == "bins" else params)
            placed = True
            break
        if not placed:
            groups.append({"names": [name], "kind": kind, "params": tuple(params), "srcs": list(srcs), "step": step})
    return groups


def _aggregate_core(ds, variables, aggwt, agglev, weights, backup_aggwt, variant=N.VARIANT_AUTO,
                    device=None, smem_budget=0, keep_on_device=False, pack_host=True, trusted_weights=False,
                    time_groups=None, time_dim="time", ingest=None, season_mask=None):
    lat, lon = _coord_labels(ds, "lat"), _coord_labels(ds, "lon")
    reqs = []
    for name in variables:
        if name not in ds._vars:
            raise KeyError(name)
        kind, params, srcs = _resolve(ds._vars[name])
        reqs.append((name, kind, params, srcs))

    out_ds = Dataset()
    for g in _group_requests(reqs):
        views = [_view(s) for s in g["srcs"]]
        v0 = views[0]
        daily = isinstance(v0, _DailyView)
        if any(getattr(v, "kind", None) != getattr(v0, "kind", None) for v in views):
            raise ValueError("inputs of a two-input transform must both be daily reductions of sub-daily data "
                             "or decoded packed sources, or neither")
        for v in views[1:]:
            if not v0.same_geometry(v):
                raise ValueError("inputs of a two-input transform must share shape, dtype and layout")
        grid = E.GridSpec(lat, lon, v0.lat_phys, v0.lon_phys, v0.nlat_phys, v0.nlon_phys)
        dev = device or (v0.data2d.device if v0.on_device else E.default_device())
        # host-resident (time, lat, lon) inputs go through a compact plan: only the referenced
        # gridcells are packed on the host and cross PCIe
        # daily reductions of sub-daily data and decoded packed sources are packed by the reduce-pack or
        # decode-pack kernel wherever the data lives
        compact = daily or ((not v0.on_device) and v0.layout == N.LAYOUT_TIME_MAJOR and pack_host)
        cell_gate = doy = None
        if season_mask is not None:
            # growing-season gate (SURVEY 8-f3): per-gridcell (first, last, wrap) into the plan, day of
            # year of every step into the launch -- the lat x lon x time mask is never built
            if v0.other_dims != (time_dim,):
                raise NotImplementedError("season_mask needs variables over ({}, lat, lon), got {}".format(
                    time_dim, v0.out_dims_template))
            cell_gate, doy = _season_gate(season_mask, ds, lat, lon, v0, time_dim)
        plan = E.get_plan(grid, weights, aggwt, agglev, backup_aggwt,
                          stage_bytes=(1 if g["step"] else len(views)) * v0.elem_bytes, device=dev,
                          smem_budget=smem_budget, compact=compact, elem_bytes=v0.elem_bytes,
                          trusted=trusted_weights, cell_gate=cell_gate)
        n_out = len(g["names"])
        groups = glabels = None
        other_shape = v0.other_shape
        if time_groups is not None:
            # fused time reduction (SURVEY 8-f4): the days of every group are summed inside the kernel
            if v0.other_dims != (time_dim,):
                raise NotImplementedError("time_groups needs variables over ({}, lat, lon), got {}".format(
                    time_dim, v0.out_dims_template))
            gid, glabels = _time_group_ids(ds, time_dim, v0.T, time_groups)
            groups = E.get_time_groups(gid, dev)
            other_shape = (groups.n_groups,)
        # host inputs, host result: the result block is handed to the engine, which may fill it in time
        # chunks while later chunks are still in flight
        host_fill = None
        if not keep_on_device and not v0.on_device and groups is None and v0.T > 0 and plan.R > 0:
            host, res_np = E.pinned_result_like(torch.empty((n_out, plan.R, v0.T), dtype=torch.float64, device="meta"))
            host_fill = [host, False]
        out = _run_group(plan, views, g["kind"], g["params"], n_out, variant, groups, ingest, host_fill, doy)  # [n_out, R, T]
        # reference dim order: agglev takes the place of the first of (lat, lon)
        tmpl = ds._vars[g["names"][0]].dims
        first = min(tmpl.index("lat"), tmpl.index("lon"))
        others = [d for d in tmpl if d not in ("lat", "lon")]
        if keep_on_device:
            res = out
        else:
            # D2H into pinned memory (57 GB/s on the round-1 box; a pageable copy runs at
            # 2 GB/s).  The block comes from a pool and returns to it when the last view of
            # the returned arrays is garbage collected.
            if host_fill is not None:
                host, res = host_fill[0], res_np
            else:
                host, res = E.pinned_result_like(out)
            if host_fill is None or not host_fill[1]:
                host.copy_(out, non_blocking=True)
                E.TRANSFER_BYTES["d2h"] += out.numel() * out.element_size()
            torch.cuda.current_stream(out.device).synchronize()
        R = plan.R
        for j, name in enumerate(g["names"]):
            a = res[j].reshape((R,) + other_shape)         # (agglev, *others) in view order
            cur = [agglev] + list(v0.other_dims)
            want = list(others)
            want.insert(first, agglev)
            perm = [cur.index(d) for d in want]
            a = a.permute(*perm) if isinstance(a, torch.Tensor) else np.transpose(a, perm)
            out_ds[name] = Variable(tuple(want), a, ds._vars[name].attrs)
        out_ds._coords[agglev] = Variable((agglev,), np.asarray(plan.region_labels))
        for d in others:
            if glabels is not None and d == time_dim:
                out_ds._coords[d] = Variable((d,), np.asarray(glabels))
            elif d in ds._coords:
                out_ds._coords[d] = Variable((d,), ds._coords[d].values, ds._coords[d].attrs)
    return out_ds


# ---------------------------------------------------------------------------
# reference API
# ---------------------------------------------------------------------------
def _pointwise_reindex(obj, indexers, new_dim):
    """``obj.sel(lon=<DataArray>, lat=<DataArray>)``: exact-label pointwise gather.
    Returns lazily reindexed variables (materialised by ``ctb_gather_rows``)."""
    if set(indexers) != {"lat", "lon"}:
        raise NotImplementedError("pointwise selection is implemented for (lat, lon) only")
    df = pd.DataFrame({"lat": np.asarray(indexers["lat"].values, dtype=np.float64),
                       "lon": np.asarray(indexers["lon"].values, dtype=np.float64)})
    ds = obj if isinstance(obj, Dataset) else Dataset({obj.name or "_da": obj}, coords=obj._coords)
    res = _reindex_spatial_data_to_regions(ds, df, new_dim=new_dim)
    return res if isinstance(obj, Dataset) else res[obj.name or "_da"]


def _reindex_spatial_data_to_regions(ds, df, new_dim="reshape_index"):
    """
    Reindexes spatial and segment weight data to regions
    (reference ``aggregations.py:8-32``).

    Every data variable with (lat, lon) dims becomes a variable over
    ``reshape_index`` (one entry per row of ``df``), found by EXACT float64 label
    match; a label that is not in the grid raises ``KeyError``.  The gather is
    lazy: ``.values`` runs the CUDA gather kernel, and
    :func:`_aggregate_reindexed_data_to_regions` fuses it away entirely.
    """
    like = ds
    ds = from_any(ds)
    lat, lon = _coord_labels(ds, "lat"), _coord_labels(ds, "lon")
    n = len(df)
    trivial = pd.DataFrame({"lat": np.asarray(df["lat"].values, dtype=np.float64),
                            "lon": np.asarray(df["lon"].values, dtype=np.float64),
                            "_r": np.zeros(n, dtype=np.int32), "_w": np.ones(n)})
    out = Dataset()
    for name, var in ds._vars.items():
        if "lat" not in var.dims or "lon" not in var.dims:
            out._vars[name] = var
            continue
        if var.deferred is not None:
            var = Variable(var.dims, var.values, var.attrs)
        view = _GridView(var)
        grid = E.GridSpec(lat, lon, view.lat_phys, view.lon_phys, view.nlat_phys, view.nlon_phys)
        dev = view.data2d.device if view.on_device else E.default_device()
        plan = E.get_plan(grid, trivial, "_w", "_r", "_w", stage_bytes=view.elem_bytes, device=dev,
                          elem_bytes=view.elem_bytes)
        first = min(var.dims.index("lat"), var.dims.index("lon"))
        others = [d for d in var.dims if d not in ("lat", "lon")]
        new_dims = list(others)
        new_dims.insert(first, new_dim)
        shape = list(view.other_shape)

        def materialise(view=view, plan=plan, dev=dev, first=first, others=others):
            x = view.data2d if view.on_device else torch.from_numpy(view.data2d).to(dev)
            T = view.T
            if view.layout == N.LAYOUT_TIME_MAJOR:
                o = torch.empty((T, plan.n_rows), dtype=x.dtype, device=dev)
            else:
                o = torch.empty((plan.n_rows, T), dtype=x.dtype, device=dev)
            tix = plan.time_index_device(view.tix)
            import ctypes as C
            N.check(N.lib().ctb_gather_rows(
                plan._h, C.c_void_p(x.data_ptr()), E._T2CTB[x.dtype], view.layout, view.stride,
                C.c_void_p(tix.data_ptr()) if tix is not None else None, T,
                C.c_void_p(o.data_ptr()), E._stream_ptr(dev)))
            a = o.cpu().numpy()
            if view.layout == N.LAYOUT_TIME_MAJOR:
                a = a.reshape(view.other_shape + (plan.n_rows,))
                cur = list(view.other_dims) + [new_dim]
            else:
                a = a.reshape((plan.n_rows,) + view.other_shape)
                cur = [new_dim] + list(view.other_dims)
            want = list(others)
            want.insert(first, new_dim)
            return np.transpose(a, [cur.index(d) for d in want])

        shape.insert(first, n)
        d = Deferred("reindex", (materialise, ds), (var,), shape=shape)
        out._vars[name] = Variable(tuple(new_dims), None, var.attrs, None, d)
    for k, c in ds._coords.items():
        if k in ("lat", "lon"):
            continue
        out._coords[k] = c
    out._coords["lat"] = Variable((new_dim,), np.asarray(df["lat"].values))
    out._coords["lon"] = Variable((new_dim,), np.asarray(df["lon"].values))
    return to_like(out, like)


def _aggregate_reindexed_data_to_regions(
    ds, variable, aggwt, agglev, weights, backup_aggwt="areawt"
):
    """
    Performs weighted avg for climate variable by region
    (reference ``aggregations.py:35-84``).

    ``w = weights[aggwt] if > 0 else weights[backup_aggwt]`` per ROW;
    ``out = sum_k nan->0(x_k * w_k) / sum_k nan->0(w_k)`` per sorted unique
    ``weights[agglev]``.  Unlike the reference, the caller's ``ds`` is not mutated.
    """
    like = ds
    ds = from_any(ds)
    names = [variable] if isinstance(variable, str) else list(variable)
    var = ds._vars[names[0]] if names[0] in ds._vars else None
    if var is None:
        raise KeyError(names[0])
    if var.deferred is not None and var.deferred.kind == "reindex":
        # lazily reindexed by _reindex_spatial_data_to_regions: fuse the gather away
        origin = var.deferred.params[1]
        if len(weights) != var.shape[var.dims.index("reshape_index")]:
            raise ValueError("weights has {} rows, reshape_index has {}".format(
                len(weights), var.shape[var.dims.index("reshape_index")]))
        w2 = weights.assign(lat=np.asarray(ds._coords["lat"].values),
                            lon=np.asarray(ds._coords["lon"].values))
        sub = Dataset()
        sub._coords = dict(origin._coords)
        for nme in names:
            sub._vars[nme] = ds._vars[nme].deferred.sources[0]
        return to_like(_aggregate_core(sub, names, aggwt, agglev, w2, backup_aggwt), like)
    # already materialised (reshape_index, ...) data: a 1 x n "grid" with identity lookup
    if "reshape_index" not in var.dims:
        raise KeyError("reshape_index")
    n = var.shape[var.dims.index("reshape_index")]
    w2 = weights.assign(lat=np.zeros(n), lon=np.arange(n, dtype=np.float64))
    sub = Dataset(coords={"lat": np.zeros(1), "lon": np.arange(n, dtype=np.float64)})
    for nme in names:
        v = ds._vars[nme]
        ax = v.dims.index("reshape_index")
        vals = v.values
        data = np.expand_dims(vals, ax)
        dims = v.dims[:ax] + ("lat", "lon") + v.dims[ax + 1:]
        sub._vars[nme] = Variable(dims, data, v.attrs)
    for k, c in ds._coords.items():
        if "reshape_index" not in c.dims and k not in ("lat", "lon"):
            sub._coords[k] = c
    return to_like(_aggregate_core(sub, names, aggwt, agglev, w2, backup_aggwt), like)


def weighted_aggregate_grid_to_regions(ds, variable, aggwt, agglev, weights=None,
                                       backup_aggwt="areawt", **engine_opts):
    """
    Computes the weighted reshape of gridded data (reference ``aggregations.py:87-124``).

    Parameters
    ----------
    ds : Dataset (this package's or ``xarray``'s)
        Must have 'lat' and 'lon' in the coordinates.  Variables may be numpy
        arrays (host; copied in time chunks) or CUDA tensors (device-resident),
        in ``(time, lat, lon)`` or ``(lat, lon, time)`` order, float32/float64.
    variable : str or list of str
        Variable(s) to aggregate.  Deferred transforms (``tas_poly``, ``tas_bins``, ``tas_rcspline``,
        ``snyder_edd``, ``snyder_gdd``) of the same source are fused into one pass.
    aggwt, agglev : str
        Weight / region-id column names in ``weights``.
    weights : pandas.DataFrame (or a CSV path, passed to
        :func:`prepare_spatial_weights_data`) with columns lat, lon, agglev, aggwt
        and ``backup_aggwt``.  ``None`` raises ``TypeError`` exactly like the
        reference (``:118-119`` calls a one-argument function without arguments).
    season_mask : extension (``engine_opts``), default None.  The object
        ``utils.get_daily_growing_season_mask`` returns (reference ``utils.py:119-153``): gridcell-days
        outside their growing season do not enter the weighted sum -- equal to aggregating
        ``ds[variable] * mask``, with the gate applied inside the kernel.
    time_groups : extension (``engine_opts``), default None.  ``"year"``, a block length or one
        label per time step: the daily region values of every group are SUMMED inside the kernel
        (``EDD_P = sum_d EDD_d``, reference ``transformations.py:17-21``) and the result has one
        time step per group -- equal to ``out.groupby(label).sum()`` of the daily result, without
        ever writing the region x day block.

    Returns
    -------
    Dataset with ``agglev`` in place of (lat, lon); float64.
    """
    if weights is None:
        weights = prepare_spatial_weights_data()  # TypeError, as in the reference
    if isinstance(weights, str):
        weights = prepare_spatial_weights_data(weights)
    like = ds
    ds = from_any(ds)
    names = [variable] if isinstance(variable, str) else list(variable)
    return to_like(_aggregate_core(ds, names, aggwt, agglev, weights, backup_aggwt,
                                   **engine_opts), like)


def _stack_weight_columns(weights, aggwts, agglevs, backup_aggwt):
    """One frame with a copy of the rows per (region level, weight column) pair: region r of level l
    under weight k becomes the virtual region ``base[l, k] + code_l(r)``.  Returns (frame[lat, lon,
    _lev, _w, _bk], {level: sorted region labels}, [(level, weight, base, R_level)], sorted virtual
    codes that have rows)."""
    n = len(weights)
    lat = np.asarray(weights["lat"].values, dtype=np.float64)
    lon = np.asarray(weights["lon"].values, dtype=np.float64)
    bk = np.asarray(weights[backup_aggwt].values, dtype=np.float64)
    labels, combos, virt, ws = {}, [], [], []
    base = 0
    for lev in agglevs:
        codes, labels[lev] = E.region_codes(weights[lev].values)
        R = len(labels[lev])
        for wt in aggwts:
            combos.append((lev, wt, base, R))
            virt.append(np.where(codes >= 0, codes.astype(np.int64) + base, -1))
            ws.append(np.asarray(weights[wt].values, dtype=np.float64))
            base += R
    virt = np.concatenate(virt) if virt else np.zeros(0, dtype=np.int64)
    K = len(combos)
    stacked = pd.DataFrame({
        "lat": np.tile(lat, K), "lon": np.tile(lon, K),
        "_lev": np.where(virt >= 0, virt, np.nan),      # NaN labels are dropped, as in the reference
        "_w": np.concatenate(ws) if ws else np.zeros(0), "_bk": np.tile(bk, K)})
    assert len(stacked) == n * K
    return stacked, labels, combos, np.unique(virt[virt >= 0])


_STACKED = {}   # (id(weights), columns) -> (weights ref, stacked frame): keeps the plan-cache fast path warm


def weighted_aggregate_grid_to_regions_multi(ds, variable, aggwts, agglev, weights,
                                             backup_aggwt="areawt", **engine_opts):
    """
    Extension (SURVEY 8-f2): aggregate ``variable`` with SEVERAL weight columns and / or to SEVERAL
    region levels in ONE pass over the gridded data.  Equivalent to one
    ``weighted_aggregate_grid_to_regions`` call per (agglev, aggwt) pair (reference
    ``aggregations.py:87-124`` run once per pair), but the data is staged once: every region is
    entered once per pair as a "virtual" region, the virtual regions of a region share their
    gridcell footprint and land in the same kernel work bundle; coarse levels (countries) are split
    over bundles and summed in fixed order like any region larger than a tile.

    ``agglev``: one column name -> variables ``"<variable>_<aggwt>"`` over ``agglev`` (as before);
    a list -> variables ``"<variable>_<aggwt>_<agglev>"``, each over its own region dimension.
    """
    if isinstance(weights, str):
        weights = prepare_spatial_weights_data(weights)
    aggwts = list(aggwts)
    single = isinstance(agglev, str)
    agglevs = [agglev] if single else list(agglev)
    for col in ["lat", "lon", backup_aggwt] + agglevs + aggwts:
        if col not in weights:
            raise KeyError(col)
    if not isinstance(variable, str):
        raise TypeError("weighted_aggregate_grid_to_regions_multi takes one variable name")
    key = (id(weights), tuple(aggwts), tuple(agglevs), backup_aggwt, len(weights))
    hit = _STACKED.get(key)
    sums = tuple(E._col_fp(weights[c].values) for c in aggwts + [backup_aggwt, "lat", "lon"] + agglevs)
    if hit is not None and hit[0] is weights and hit[2] == sums:
        stacked, labels, combos, present = hit[1], hit[3], hit[4], hit[5]
    else:
        stacked, labels, combos, present = _stack_weight_columns(weights, aggwts, agglevs, backup_aggwt)
        if len(_STACKED) > 8:
            _STACKED.clear()
        _STACKED[key] = (weights, stacked, sums, labels, combos, present)
    like = ds
    ds = from_any(ds)
    res = _aggregate_core(ds, [variable], "_w", "_lev", stacked, "_bk", trusted_weights=True, **engine_opts)
    var = res._vars[variable]
    ax = var.dims.index("_lev")
    out = Dataset()
    data = var.physical      # numpy (pinned block) or, with keep_on_device, the CUDA tensor itself
    for lev, wt, base, R in combos:
        dims = tuple(lev if d == "_lev" else d for d in var.dims)
        sel = np.flatnonzero((present >= base) & (present < base + R))
        if len(sel) and sel[-1] - sel[0] + 1 == len(sel):      # the usual case: a contiguous block -> a view
            idx = [slice(None)] * len(var.dims)
            idx[ax] = slice(int(sel[0]), int(sel[-1]) + 1)
            a = data[tuple(idx)]
        elif isinstance(data, torch.Tensor):
            a = data.index_select(ax, torch.as_tensor(sel, device=data.device))
        else:
            a = np.take(data, sel, axis=ax)
        name = "{}_{}".format(variable, wt) if single else "{}_{}_{}".format(variable, wt, lev)
        out[name] = Variable(dims, a, var.attrs)
    for lev in agglevs:
        out._coords[lev] = Variable((lev,), np.asarray(labels[lev]))
    for d, c in res._coords.items():
        if d != "_lev":
            out._coords[d] = c
    return to_like(out, like)


def _weights_cache_file(weights_file, cache_dir):
    """Path of the parsed-frame cache of a weights CSV: keyed by absolute path, size and mtime."""
    import hashlib
    st = os.stat(weights_file)
    key = "{}|{}|{}".format(os.path.abspath(weights_file), st.st_size, st.st_mtime_ns)
    return os.path.join(cache_dir, "ctb_weights_{}.feather".format(hashlib.sha1(key.encode()).hexdigest()[:20]))


@functools.lru_cache(maxsize=8)
def prepare_spatial_weights_data(weights_file, cache_dir=None):
    """
    Rescales the pix_cent_x column values (reference ``aggregations.py:127-152``).

    ``pix_cent_x == 180.125`` is relabelled ``-179.875`` (the reference's
    ``df.set_value`` call, removed in pandas 1.0, intended exactly this);
    duplicates are KEPT (the reference's ``drop_duplicates()`` discards its
    result); columns renamed to ``lon`` / ``lat``; index named ``reshape_index``.
    Memoised per path like the reference's ``toolz.memoize``.

    ``cache_dir`` (or the environment variable ``CTB_WEIGHTS_CACHE``; SURVEY 8-f2): the parsed frame
    is also kept on disk in Arrow IPC format, keyed by the CSV's path, size and modification time,
    so that the next PROCESS skips the CSV parse (a segment-weights file of 420k rows: seconds of
    ``read_csv`` against tens of milliseconds).  The device plan is rebuilt from the frame
    (``_engine.get_plan``: one-time, ~0.15 s) and cached by content in the process.
    """
    cache_dir = cache_dir or os.environ.get("CTB_WEIGHTS_CACHE")
    cached = None
    if cache_dir:
        cached = _weights_cache_file(weights_file, cache_dir)
        if os.path.exists(cached):
            df = pd.read_feather(cached)
            df.index.names = ["reshape_index"]
            return df
    df = pd.read_csv(weights_file)
    df.loc[df["pix_cent_x"] == 180.125, "pix_cent_x"] = -179.875
    df.index.names = ["reshape_index"]
    df = df.rename(columns={"pix_cent_x": "lon", "pix_cent_y": "lat"})
    if cached:
        os.makedirs(cache_dir, exist_ok=True)
        tmp = "{}.{}.tmp".format(cached, os.getpid())
        df.reset_index(drop=True).to_feather(tmp)
        os.replace(tmp, cached)       # atomic: concurrent ranks may race to write the same file
    return df
