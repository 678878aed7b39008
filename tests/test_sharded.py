"""Time-sharded aggregation (``climate_toolbox_b200/parallel.py``) against the single-process result.

Every rank of a group aggregates a contiguous block of days (``shard_range``: starts on multiples of the
32-day tile) and the blocks are gathered.  Three tiers:

* **CPU** (gloo): the per-shard aggregation is a stand-in, the numpy oracle behind the public signature,
  that honours ``time_groups``, ``season_mask`` and ``time_dim``.  It rounds each daily region value to a
  multiple of 2^-16, so every partial sum of a time group is exact in float64: the sharded result must then
  equal the unsharded stand-in exactly, whatever order the parts of a group that spans a shard boundary
  are added in.  What is under test is the partition, the group bookkeeping and the reassembly.
* **one GPU** (gloo, two and three ranks sharing device 0): the real ``weighted_aggregate_grid_to_regions``
  on host inputs, against the single-process call on the same inputs.  Daily results are bit identical:
  each rank's tiles are the global tiles, so every region-day is summed in the same order from the same
  values.  A time group inside one shard is bit identical for the same reason (its per-tile partial sums,
  or for a split region its per-day sums, are the same numbers added in the same order).  A group that
  spans shards is the same addends added in another order, so it differs by at most
  ``2 n_days(g) 2^-53 sum_d |daily_{r,d}|`` (the tile partials of unsplit regions and the day values of
  split regions are at most ``n_days(g)`` addends; the two summation trees share their first shard's
  prefix, and every other addition rounds by at most 2^-53 of a sum bounded by ``sum_d |daily|``).
* **multi-GPU** (NCCL, one rank per GPU): the device-level entry points against the single-GPU launch of
  the same plan, bit for bit; skipped when fewer than two GPUs are visible.

Results are compared as int64 wherever bit identity is claimed, so NaN payloads and signed zeros count.
Every worker is joined, and terminated if it outlives its test; every queue read has a timeout.
"""
import os
import queue
import socket
import time
import traceback

import numpy as np
import pandas as pd
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

TOL = 1e-9                  # test_gpu_parity.TOL
U = 2.0 ** -53
QUANTUM = 16                # the CPU stand-in rounds daily values to multiples of 2^-QUANTUM


# ----------------------------------------------------------------------------
# processes
# ----------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _entry(fn, rank, world, port, backend, q, args):
    """One rank: joins the group, runs ``fn(rank, world, *args)`` and reports ``(rank, result)``, or the
    traceback of whatever it raised."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    try:
        kw = {}
        if backend == "nccl":
            torch.cuda.set_device(rank)
            kw["device_id"] = torch.device("cuda", rank)
        dist.init_process_group(backend, rank=rank, world_size=world, **kw)
        try:
            res = fn(rank, world, *args)
        finally:
            dist.destroy_process_group()
        q.put((rank, res))
    except BaseException:      # noqa: BLE001 -- the parent reports it
        q.put((rank, "rank {} raised:\n{}".format(rank, traceback.format_exc())))


def run_ranks(fn, world, *args, backend="gloo", timeout=200):
    """``fn`` on ``world`` spawned ranks -> the list of their results in rank order.  No process outlives
    the call: workers are joined, and terminated (then killed) if they have not ended."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_entry, args=(fn, r, world, port, backend, q, args)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        res, deadline = {}, time.monotonic() + timeout
        while len(res) < world:
            try:
                rank, out = q.get(timeout=5)
                res[rank] = out
            except queue.Empty:
                dead = [r for r, p in enumerate(procs) if r not in res and p.exitcode is not None]
                assert not dead, "ranks {} ended without a result (exit codes {})".format(
                    dead, [procs[r].exitcode for r in dead])
                assert time.monotonic() < deadline, "ranks {} gave no result in {} s".format(
                    sorted(set(range(world)) - set(res)), timeout)
        for p in procs:
            p.join(60)
        errors = [v for v in res.values() if isinstance(v, str)]
        assert not errors, "\n".join(errors)
        assert [p.exitcode for p in procs] == [0] * world
        return [res[r] for r in range(world)]
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(10)
            if p.is_alive():
                p.kill()
                p.join(10)
        q.close()
        q.join_thread()


def _failures(results):
    return [(rank, name, detail) for rank, rows in enumerate(results) for name, ok, detail in rows if not ok]


# ----------------------------------------------------------------------------
# group bookkeeping shared by the tiers
# ----------------------------------------------------------------------------
def group_ranks(gid, T, world):
    """Number of ranks whose days touch each group of the full axis."""
    from climate_toolbox_b200.parallel import shard_range
    k = np.zeros(int(gid.max()) + 1 if len(gid) else 0, dtype=np.int64)
    for r in range(world):
        t0, t1 = shard_range(T, world, r)
        if t1 > t0:
            k[np.unique(gid[t0:t1])] += 1
    return k


def bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.int64)


def test_sum_group_blocks_copies_first_part_and_adds_later_ones():
    """The combine step on its own: a group inside one shard keeps its bits (signed zero, NaN payload), a
    group continued from an earlier shard gets the later part added, in rank order."""
    from climate_toolbox_b200.parallel import _sum_group_blocks
    nan_p = np.array([0x7FF8000000000123], dtype=np.uint64).view(np.float64)[0]
    # groups 0, 1 on rank 0; group 1 continues on rank 1 with groups 2, 3; rank 2 empty; rank 3 continues 3
    firsts, counts = [0, 1, 0, 3], [2, 3, 0, 1]
    recv = torch.full((4, 2, 3), 99.0, dtype=torch.float64)
    recv[0, :, :2] = torch.tensor([[-0.0, 1.5], [nan_p, 2.0]], dtype=torch.float64)
    recv[1, :, :3] = torch.tensor([[0.25, -0.0, 3.0], [0.5, nan_p, 4.0]], dtype=torch.float64)
    recv[3, :, :1] = torch.tensor([[1.0], [-4.0]], dtype=torch.float64)
    full = torch.empty((2, 4), dtype=torch.float64)
    _sum_group_blocks(full, recv, firsts, counts)
    exp = np.array([[-0.0, 1.5 + 0.25, -0.0, 3.0 + 1.0], [nan_p, 2.0 + 0.5, nan_p, 4.0 - 4.0]])
    np.testing.assert_array_equal(bits(full.numpy()), bits(exp))


# ----------------------------------------------------------------------------
# CPU tier: gloo, the oracle as stand-in for the aggregation
# ----------------------------------------------------------------------------
def _stand_in(ds, variable, aggwt, agglev, weights=None, backup_aggwt="areawt", time_groups=None, season_mask=None,
              time_dim="time", **kw):
    """The oracle behind the public signature.  ``season_mask`` multiplies the data by the dense mask over
    the day of year of ``ds``'s own time coordinate; ``time_groups`` sums the daily result with
    ``oracle.time_group_sum`` over the groups ``_time_group_ids`` forms.  Daily values are rounded to
    multiples of 2^-16 (see the module docstring)."""
    import oracle
    from climate_toolbox_b200 import Dataset
    from climate_toolbox_b200.aggregations.aggregations import _time_group_ids
    from climate_toolbox_b200.utils.utils import _day_of_year
    v = ds[variable]
    x, dims = np.asarray(v.values, dtype=np.float64), v.dims
    lat, lon = ds["lat"].values, ds["lon"].values
    if season_mask is not None:
        assert np.array_equal(season_mask.lat, lat) and np.array_equal(season_mask.lon, lon)
        doy = _day_of_year(ds[time_dim].values)[None, None, :]
        on = ((doy >= season_mask.first[:, :, None]) & (doy <= season_mask.last[:, :, None])) != \
            season_mask.wrap[:, :, None]
        dense = np.where(season_mask.missing[:, :, None], np.nan, on.astype(np.float64))   # (lat, lon, time)
        x = x * np.moveaxis(dense, [0, 1, 2], [dims.index("lat"), dims.index("lon"), dims.index(time_dim)])
    out, rd, labels = oracle.weighted_aggregate_grid_to_regions(x, dims, lat, lon, weights, aggwt, agglev,
                                                                backup_aggwt)
    out = np.ldexp(np.round(np.ldexp(out, QUANTUM)), -QUANTUM)
    t = ds[time_dim].values
    if time_groups is not None:
        gid, t = _time_group_ids(ds, time_dim, len(t), time_groups)
        out, _ = oracle.time_group_sum(out, rd, gid, time_dim)
    coords = {time_dim: t, agglev: labels}
    for d in rd:
        if d not in coords and d in ds.coords:
            coords[d] = ds[d].values
    return Dataset({variable: (rd, out)}, coords=coords)


def _cpu_data(T, start="2019-11-01", lead=False, time_dim="time", time_kind="datetime"):
    from climate_toolbox_b200 import Dataset, synthetic
    lat, lon = synthetic.grid_labels(4.0)
    df = synthetic.weights_table(4.0, 60, seed=2)
    n = 3 * T if lead else T
    tas, _, _ = synthetic.tas_field(n, len(lat), len(lon), seed=1, nan_frac=0.01, dtype=np.float64)
    time = pd.date_range(start, periods=T).values
    if time_kind == "yyyyddd":          # the integer axis tas_poly writes: year * 1000 + day count
        time = pd.DatetimeIndex(time).year.values.astype(np.int64) * 1000 + np.arange(1, T + 1)
    coords = {time_dim: time, "lat": lat, "lon": lon}
    if lead:
        coords["model"] = ["a", "b", "c"]
        return Dataset({"tas": (("model", time_dim, "lat", "lon"), tas.reshape(3, T, len(lat), len(lon)))},
                       coords=coords), df
    return Dataset({"tas": ((time_dim, "lat", "lon"), tas)}, coords=coords), df


def _season_mask(ds, seed=21):
    from climate_toolbox_b200 import Dataset
    from climate_toolbox_b200.utils.utils import get_daily_growing_season_mask
    lat, lon = ds["lat"].values, ds["lon"].values
    rng = np.random.default_rng(seed)
    plant = rng.integers(1, 366, (len(lat), len(lon))).astype(np.float64)
    harv = rng.integers(1, 366, (len(lat), len(lon))).astype(np.float64)
    harv[rng.random(harv.shape) < 0.05] = np.nan
    plant[rng.random(plant.shape) < 0.05] = np.nan
    gd = Dataset({"variable": (("z", "latitude", "longitude"), np.stack([plant, harv]))},
                 coords={"z": np.array([1, 2]), "latitude": lat, "longitude": lon + 180})
    return get_daily_growing_season_mask(ds["lat"], ds["lon"], ds["time"], gd)


def _irregular_labels(T):
    """String labels in runs of irregular length, some of them one day long."""
    lengths = [3, 29, 1, 31, 33, 2, 1, 40, 7]
    lab, k = [], 0
    while len(lab) < T:
        lab += ["p{:03d}".format(k)] * lengths[k % len(lengths)]
        k += 1
    return np.array(lab[:T])


def _same(got, ref, name, time_dim="time", agglev="hierid"):
    g, r = got[name], ref[name]
    if g.dims != r.dims or g.shape != r.shape:
        return False, "dims/shape {} {} != {} {}".format(g.dims, g.shape, r.dims, r.shape)
    if not np.array_equal(np.asarray(got[time_dim].values), np.asarray(ref[time_dim].values)):
        return False, "time labels {} != {}".format(got[time_dim].values, ref[time_dim].values)
    if not np.array_equal(got[agglev].values, ref[agglev].values):
        return False, "region labels differ"
    gv, rv = np.asarray(g.values), np.asarray(r.values)
    if not np.array_equal(gv, rv, equal_nan=True):
        bad = ~((gv == rv) | (np.isnan(gv) & np.isnan(rv)))
        return False, "{} of {} values differ".format(int(bad.sum()), bad.size)
    return True, ""


def _cpu_cases(rank, world, T):
    from climate_toolbox_b200.aggregations.aggregations import _time_group_ids
    from climate_toolbox_b200.parallel import aggregate_time_sharded
    rows = []

    def case(name, ds, df, time_dim="time", **opts):
        try:
            got = aggregate_time_sharded(ds, "tas", "popwt", "hierid", df, aggregate_fn=_stand_in,
                                         time_dim=time_dim, **opts)
            ref = _stand_in(ds, "tas", "popwt", "hierid", weights=df, time_dim=time_dim, **opts)
            rows.append((name,) + _same(got, ref, "tas", time_dim))
        except Exception as e:      # noqa: BLE001
            rows.append((name, False, repr(e)[:300]))

    ds, df = _cpu_data(T)
    case("daily", ds, df)
    case("blocks10", ds, df, time_groups=10)
    case("blocks100", ds, df, time_groups=100)
    case("labels", ds, df, time_groups=_irregular_labels(T))
    case("year_datetime", ds, df, time_groups="year")
    ds_i, _ = _cpu_data(T, time_kind="yyyyddd")
    case("year_yyyyddd", ds_i, df, time_groups="year")
    ds500, _ = _cpu_data(500)
    case("year_500_days", ds500, df, time_groups="year")
    ds_m, _ = _cpu_data(T, lead=True)
    case("model_daily", ds_m, df)
    case("model_blocks10", ds_m, df, time_groups=10)
    case("model_year", ds_m, df, time_groups="year")
    m = _season_mask(ds)
    case("season_daily", ds, df, season_mask=m)
    case("season_year", ds, df, season_mask=m, time_groups="year")
    case("season_blocks10", ds, df, season_mask=m, time_groups=10)
    ds_d, _ = _cpu_data(T, time_dim="day")
    case("time_dim_year", ds_d, df, time_dim="day", time_groups="year")

    # gather=False: every rank's groups carry their global labels, and the parts summed over ranks (in rank
    # order) are the gathered result
    for spec in (10, 100, "year"):
        name = "partials_{}".format(spec)
        try:
            part = aggregate_time_sharded(ds, "tas", "popwt", "hierid", df, gather=False, aggregate_fn=_stand_in,
                                          time_groups=spec)
            full = aggregate_time_sharded(ds, "tas", "popwt", "hierid", df, aggregate_fn=_stand_in,
                                          time_groups=spec)
            parts = [None] * world
            dist.all_gather_object(parts, (np.asarray(part["time"].values), np.asarray(part["tas"].values)))
            gid, glabels = _time_group_ids(ds, "time", T, spec)
            acc = np.zeros(full["tas"].shape)
            seen = np.zeros(len(glabels), dtype=bool)
            for lab, vals in parts:
                cols = np.searchsorted(glabels, lab) if len(lab) else np.zeros(0, dtype=np.int64)
                assert np.array_equal(glabels[cols], lab), "partial labels are not global group labels"
                acc[cols] = np.where(seen[cols][:, None], acc[cols] + vals, vals)
                seen[cols] = True
            ok = seen.all() and np.array_equal(acc, full["tas"].values, equal_nan=True)
            rows.append((name, bool(ok), "" if ok else "partials do not sum to the gathered result"))
        except Exception as e:      # noqa: BLE001
            rows.append((name, False, repr(e)[:300]))

    # a spec the single-process call refuses is refused on every rank, with the same message
    for name, spec in (("bad_str", "month"), ("bad_len", np.arange(T + 1)), ("bad_runs", np.arange(T) % 2),
                       ("bad_block", 0)):
        try:
            _time_group_ids(ds, "time", T, spec)
            want = None
        except ValueError as e:
            want = str(e)
        try:
            aggregate_time_sharded(ds, "tas", "popwt", "hierid", df, aggregate_fn=_stand_in, time_groups=spec)
            rows.append((name, False, "no error"))
        except ValueError as e:
            rows.append((name, want is not None and str(e) == want, "{!r} vs {!r}".format(str(e), want)))
    return rows


@pytest.mark.parametrize("T", [70, 140, 40])
@pytest.mark.parametrize("world", [2, 3, 4])
def test_time_sharded_cpu_matches_unsharded(world, T):
    """Daily, block-length, label-array and annual groups, partial outputs, a leading dim, the season gate and
    another time dim name: every rank's gathered result equals the unsharded stand-in.  T = 40 at world 4
    leaves two ranks without days; a block of 100 days at T = 140 and world 4 spans three ranks."""
    res = run_ranks(_cpu_cases, world, T)
    assert not _failures(res), _failures(res)


# ----------------------------------------------------------------------------
# one-GPU tier: real kernels, ranks sharing device 0, gloo on host results
# ----------------------------------------------------------------------------
EDD_T = 288.15


def _gpu_inputs(T, start="2019-11-01"):
    from climate_toolbox_b200 import DataArray, Dataset, synthetic
    from climate_toolbox_b200.transformations.transformations import snyder_edd, tas_poly
    lat, lon = synthetic.grid_labels(1.0)
    tas, tmin, tmax = synthetic.tas_field(T, len(lat), len(lon), seed=7, nan_frac=0.001)
    time = pd.date_range(start, periods=T)
    dims = ("time", "lat", "lon")
    coords = {"time": time, "lat": lat, "lon": lon}
    plain = Dataset({"tas": (dims, tas)}, coords=coords)
    poly = tas_poly(plain, [1, 2, 3, 4], ["p1", "p2", "p3", "p4"])
    edd = Dataset(coords=coords)
    edd["edd"] = snyder_edd(DataArray(tmin, dims=dims, coords=coords, attrs={"units": "K"}),
                            DataArray(tmax, dims=dims, coords=coords, attrs={"units": "K"}), EDD_T)
    return {"lat": lat, "lon": lon, "time": time, "tas": tas, "tmin": tmin, "tmax": tmax,
            "plain": plain, "poly": poly, "edd": edd}


def _oracle_daily(inp, which, names, df, aggwt, mask_dense=None):
    """float64 oracle daily values [name][time, R] and their scale (sum w|f| / sum w) on the days the
    aggregation sees."""
    import oracle
    dims = ("time", "lat", "lon")
    fs = []
    if which == "plain":
        fs = [inp["tas"].astype(np.float64)]
    elif which == "edd":
        fs = [oracle.snyder_edd(inp["tmin"], inp["tmax"], EDD_T)]
    else:
        fs = [oracle.tas_poly(inp["tas"], inp["time"], p)[0] for p in range(1, len(names) + 1)]
    out = []
    for f in fs:
        if mask_dense is not None:
            f = f * mask_dense
        ref, rd, _ = oracle.weighted_aggregate_grid_to_regions(f, dims, inp["lat"], inp["lon"], df, aggwt, "hierid")
        sc = oracle.weighted_aggregate_grid_to_regions(np.abs(f), dims, inp["lat"], inp["lon"], df, aggwt, "hierid")[0]
        out.append((ref, np.nan_to_num(sc)))
    return out


def _gpu_cases(rank, world, T, smem_budget, R):
    import oracle
    from climate_toolbox_b200 import synthetic
    from climate_toolbox_b200.aggregations.aggregations import _time_group_ids, weighted_aggregate_grid_to_regions
    from climate_toolbox_b200.parallel import aggregate_time_sharded
    from climate_toolbox_b200.utils.utils import get_daily_growing_season_mask
    torch.cuda.set_device(0)
    inp = _gpu_inputs(T)
    df = synthetic.weights_table(1.0, R, seed=1234)
    lat, lon = inp["lat"], inp["lon"]
    rng = np.random.default_rng(21)
    plant = rng.integers(1, 366, (len(lat), len(lon))).astype(np.float64)
    harv = rng.integers(1, 366, (len(lat), len(lon))).astype(np.float64)
    harv[rng.random(harv.shape) < 0.05] = np.nan
    plant[rng.random(plant.shape) < 0.05] = np.nan
    from climate_toolbox_b200 import Dataset
    gd = Dataset({"variable": (("z", "latitude", "longitude"), np.stack([plant, harv]))},
                 coords={"z": np.array([1, 2]), "latitude": lat, "longitude": lon + 180})
    mask = get_daily_growing_season_mask(inp["plain"]["lat"], inp["plain"]["lon"], inp["plain"]["time"], gd)
    dense = oracle.growing_season_mask(plant, harv, inp["time"].dayofyear.values).transpose(2, 0, 1)
    opts = {"smem_budget": smem_budget}
    rows = []

    def run(which, names, aggwt, **kw):
        ds = inp[which]
        got = aggregate_time_sharded(ds, names, aggwt, "hierid", df, **opts, **kw)
        ref = weighted_aggregate_grid_to_regions(ds, names, aggwt, "hierid", weights=df, **opts, **kw)
        return ds, got, ref

    def head(got, ref, names):
        for n in names:
            if got[n].dims != ref[n].dims or got[n].shape != ref[n].shape:
                return "{}: dims/shape {} {} != {} {}".format(n, got[n].dims, got[n].shape, ref[n].dims, ref[n].shape)
        if not np.array_equal(np.asarray(got["time"].values), np.asarray(ref["time"].values)):
            return "time labels differ"
        if not np.array_equal(got["hierid"].values, ref["hierid"].values):
            return "region labels differ"
        return ""

    def daily(name, which, names, aggwt="popwt", **kw):
        try:
            _, got, ref = run(which, names, aggwt, **kw)
            err = head(got, ref, names)
            for n in names:
                if not err and not np.array_equal(bits(got[n].values), bits(ref[n].values)):
                    err = "{}: {} of {} values differ in their bits".format(
                        n, int((bits(got[n].values) != bits(ref[n].values)).sum()), got[n].values.size)
            rows.append((name, not err, err))
        except Exception as e:      # noqa: BLE001
            rows.append((name, False, traceback.format_exc()[-1500:]))

    def grouped(name, which, names, spec, aggwt="popwt", season=False):
        try:
            kw = {"season_mask": mask} if season else {}
            ds, got, ref = run(which, names, aggwt, time_groups=spec, **kw)
            day = weighted_aggregate_grid_to_regions(ds, names, aggwt, "hierid", weights=df, **opts, **kw)
            Tn = ds.dims["time"]
            gid, glabels = _time_group_ids(ds, "time", Tn, spec)
            k = group_ranks(gid, Tn, world)
            n_days = np.bincount(gid, minlength=len(glabels))
            err = head(got, ref, names)
            orc = _oracle_daily(inp, which, names, df, aggwt, dense if season else None)
            worst = 0.0
            for n, (od, osc) in zip(names, orc):
                if err:
                    break
                g, r = np.asarray(got[n].values), np.asarray(ref[n].values)        # (group, R)
                inside = k == 1
                if not np.array_equal(bits(g[inside]), bits(r[inside])):
                    err = "{}: a group inside one shard differs in its bits".format(n)
                    break
                if not np.array_equal(np.isnan(g), np.isnan(r)):
                    err = "{}: NaN pattern differs".format(n)
                    break
                S, _ = oracle.time_group_sum(np.abs(np.nan_to_num(day[n].values)), ("time", "hierid"), gid)
                bound = 2.0 * n_days[:, None] * U * S
                fin = ~np.isnan(r)
                over = np.abs(g - r)[fin] > bound[fin]
                if over.any():
                    err = "{}: {} crossing values exceed the bound".format(n, int(over.sum()))
                    break
                worst = max(worst, float(np.max(np.where(fin, np.abs(g - r) / np.maximum(bound, 1e-300), 0))))
                og, _ = oracle.time_group_sum(od, ("time", "hierid"), gid)
                osg, _ = oracle.time_group_sum(osc, ("time", "hierid"), gid)
                for a in (g, r):
                    e = _rel_err(a, og, osg + 1e-300)
                    if e > TOL:
                        err = "{}: {} against the oracle".format(n, e)
            rows.append((name, not err, err or "groups across shards: {} of {}, worst |diff| / bound {:.3g}".format(
                int((k > 1).sum()), len(k), worst)))
        except Exception as e:      # noqa: BLE001
            rows.append((name, False, traceback.format_exc()[-1500:]))

    poly = ["p1", "p2", "p3", "p4"]
    daily("identity", "plain", ["tas"])
    daily("tas_poly_1_4", "poly", poly)
    daily("snyder_edd", "edd", ["edd"])
    daily("season", "plain", ["tas"], aggwt="cropwt", season_mask=mask)
    grouped("identity_blocks10", "plain", ["tas"], 10)
    grouped("identity_blocks100", "plain", ["tas"], 100)
    grouped("identity_year", "plain", ["tas"], "year")
    grouped("tas_poly_year_yyyyddd", "poly", poly, "year")
    grouped("snyder_edd_labels", "edd", ["edd"], _irregular_labels(T))
    grouped("season_year", "plain", ["tas"], "year", aggwt="cropwt", season=True)
    grouped("season_blocks10", "plain", ["tas"], 10, aggwt="cropwt", season=True)
    return rows


def _rel_err(got, ref, scale):
    from conftest import rel_err
    return rel_err(got, ref, scale)


_GPU_PLANS = [pytest.param(0, 3000, id="whole_regions"), pytest.param(8 * 1024, 40, id="split_regions")]


@pytest.mark.gpu
@pytest.mark.parametrize("smem_budget,R", _GPU_PLANS)
@pytest.mark.parametrize("world,T", [(2, 140), (3, 140), (3, 40)])
def test_time_sharded_gpu_matches_single_process(world, T, smem_budget, R):
    """Host inputs through ``aggregate_time_sharded`` on two or three ranks sharing device 0: daily results
    (identity, tas_poly orders 1..4, Snyder EDD, the season gate) bit for bit against the single-process
    call; time groups bit for bit inside a shard, at the summation-order bound across shards, and both
    against the oracle.  140 days from 2019-11-01 put a year boundary and a leap day in the data; 40 days
    on three ranks leave the last rank without days."""
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    res = run_ranks(_gpu_cases, world, T, smem_budget, R, timeout=240)
    assert not _failures(res), _failures(res)
    if smem_budget:
        from climate_toolbox_b200 import _engine as E
        from climate_toolbox_b200 import synthetic
        lat, lon = synthetic.grid_labels(1.0)
        plan = E.get_plan(E.GridSpec(lat, lon), synthetic.weights_table(1.0, R, seed=1234), "popwt", "hierid",
                          smem_budget=smem_budget, compact=True)
        assert plan.info["n_split_regions"] > 0


# ----------------------------------------------------------------------------
# multi-GPU tier: NCCL, one rank per GPU, device-level entry points
# ----------------------------------------------------------------------------
def _multi_gpu_cases(rank, world, T):
    from climate_toolbox_b200 import Dataset, synthetic
    from climate_toolbox_b200 import _engine as E
    from climate_toolbox_b200 import _native as N
    from climate_toolbox_b200.aggregations.aggregations import weighted_aggregate_grid_to_regions
    from climate_toolbox_b200.parallel import (PeerOutput, aggregate_shard_overlapped, aggregate_shard_p2p,
                                               aggregate_time_sharded)
    dev = torch.device("cuda", rank)
    lat, lon = synthetic.grid_labels(1.0)
    df = synthetic.weights_table(1.0, 3000, seed=1234)
    ncell = len(lat) * len(lon)
    xs = []
    for seed in (3, 4, 5):
        tas, _, _ = synthetic.tas_field(T, len(lat), len(lon), seed=seed, nan_frac=0.001)
        xs.append(torch.from_numpy(tas).to(dev).view(T, ncell))
    plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", device=dev)
    rows = []

    def same(name, got, ref):
        got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
        ref = ref.detach().cpu().numpy() if isinstance(ref, torch.Tensor) else np.asarray(ref)
        ok = got.shape == ref.shape and np.array_equal(bits(got), bits(ref))
        rows.append((name, ok, "" if ok else "shape {} vs {}, or bits differ".format(got.shape, ref.shape)))

    def single(x, kind="identity", params=(), n_out=1):
        out = E.aggregate_device(plan, x, None, N.LAYOUT_TIME_MAJOR, ncell, None, T, kind, params, n_out)
        torch.cuda.synchronize(dev)
        return out.clone()

    # the Dataset-level entry on device inputs, the result kept on the device
    ds = Dataset({"tas": (("time", "lat", "lon"), xs[0].view(T, len(lat), len(lon)))},
                 coords={"time": np.arange(T), "lat": lat, "lon": lon})
    got = aggregate_time_sharded(ds, "tas", "popwt", "hierid", df, keep_on_device=True)
    ref = weighted_aggregate_grid_to_regions(ds, "tas", "popwt", "hierid", weights=df, keep_on_device=True)
    rows.append(("time_sharded_on_device", bool(got["tas"].physical.is_cuda), "result left the device"))
    same("time_sharded_vs_single_process", got["tas"].physical, ref["tas"].physical)
    same("time_sharded_vs_aggregate_device", got["tas"].physical, single(xs[0])[0].T)

    # the overlapped gather: its own buffer and a caller's, called twice in a row with different inputs
    poly = (273.15, 1.0, 2.0)
    for pieces in (1, 3):
        for own in (True, False):
            for kind, params, n_out in (("identity", (), 1), ("poly", poly, 2)):
                caller = None if own else torch.empty((n_out, plan.R, T), dtype=torch.float64, device=dev)
                for call, x in enumerate(xs[:2]):
                    out, _ = aggregate_shard_overlapped(plan, x, None, ncell, T, kind, params, n_out, pieces=pieces,
                                                        out=caller)
                    torch.cuda.synchronize(dev)
                    if caller is not None:
                        rows.append(("overlapped_caller_out_is_returned", out is caller, ""))
                    same("overlapped_pieces{}_{}_{}_call{}".format(pieces, "own" if own else "caller", kind, call),
                         out, single(x, kind, params, n_out))
                    dist.barrier()

    # the gather fused into the kernel (fused stores to every peer; pushed rows, SM copy or copy engine)
    po = PeerOutput(plan, T)
    try:
        pos = np.asarray(plan.region_order())
        for mode, pieces, x in (("fused", 1, xs[0]), ("push", 1, xs[1]), ("push", 2, xs[2])):
            got = aggregate_shard_p2p(plan, x, None, ncell, T, po, mode=mode, pieces=pieces)
            torch.cuda.synchronize(dev)
            ref = single(x)
            tag = "p2p_{}_pieces{}".format(mode, pieces)
            same(tag + "_gathered", got, ref)
            raw = po.raw.cpu().numpy()
            same(tag + "_raw", raw[:, pos, :] if mode == "fused" else raw, ref)
            torch.cuda.synchronize(dev)
            dist.barrier()          # nobody's next call stores into a buffer this rank still reads
    finally:
        po.close()
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("T", [70, 33])
@pytest.mark.parametrize("world", [2, 4])
def test_multi_gpu_sharded_matches_single_gpu(world, T):
    """NCCL, one rank per GPU, device-resident float32 inputs: ``aggregate_time_sharded`` with the result
    kept on the device, ``aggregate_shard_overlapped`` (1 and 3 pieces, own and caller's output, buffers
    reused by a second call) and ``aggregate_shard_p2p`` (fused, push, push in two pieces), every rank's
    result bit for bit against the single-GPU launch of the same plan.  T = 33 leaves a one-day last shard
    at world 2 and two empty shards at world 4."""
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n < world:
        pytest.skip("needs {} GPUs, {} visible".format(world, n))
    res = run_ranks(_multi_gpu_cases, world, T, backend="nccl", timeout=240)
    assert not _failures(res), _failures(res)
