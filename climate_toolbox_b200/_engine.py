"""Host planner + launcher for the grid->region aggregation kernels.

Python here is plumbing only: it factorises region labels, keeps a content-keyed
plan cache (the analogue of ``toolz.memoize`` at
``/root/reference/climate_toolbox/aggregations/aggregations.py:127``), owns device
buffers through torch, and calls the C-ABI in ``libctb.so``.  All arithmetic of
the path runs in the CUDA kernels; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import threading
from collections import OrderedDict

import numpy as np
import pandas as pd
import torch

from . import _native as N

__all__ = ["Plan", "GridSpec", "TimeGroups", "get_plan", "get_time_groups", "aggregate_device", "aggregate_host",
           "aggregate_daily", "DailySource", "materialize_deferred", "default_device", "launch_count"]

_NP2CTB = {np.dtype("float32"): N.F32, np.dtype("float64"): N.F64}
_T2CTB = {torch.float32: N.F32, torch.float64: N.F64}
_KIND = {"identity": N.TR_IDENTITY, "poly": N.TR_POLY, "edd": N.TR_EDD, "gdd": N.TR_GDD, "bins": N.TR_BINS,
         "rcspline": N.TR_RCSPLINE}


def default_device():
    if not torch.cuda.is_available():
        raise RuntimeError("climate_toolbox_b200 needs a CUDA device (B200, sm_100a); "
                           "there is no CPU fallback for the aggregation path")
    return torch.device("cuda", torch.cuda.current_device())


def launch_count():
    return int(N.lib().ctb_launch_count())


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))


class GridSpec:
    """Coordinate labels of the spatial axes + where each label physically lives."""

    def __init__(self, lat, lon, lat_phys=None, lon_phys=None, nlat_phys=None, nlon_phys=None):
        self.lat = np.ascontiguousarray(lat, dtype=np.float64)
        self.lon = np.ascontiguousarray(lon, dtype=np.float64)
        self.lat_phys = None if lat_phys is None else np.ascontiguousarray(lat_phys, dtype=np.int32)
        self.lon_phys = None if lon_phys is None else np.ascontiguousarray(lon_phys, dtype=np.int32)
        self.nlat_phys = int(nlat_phys if nlat_phys is not None else len(self.lat))
        self.nlon_phys = int(nlon_phys if nlon_phys is not None else len(self.lon))

    def digest(self, h):
        for a in (self.lat, self.lon, self.lat_phys, self.lon_phys):
            h.update(b"-" if a is None else a.tobytes())
        h.update(np.array([self.nlat_phys, self.nlon_phys]).tobytes())


class Plan:
    """Owns a ``ctb_plan*`` (region-sorted CSR + staging bundles on the device)."""

    def __init__(self, handle, device, region_labels, n_rows):
        self._h = handle
        self.device = device
        self.region_labels = region_labels
        self.n_rows = n_rows
        info = N.PlanInfo()
        N.check(N.lib().ctb_plan_get_info(self._h, C.byref(info)))
        self.info = info.as_dict()
        self._tix_cache = {}
        self._ws_cache = {}

    R = property(lambda s: s.info["n_regions"])
    compact = property(lambda s: s.info["n_packed_cells"] > 0)

    def _host_array(self, fn, n, dtype, ptr):
        out = np.empty(n, dtype=dtype)
        N.check(getattr(N.lib(), fn)(self._h, ptr(out)))
        return out

    def row_cells(self):
        """Physical flat gridcell index of every weights row (the index map)."""
        return self._host_array("ctb_plan_row_cells", self.n_rows, np.int32, _ip)

    def row_weights(self):
        return self._host_array("ctb_plan_row_weights", self.n_rows, np.float64, _dp)

    def den(self):
        return self._host_array("ctb_plan_den", self.R, np.float64, _dp)

    def region_order(self):
        """Position of every region along the bundle sequence (spatial order): a permutation of 0..R-1."""
        return self._host_array("ctb_plan_region_order", self.R, np.int32, _ip)

    def algorithmic_bytes(self, T, n_in, elem_bytes, n_out):
        """SURVEY.md section 8(d): T*(n_in*s_in*U + n_out*8*R) + 12*nnz."""
        i = self.info
        return T * (n_in * elem_bytes * i["n_cells_distinct"] + n_out * 8 * i["n_regions"]) \
            + 12 * i["nnz"]

    def time_index_device(self, tix):
        if tix is None:
            return None
        # arrays of another dtype or shape can hold the same bytes ([5, 0] int32 and [5] int64)
        key = (tix.dtype.str, tix.shape, hashlib.sha1(tix.tobytes()).hexdigest())
        if key not in self._tix_cache:
            if len(self._tix_cache) > 16:
                self._tix_cache.clear()
            self._tix_cache[key] = torch.as_tensor(tix.astype(np.int32), device=self.device)
        return self._tix_cache[key]

    def close(self):
        if self._h:
            N.lib().ctb_plan_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_PLAN_CACHE: "OrderedDict[str, Plan]" = OrderedDict()
_PLAN_CACHE_SIZE = 8
_PLAN_FAST = {}   # fingerprint of (DataFrame object, columns, grid) -> content key


def _buf_fp(u8):
    """Position-sensitive 64-bit fingerprint of a byte buffer (``ctb_fingerprint``: 8 polynomial lanes
    over the 64-bit words; about 0.1 ms for the 3.4 MB of a 420k-row column; swapping two different
    words, or editing any word, changes it)."""
    u8 = np.ascontiguousarray(u8)
    if u8.size == 0:
        return 0
    return int(N.lib().ctb_fingerprint(u8.ctypes.data, u8.size))


def _col_fp(values):
    """Content fingerprint of one weights column, position-sensitive, for the plan-cache fast path.
    Numeric columns and Arrow-backed string columns (the pandas >= 3 default) are hashed from their
    buffers; object columns through the (cached) hashes of their elements."""
    pa = getattr(values, "_pa_array", None)
    if pa is not None:
        h = [len(values)]
        for ch in pa.chunks:
            h.append((ch.offset, len(ch), ch.null_count))
            for b in ch.buffers():
                h.append(-1 if b is None else _buf_fp(np.frombuffer(b, dtype=np.uint8)))
        return tuple(h)
    a = np.asarray(values)
    if a.dtype == object or a.dtype.kind in "US":
        return hash(tuple(a.tolist()))
    a = np.ascontiguousarray(a)
    return (str(a.dtype), _buf_fp(a.view(np.uint8).reshape(-1)))


_FP_POOL = None


def _columns_fp(weights, cols):
    """Fingerprints of several columns, hashed concurrently (the native hash releases the GIL)."""
    global _FP_POOL
    vals = [weights[c].values for c in cols]
    if len(weights) < 50000:
        return tuple(_col_fp(v) for v in vals)
    if _FP_POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _FP_POOL = ThreadPoolExecutor(max_workers=4, thread_name_prefix="ctb-fp")
    return tuple(_FP_POOL.map(_col_fp, vals))


def region_codes(labels):
    """Sorted-unique region labels and the code of every row (NaN label -> -1);
    ``xarray.groupby`` orders groups like ``pd.factorize(sort=True)``."""
    codes, uniques = pd.factorize(np.asarray(labels), sort=True)
    return codes.astype(np.int32), np.asarray(uniques)


def get_plan(grid, weights, aggwt, agglev, backup_aggwt="areawt", stage_bytes=4, device=None,
             smem_budget=0, cache=True, compact=False, elem_bytes=4, trusted=False, cell_gate=None):
    """Build (or fetch) the device plan for (grid, weights[lat, lon, agglev, aggwt, backup]).
    ``cell_gate``: uint32 per PHYSICAL gridcell (growing-season gate, ``_native.gate_word``) or None."""
    if cell_gate is not None:
        cell_gate = np.ascontiguousarray(cell_gate, dtype=np.uint32).reshape(-1)
        if cell_gate.size != grid.nlat_phys * grid.nlon_phys:
            raise ValueError("cell_gate has {} entries for {} gridcells".format(
                cell_gate.size, grid.nlat_phys * grid.nlon_phys))
    gate_fp = None if cell_gate is None else _buf_fp(cell_gate.view(np.uint8))
    device = device or default_device()
    for col in ("lat", "lon", agglev, aggwt, backup_aggwt):
        if col not in weights:
            raise KeyError(col)
    # fast path: the same DataFrame object asked for again (the reference memoises its weights
    # frame per path, aggregations.py:127).  Guarded by position-sensitive content fingerprints of
    # EVERY column the plan is built from -- the region column included -- so an in-place edit or
    # permutation of the frame rebuilds the plan (under 1 ms per call at 420k rows).
    fp = None
    if cache:
        gh = hashlib.sha1()
        grid.digest(gh)
        with np.errstate(all="ignore"):
            fp = (id(weights), len(weights), aggwt, agglev, backup_aggwt, stage_bytes, smem_budget,
                  bool(compact), int(elem_bytes), str(device), gh.hexdigest(), gate_fp,
                  # `trusted`: a private frame of the caller (never edited in place): identity is enough
                  () if trusted else _columns_fp(weights, ("lat", "lon", aggwt, backup_aggwt, agglev)))
        hit = _PLAN_FAST.get(fp)
        if hit is not None and hit in _PLAN_CACHE:
            _PLAN_CACHE.move_to_end(hit)
            return _PLAN_CACHE[hit]
    row_lat = np.ascontiguousarray(weights["lat"].values, dtype=np.float64)
    row_lon = np.ascontiguousarray(weights["lon"].values, dtype=np.float64)
    wp = np.ascontiguousarray(weights[aggwt].values, dtype=np.float64)
    wb = np.ascontiguousarray(weights[backup_aggwt].values, dtype=np.float64)
    codes, labels = region_codes(weights[agglev].values)
    codes = np.ascontiguousarray(codes)

    h = hashlib.sha1()
    grid.digest(h)
    for a in (row_lat, row_lon, wp, wb, codes):
        h.update(a.tobytes())
    h.update(repr((stage_bytes, smem_budget, bool(compact), int(elem_bytes), str(device), len(labels))).encode())
    if cell_gate is not None:
        h.update(cell_gate.tobytes())
    key = h.hexdigest()
    if cache and key in _PLAN_CACHE:
        _PLAN_CACHE.move_to_end(key)
        _PLAN_FAST[fp] = key
        return _PLAN_CACHE[key]

    opts = N.PlanOpts()
    opts.stage_bytes_per_cell_day = int(stage_bytes)
    opts.smem_budget_bytes = int(smem_budget)
    opts.compact = 1 if compact else 0
    opts.elem_bytes = int(elem_bytes)
    opts.cell_gate = cell_gate.ctypes.data if cell_gate is not None else None
    handle = C.c_void_p()
    bad_row, bad_axis = C.c_int64(-1), C.c_int32(-1)
    rc = N.lib().ctb_plan_build(
        _dp(grid.lat), len(grid.lat), _ip(grid.lat_phys), grid.nlat_phys,
        _dp(grid.lon), len(grid.lon), _ip(grid.lon_phys), grid.nlon_phys,
        _dp(row_lat), _dp(row_lon), _ip(codes), _dp(wp), _dp(wb), len(row_lat), len(labels),
        C.byref(opts), device.index or 0, C.byref(handle), C.byref(bad_row), C.byref(bad_axis))
    N.check(rc)
    plan = Plan(handle, device, labels, len(row_lat))
    if cache:
        _PLAN_CACHE[key] = plan
        _PLAN_FAST[fp] = key
        while len(_PLAN_CACHE) > _PLAN_CACHE_SIZE:
            _PLAN_CACHE.popitem(last=False)
        if len(_PLAN_FAST) > 4 * _PLAN_CACHE_SIZE:
            for k in [k for k, v in _PLAN_FAST.items() if v not in _PLAN_CACHE]:
                del _PLAN_FAST[k]
    return plan


class TimeGroups:
    """Owns a ``ctb_time_groups*``: the output column of every day for the fused time reduction
    (annual sums).  ``group_of_day``: int array, starts at 0, grows by 0 or 1 per day."""

    def __init__(self, group_of_day, device):
        g = np.ascontiguousarray(group_of_day, dtype=np.int32)
        self._h = C.c_void_p()
        self.device = device
        self.T = int(g.size)
        N.check(N.lib().ctb_time_groups_create(_ip(g) if g.size else None, g.size, device.index or 0,
                                               C.byref(self._h)))
        self.n_groups = int(N.lib().ctb_time_groups_count(self._h))

    def close(self):
        if self._h:
            N.lib().ctb_time_groups_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_GROUPS_CACHE: "OrderedDict[tuple, TimeGroups]" = OrderedDict()


def get_time_groups(group_of_day, device=None):
    device = device or default_device()
    g = np.ascontiguousarray(group_of_day, dtype=np.int32)
    key = (str(device), g.size, hashlib.sha1(g.tobytes()).hexdigest())
    hit = _GROUPS_CACHE.get(key)
    if hit is None:
        hit = _GROUPS_CACHE[key] = TimeGroups(g, device)
        while len(_GROUPS_CACHE) > 16:
            _GROUPS_CACHE.popitem(last=False)
    else:
        _GROUPS_CACHE.move_to_end(key)
    return hit


_PARAMS_CACHE = {}


def _params_array(kind, params):
    """(float64 array, ctypes pointer) of a transform's parameters; cached: the launch path of a small
    problem (config 1: a 10 us kernel) is host-bound."""
    key = (kind, tuple(float(p) for p in params))
    hit = _PARAMS_CACHE.get(key)
    if hit is None:
        a = np.ascontiguousarray(params, dtype=np.float64)
        if len(_PARAMS_CACHE) > 64:
            _PARAMS_CACHE.clear()
        hit = _PARAMS_CACHE[key] = (a, (_dp(a) if a.size else None))
    return hit


def _stream_ptr(device, stream=None):
    s = stream if stream is not None else torch.cuda.current_stream(device)
    return C.c_void_p(s.cuda_stream)


def _workspace(plan, T, n_out, layout, variant, groups, workspace):
    staged = (variant & 0xff) != N.VARIANT_DIRECT and layout == N.LAYOUT_TIME_MAJOR
    key = (int(T), int(n_out), staged)
    ws_bytes = plan._ws_cache.get(key) if groups is None else None
    if ws_bytes is None:
        L = N.lib()
        if groups is not None:
            ws_bytes = L.ctb_aggregate_grouped_workspace_bytes(plan._h, groups._h, n_out)
        else:
            ws_bytes = L.ctb_aggregate_workspace_bytes(plan._h, T, n_out) if staged else 0
        if groups is None:
            if len(plan._ws_cache) > 64:
                plan._ws_cache.clear()
            plan._ws_cache[key] = ws_bytes
    if ws_bytes and (workspace is None or workspace.numel() * 8 < ws_bytes):
        workspace = torch.empty((ws_bytes + 7) // 8, dtype=torch.float64, device=plan.device)
    return workspace


def _launch(plan, p0, p1, ctb_dtype, layout, stride, tix, T, kind, params, n_out, variant, out, out_ld,
            workspace, stream, groups=None, t_begin=0, flush=True, doy=None, peer_ptrs=None, peer_row=None):
    """Raw-pointer call of ctb_aggregate_ex (p0/p1: device or mapped-host addresses).  With ``groups``
    the result is [n_out, R, n_groups]; ``doy`` (int array, day of year of every day of the time axis)
    switches the growing-season gate of a plan built with ``cell_gate`` on; ``peer_ptrs`` (device
    addresses laid out like ``out``) makes the kernel store every result to all of them."""
    dev = plan.device
    L = N.lib()
    if out is None:
        out = torch.empty((n_out, plan.R, T if groups is None else groups.n_groups), dtype=torch.float64,
                          device=dev)
    workspace = _workspace(plan, T, n_out, layout, variant, groups, workspace)
    tix_d = plan.time_index_device(tix)
    doy_d = plan.time_index_device(doy)
    pa, pp = _params_array(kind, params)
    o = N.AggOpts()
    o.groups = groups._h if groups is not None else None
    o.t_begin, o.flush = int(t_begin), 1 if flush else 0
    o.day_of_year = doy_d.data_ptr() if doy_d is not None else None
    if peer_ptrs:
        arr = (C.c_void_p * len(peer_ptrs))(*[int(p) for p in peer_ptrs])
        o.peer_out, o.n_peer_out = arr, len(peer_ptrs)
        o.peer_row = peer_row.data_ptr() if peer_row is not None else None
    rc = L.ctb_aggregate_ex(
        plan._h, C.c_void_p(p0), C.c_void_p(p1) if p1 else None, ctb_dtype, layout, int(stride),
        C.c_void_p(tix_d.data_ptr()) if tix_d is not None else None, int(T),
        _KIND[kind], pp, int(pa.size), int(n_out), C.byref(o), C.c_void_p(out.data_ptr()), int(out_ld),
        C.c_void_p(workspace.data_ptr()) if workspace is not None else None,
        int(workspace.numel() * 8) if workspace is not None else 0, int(variant),
        _stream_ptr(dev, stream))
    N.check(rc)
    return out


def aggregate_device(plan, x0, x1, layout, stride, tix, T, kind="identity", params=(), n_out=1,
                     variant=N.VARIANT_AUTO, out=None, out_ld=0, stream=None, workspace=None, groups=None,
                     t_begin=0, flush=True, doy=None, peer_ptrs=None, peer_row=None):
    """Launch the fused kernel on device-resident inputs.

    ``x0`` / ``x1``: contiguous CUDA tensors (f32/f64).  ``tix``: numpy int array of
    physical time positions or None.  Returns ``out`` ([n_out, R, T] float64 CUDA; with
    ``groups`` -- a :class:`TimeGroups` -- [n_out, R, n_groups]: the days of every group summed).
    """
    dev = plan.device
    if x0.device != dev or not x0.is_contiguous():
        raise ValueError("input must be a contiguous tensor on {}".format(dev))
    if x0.dtype not in _T2CTB:
        raise TypeError("unsupported dtype {}".format(x0.dtype))
    if x1 is not None and (x1.dtype != x0.dtype or x1.shape != x0.shape):
        raise ValueError("the two inputs must agree in dtype and shape")
    return _launch(plan, x0.data_ptr(), x1.data_ptr() if x1 is not None else 0, _T2CTB[x0.dtype], layout,
                   stride, tix, T, kind, params, n_out, variant, out, out_ld, workspace, stream, groups,
                   t_begin, flush, doy, peer_ptrs, peer_row)


def _all_pinned(xs):
    try:
        return all(torch.from_numpy(x).is_pinned() for x in xs)
    except Exception:
        return False


# (device index, slot, k) -> [pinned staging tensor for packed chunks, event of the last H2D copy that
# read it].  The buffers are reused across calls, so the event outlives the call that recorded it: a
# later call (or another thread) waits for it before it packs into the buffer again.
_PINNED = {}
_HOST_LOCK = threading.Lock()   # one packed host call at a time: they share the buffers and the cores
TRANSFER_BYTES = {"h2d": 0, "d2h": 0}   # bytes actually copied across PCIe by this module (bench e2e)


# ---------------------------------------------------------------------------
# pinned result buffers
# ---------------------------------------------------------------------------
# Results go back to the host through pinned memory (a pageable D2H runs at 2 GB/s).  A fresh
# cudaHostAlloc of a 285 MB block costs 200-400 ms, and torch's caching host allocator hands out a new
# block whenever the previous one is not provably idle -- so the blocks are pooled here and return to
# the pool when the last numpy view of a result is garbage collected.
_RESULT_POOL = {}
_RESULT_OUT = {}    # size -> number of blocks ever allocated (in the pool or out with a result)


class _PinnedOwner:
    """Base object of a result array: exposes a pinned block through __array_interface__."""

    def __init__(self, block, shape, typestr):
        self.__array_interface__ = {"shape": tuple(int(v) for v in shape), "typestr": typestr,
                                    "data": (block.data_ptr(), False), "version": 3}


RESULT_POOL_CAP_BYTES = int(os.environ.get("CTB_RESULT_POOL_BYTES", str(2 << 30)))


def _release_result(block):
    """A result's last view is gone: keep its pinned block for the next result of that size, unless the
    idle blocks already hold RESULT_POOL_CAP_BYTES of page-locked memory (then it is freed)."""
    idle = sum(b.numel() for blocks in _RESULT_POOL.values() for b in blocks)
    if idle + block.numel() <= RESULT_POOL_CAP_BYTES:
        _RESULT_POOL.setdefault(block.numel(), []).append(block)
    else:
        _RESULT_OUT[block.numel()] = max(0, _RESULT_OUT.get(block.numel(), 1) - 1)


def pinned_result_like(t):
    """(torch view, numpy array) over a pooled pinned block shaped like the CUDA tensor ``t``."""
    import weakref
    nbytes = max(1, t.numel() * t.element_size())
    free = _RESULT_POOL.setdefault(nbytes, [])
    if not free and _RESULT_OUT.get(nbytes, 0) > 0:
        # blocks of this size are out with results that may already be unreachable but sit in a
        # reference cycle: a collection (tens of ms) is far cheaper than a fresh cudaHostAlloc
        import gc
        gc.collect()
    if free:
        block = free.pop()
    else:
        block = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        _RESULT_OUT[nbytes] = _RESULT_OUT.get(nbytes, 0) + 1
    view = block[: t.numel() * t.element_size()].view(t.dtype).view(t.shape)
    owner = _PinnedOwner(block, t.shape, np.dtype(str(t.dtype).replace("torch.", "")).str)
    arr = np.asarray(owner)
    weakref.finalize(owner, _release_result, block)
    return view, arr


def _pinned_buffer(key, nbytes):
    """Staging buffer `key`, idle: waits for the last H2D copy that read it (this or an earlier call)."""
    ent = _PINNED.get(key)
    if ent is not None and ent[1] is not None:
        ent[1].synchronize()
        ent[1] = None
    if ent is None or ent[0].numel() < nbytes:
        ent = [torch.empty(nbytes, dtype=torch.uint8, pin_memory=True), None]
        _PINNED[key] = ent
    return ent


def pack_threads():
    """Host threads ``ctb_host_pack`` may use: CTB_PACK_THREADS, else three quarters of the usable
    cores (with every core packing, the CUDA driver's own threads and the caller get descheduled and
    single calls take 2-3x longer, profiles/r1_e2e_notes.md)."""
    threads = int(os.environ.get("CTB_PACK_THREADS", "0"))
    if threads:
        return threads
    try:
        ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        ncpu = os.cpu_count() or 1
    return max(1, (3 * ncpu) // 4)


def _chunk_days(chunk_bytes, day_bytes):
    """Days per time chunk: as many as ``chunk_bytes`` holds, in multiples of 32, at least 32."""
    return max(32, int(chunk_bytes // max(day_bytes, 1)) // 32 * 32)


def _run_chunks(plan, T, days, stage, kind, params, n_out, variant, groups, out, doy, host_out=None,
                layout=N.LAYOUT_TIME_MAJOR):
    """Aggregate T days in time chunks of ``days``, one launch each -> ``(out, host_out filled)``; ``out`` is
    allocated when None.
    ``stage(ci, t0, n, done)`` queues on the current stream what makes days t0 .. t0 + n - 1 readable and returns
    ``(bufs, stride, tix)``: 1 or 2 input tensors (on the device, or CPU tensors over mapped pinned memory), kept
    referenced until their launch is queued; ``done[k]`` is the event recorded after the launch of chunk k.
    With ``host_out`` (a pinned [n_out, R, T] tensor) and no time groups, each chunk's columns go back on a second
    stream while the next chunk is staged (PCIe is full duplex); the caller then only has to synchronise."""
    dev = plan.device
    if out is None:
        out = torch.empty((n_out, plan.R, T if groups is None else groups.n_groups), dtype=torch.float64, device=dev)
    if T == 0 or plan.R == 0:
        return (out.zero_() if groups is not None else out), False
    # one workspace for the whole call: split-region rows of a chunk, or -- with time groups -- of the whole
    # time axis plus the per-tile partial sums
    ws = _workspace(plan, min(days, T), n_out, layout, variant, groups, None)
    main = torch.cuda.current_stream(dev)
    back = torch.cuda.Stream(dev) if host_out is not None and groups is None else None
    done = []
    for ci, t0 in enumerate(range(0, T, days)):
        n = min(T, t0 + days) - t0
        bufs, stride, tix = stage(ci, t0, n, done)
        if groups is None:      # columns t0 .. t0 + n - 1 of out, and those days of the day-of-year axis
            o, ld, d = _OffsetOut(out, t0), T, None if doy is None else doy[t0: t0 + n]
        else:                   # a window of the time groups; the last chunk flushes them
            o, ld, d = out, 0, doy
        _launch(plan, bufs[0].data_ptr(), bufs[1].data_ptr() if len(bufs) > 1 else 0, _T2CTB[bufs[0].dtype], layout,
                stride, tix, n, kind, params, n_out, variant, o, ld, ws, None, groups, t0, t0 + n == T, d)
        ev = torch.cuda.Event()
        ev.record(main)
        done.append(ev)
        if back is not None:
            back.wait_event(ev)
            N.check(N.lib().ctb_copy_rows_to_host(
                C.c_void_p(host_out.data_ptr() + 8 * t0), 8 * T, C.c_void_p(out.data_ptr() + 8 * t0), 8 * T,
                8 * n, n_out * plan.R, C.c_void_p(back.cuda_stream)))
            TRANSFER_BYTES["d2h"] += 8 * n * n_out * plan.R
    if back is not None:
        out.record_stream(back)
        main.wait_stream(back)
    return out, back is not None


def _aggregate_packed(plan, pack, n_planes, itemsize, T, kind, params, n_out, variant, groups, out, host_out=None,
                      chunk_bytes=4 << 30, doy=None):
    """Compact plan whose inputs the GPU packs itself: ``pack(t0, n, bufs)`` queues on the current stream
    what fills ``bufs`` (``n_planes`` fresh device tensors [n, n_packed_cells] of ``itemsize``-byte elements)
    with days t0 .. t0 + n - 1, then the kernel aggregates the packed planes.  Packs and kernels queue on one
    stream; ``out`` and ``host_out`` as :func:`_run_chunks`."""
    width = plan.info["n_packed_cells"]
    tdt = torch.float32 if itemsize == 4 else torch.float64
    days = _chunk_days(chunk_bytes, width * itemsize * n_planes)
    if host_out is not None and groups is None:
        days = min(days, max(32, (-(-T // 4) + 31) // 32 * 32))      # about four chunks: the last D2H is exposed

    def stage(ci, t0, n, done):
        bufs = [torch.empty((n, width), dtype=tdt, device=plan.device) for _ in range(n_planes)]
        pack(t0, n, bufs)
        return bufs, width, None

    return _run_chunks(plan, T, days, stage, kind, params, n_out, variant, groups, out, doy, host_out)


def _aggregate_pull(plan, xs, stride, tix, T, kind, params, n_out, variant, groups, out, host_out=None,
                    chunk_bytes=4 << 30, doy=None):
    """Pinned host arrays + compact plan: the GPU packs for itself (``ctb_pull_pack`` reads the
    referenced pieces over PCIe into a packed device buffer), then the kernel aggregates the packed
    planes.  No host core touches the data (:func:`_aggregate_packed`)."""
    dev = plan.device
    itemsize = xs[0].dtype.itemsize
    tix_d = plan.time_index_device(tix)

    def pack(t0, n, bufs):
        for x, b in zip(xs, bufs):
            N.check(N.lib().ctb_pull_pack(
                plan._h, C.c_void_p(x.ctypes.data), _NP2CTB[x.dtype], int(stride),
                C.c_void_p(tix_d.data_ptr()) if tix_d is not None else None, int(t0), int(n),
                C.c_void_p(b.data_ptr()), _stream_ptr(dev)))
        TRANSFER_BYTES["h2d"] += len(xs) * n * plan.info["n_pieces_distinct"] * 4 * itemsize

    return _aggregate_packed(plan, pack, len(xs), itemsize, T, kind, params, n_out, variant, groups, out, host_out,
                             chunk_bytes, doy)


# ---------------------------------------------------------------------------
# sub-daily sources: daily mean / min / max reduced while the referenced pieces are packed
# ---------------------------------------------------------------------------
_DAILY_OP = {"mean": N.DAILY_MEAN, "min": N.DAILY_MIN, "max": N.DAILY_MAX}
DAILY_STAGE_BYTES = 256 << 20    # pinned staging slot of a pageable sub-daily source


class DailySource:
    """What ``ctb_pull_pack_daily`` reads for one deferred daily variable (``utils.resample_daily``): the
    sub-daily source as 2-D [t_phys, ncell], its steps per day, its first step and the physical day of
    every day."""

    def __init__(self, var):
        d = var.deferred
        self.how, self.S, self.t0, self.day = d.params
        src = d.sources[0]
        self.phys = x = src.physical
        if isinstance(x, torch.Tensor) and not x.is_cuda:
            x = x.numpy()
        if isinstance(x, torch.Tensor):
            x = (x if x.dtype in _T2CTB else x.to(torch.float64)).contiguous()
            self.dtype = _T2CTB[x.dtype]
            self.pinned = False
        else:
            x = np.ascontiguousarray(x if x.dtype in _NP2CTB else x.astype(np.float64))
            self.dtype = _NP2CTB[x.dtype]
            self.pinned = _all_pinned([x])
        self.on_device = isinstance(x, torch.Tensor)
        self.nlat_phys, self.nlon_phys = int(x.shape[1]), int(x.shape[2])
        self.stride = self.nlat_phys * self.nlon_phys
        self.x = x.reshape(x.shape[0], self.stride)
        self.itemsize = 4 if self.dtype == N.F32 else 8
        self.lat_phys, self.lon_phys = src.takes.get("lat"), src.takes.get("lon")
        self.T = len(self.day)

    def ptr(self):
        base = self.x.data_ptr() if self.on_device else self.x.ctypes.data
        return base + self.t0 * self.stride * self.itemsize

    def same_read(self, other):
        """Both read the same steps of the same buffer."""
        return (self.phys is other.phys and (self.S, self.t0) == (other.S, other.t0) and
                np.array_equal(self.day, other.day))


def _day_arg(plan, day):
    """Device day index for the kernel, or None when day d is physical day d."""
    if np.array_equal(day, np.arange(len(day))):
        return None
    return plan.time_index_device(np.asarray(day))


def _pull_daily(plan, src, dsts, d0, n):
    """Queue ``ctb_pull_pack_daily`` for days d0 .. d0 + n - 1 of ``src`` into ``dsts`` ({how: device tensor
    [>= n, n_packed_cells]}, all from one read).  A pageable host source is staged first: whole days are
    copied into pinned buffers (those of the host path, two in turn) that the kernel then reads."""
    dev = plan.device
    L = N.lib()
    ops = 0
    for how in dsts:
        ops |= _DAILY_OP[how]

    def call(x_ptr, day, t_begin, k, m):
        day_d = _day_arg(plan, day) if day is not None else None
        ptrs = {h: C.c_void_p(t.data_ptr() + k * t.shape[1] * t.element_size()) for h, t in dsts.items()}
        N.check(L.ctb_pull_pack_daily(
            plan._h, C.c_void_p(x_ptr), src.dtype, int(src.stride), int(src.S),
            C.c_void_p(day_d.data_ptr()) if day_d is not None else None, int(t_begin), int(m), ops,
            ptrs.get("mean"), ptrs.get("min"), ptrs.get("max"), _stream_ptr(dev)))
        if not src.on_device:
            TRANSFER_BYTES["h2d"] += m * src.S * plan.info["n_pieces_distinct"] * 4 * src.itemsize

    if n == 0:
        return
    if src.on_device or src.pinned:
        call(src.ptr(), src.day, d0, 0, n)
        return
    day = src.day[d0: d0 + n]
    per_day = src.S * src.stride * src.itemsize
    cap = max(1, DAILY_STAGE_BYTES // per_day)
    np_dt = np.float32 if src.itemsize == 4 else np.float64
    main = torch.cuda.current_stream(dev)
    k, slot = 0, 0
    with _HOST_LOCK:
        while k < n:
            lo = hi = int(day[k])
            m = 1
            while k + m < n and lo <= day[k + m] < lo + cap:
                hi = max(hi, int(day[k + m]))
                m += 1
            ent = _pinned_buffer((dev.index or 0, "daily", slot), cap * per_day)   # waits for its last reader
            stage = ent[0][: (hi + 1 - lo) * per_day].numpy().view(np_dt).reshape(-1, src.stride)
            first = src.t0 + lo * src.S
            np.copyto(stage, src.x[first: first + (hi + 1 - lo) * src.S])
            call(ent[0].data_ptr(), day[k: k + m] - lo, 0, k, m)
            ev = torch.cuda.Event()
            ev.record(main)
            ent[1] = ev
            k += m
            slot ^= 1


def aggregate_daily(plan, srcs, kind="identity", params=(), n_out=1, variant=N.VARIANT_AUTO, groups=None,
                    host_out=None, doy=None):
    """Deferred daily reductions of sub-daily data -> CUDA tensor [n_out, R, T] (with ``groups``:
    [n_out, R, n_groups]).  ``srcs``: 1 or 2 (:class:`DailySource`, how).  Each chunk of days is
    reduce-packed by ``ctb_pull_pack_daily`` into packed daily planes (float64 for the mean, the source
    dtype for min / max; the plan is built for that element size) and aggregated by the compact-plan
    launch; sources that read the same steps -- the daily minimum and maximum of one variable -- come from
    one call.  ``host_out``: as :func:`aggregate_host`."""
    calls = []          # [(DailySource, {how: plane index})]
    for i, (src, how) in enumerate(srcs):
        for c in calls:
            if c[0].same_read(src) and how not in c[1]:
                c[1][how] = i
                break
        else:
            calls.append((src, {how: i}))

    def pack(t0, n, bufs):
        for src, planes in calls:
            _pull_daily(plan, src, {h: bufs[i] for h, i in planes.items()}, t0, n)

    itemsize = 8 if srcs[0][1] == "mean" else srcs[0][0].itemsize
    out, filled = _aggregate_packed(plan, pack, len(srcs), itemsize, srcs[0][0].T, kind, params, n_out, variant,
                                    groups, None, host_out[0] if host_out is not None else None, doy=doy)
    if host_out is not None:
        host_out[1] = filled
    return out


_FULL_GRID = {}


def _full_grid_plan(nlat, nlon, elem_bytes, dev):
    """Compact plan that references every gridcell of an nlat x nlon grid once: its packed planes are the
    physical planes (one run from piece 0)."""
    hit = _FULL_GRID.get((nlat, nlon))
    if hit is None:
        ii, jj = np.meshgrid(np.arange(nlat, dtype=np.float64), np.arange(nlon, dtype=np.float64), indexing="ij")
        df = pd.DataFrame({"lat": ii.ravel(), "lon": jj.ravel(), "_r": np.zeros(ii.size, dtype=np.int32),
                           "_w": np.ones(ii.size)})
        grid = GridSpec(np.arange(nlat, dtype=np.float64), np.arange(nlon, dtype=np.float64))
        if len(_FULL_GRID) > 8:
            _FULL_GRID.clear()
        hit = _FULL_GRID[(nlat, nlon)] = (grid, df)
    grid, df = hit
    return get_plan(grid, df, "_w", "_r", "_w", stage_bytes=elem_bytes, device=dev, compact=True,
                    elem_bytes=elem_bytes, trusted=True)


def daily_device(var, dev):
    """A deferred daily variable evaluated for the whole grid by ``ctb_pull_pack_daily``: CUDA tensor
    [days, lat, lon] with the variable's lat / lon takes applied."""
    src = DailySource(var)
    es = 8 if src.how == "mean" else src.itemsize
    plan = _full_grid_plan(src.nlat_phys, src.nlon_phys, es, dev)
    o = torch.empty((src.T, plan.info["n_packed_cells"]), dtype=torch.float32 if es == 4 else torch.float64,
                    device=dev)
    _pull_daily(plan, src, {src.how: o}, 0, src.T)
    t = o[:, : src.stride].reshape(src.T, src.nlat_phys, src.nlon_phys)
    for ax, pos in ((1, src.lat_phys), (2, src.lon_phys)):
        if pos is not None:
            t = t.index_select(ax, torch.as_tensor(pos, device=dev))
    return t.contiguous()


def _ingest_route(layout, compact, variant, dtype_ok, aligned, pinned, zero_copy=None, ingest=None):
    """Route of host inputs to the kernel: "cell_major", "zero_copy", "pull", "host_pack" or "full_copy" (see
    :func:`aggregate_host`).  ``aligned``: 16-byte aligned inputs and planes, whole 4-cell pieces; ``zero_copy`` /
    ``ingest`` None: ``CTB_ZERO_COPY`` / ``CTB_INGEST``."""
    if layout == N.LAYOUT_CELL_MAJOR:
        return "cell_major"
    if zero_copy is None:
        # opt-in: on the round-1 box the in-place read moved 2.5 GB at ~7 GB/s (16-byte requests
        # over PCIe) and lost to copying all 6 GB at ~21 GB/s (profiles/r1_e2e_notes.md)
        zero_copy = os.environ.get("CTB_ZERO_COPY", "0") == "1"
    if zero_copy and not compact and (variant & 0xff) != N.VARIANT_DIRECT and dtype_ok and pinned:
        return "zero_copy"
    if ingest is None:
        ingest = os.environ.get("CTB_INGEST", "auto")
    if compact and ingest in ("auto", "pull") and dtype_ok and aligned and pinned:
        return "pull"
    if ingest == "pull":
        raise ValueError("ingest='pull' needs a compact plan and 16-byte aligned inputs in pinned host memory")
    return "host_pack" if compact else "full_copy"


def aggregate_host(plan, xs, layout, stride, tix, T, kind="identity", params=(), n_out=1,
                   variant=N.VARIANT_AUTO, chunk_bytes=192 << 20, zero_copy=None, threads=0, groups=None,
                   ingest=None, host_out=None, doy=None):
    """Host (numpy) inputs -> CUDA tensor [n_out, R, T] (with ``groups``: [n_out, R, n_groups]).

    ``xs``: list of 1 or 2 C-contiguous numpy arrays viewed as 2-D
    (TIME_MAJOR: [t_phys, stride]; CELL_MAJOR: [ncell, stride]).

    * compact plan (the default for TIME_MAJOR host inputs), source in PINNED memory: the GPU pulls
      the referenced gridcells over PCIe itself (``ctb_pull_pack``; ``ingest="pull"``);
    * compact plan, pageable source (``ingest="pack"``): time chunks are PACKED on the
      host (``ctb_host_pack``, all cores) into pinned staging buffers that hold only the
      referenced gridcells, copied asynchronously and reduced while the next chunk is packed;
    * full-grid plan: time chunks are copied whole (pinned: asynchronously at PCIe speed;
      pageable: through the driver's staging), or -- opt-in, pinned arrays only -- read in
      place by the kernel (zero-copy).

    ``host_out``: ``[pinned tensor [n_out, R, T], False]`` -- a path that can return the result in
    time chunks while later chunks are still in flight fills the tensor and sets the flag (the
    caller synchronises the stream); otherwise the flag stays False and the caller copies ``out``.
    """
    dev = plan.device
    if len(xs) > 1 and (xs[1].dtype != xs[0].dtype or xs[1].shape != xs[0].shape):
        raise ValueError("the two inputs must agree in dtype and shape")
    itemsize = xs[0].dtype.itemsize
    aligned = ((stride * itemsize) % 16 == 0 and plan.info["n_cells_grid"] % 4 == 0 and
               all(x.ctypes.data % 16 == 0 for x in xs))
    route = _ingest_route(layout, plan.compact, variant, xs[0].dtype in _NP2CTB, aligned, _all_pinned(xs),
                          zero_copy, ingest)
    if route == "pull":
        out, filled = _aggregate_pull(plan, xs, stride, tix, T, kind, params, n_out, variant, groups, None,
                                      host_out[0] if host_out is not None else None, doy=doy)
        if host_out is not None:
            host_out[1] = filled
        return out
    if route in ("cell_major", "zero_copy"):
        if route == "zero_copy":
            # pinned (mapped) host arrays: the kernel reads them in place over PCIe, so only the
            # referenced gridcells (~30 % of a global land/ocean grid) cross the bus
            variant = N.VARIANT_STAGED | N.VARIANT_MAPPED_HOST

        def stage(ci, t0, n, done):
            if route == "zero_copy":
                return [torch.from_numpy(x) for x in xs], stride, tix
            TRANSFER_BYTES["h2d"] += sum(x.nbytes for x in xs)
            return [torch.from_numpy(x).to(dev, non_blocking=True) for x in xs], stride, tix

        return _run_chunks(plan, T, T, stage, kind, params, n_out, variant, groups, None, doy, layout=layout)[0]

    # host_pack / full_copy: two staging slots in turn, copied on a second stream
    threads = threads or pack_threads()
    main = torch.cuda.current_stream(dev)
    copy_stream = torch.cuda.Stream(dev)
    copy_stream.wait_stream(main)
    tix_full = None if tix is None else np.ascontiguousarray(tix, dtype=np.int64)
    width = plan.info["n_packed_cells"] if plan.compact else xs[0].shape[1]
    days = _chunk_days(chunk_bytes, width * itemsize * len(xs))
    tdt = torch.float32 if itemsize == 4 else torch.float64
    dbuf = {}
    di = dev.index or 0

    def stage(ci, t0, n, done):
        slot = ci % 2
        rel = None
        pin_ents = []
        if plan.compact:
            # pack on the host (GIL released) while the previous chunk is in flight
            srcs = []
            for k, x in enumerate(xs):
                ent = _pinned_buffer((di, slot, k), days * width * itemsize)   # waits for its last H2D
                pin_ents.append(ent)
                N.check(N.lib().ctb_host_pack(
                    plan._h, C.c_void_p(x.ctypes.data), _NP2CTB[x.dtype], int(stride),
                    tix_full.ctypes.data_as(C.POINTER(C.c_int64)) if tix_full is not None else None,
                    int(t0), int(n), C.c_void_p(ent[0].data_ptr()), int(threads)))
                srcs.append(ent[0][: n * width * itemsize].view(tdt).view(n, width))
        else:
            sub = np.arange(t0, t0 + n) if tix_full is None else tix_full[t0: t0 + n]
            lo, hi = int(sub.min()), int(sub.max()) + 1
            srcs = [torch.from_numpy(x)[lo:hi] for x in xs]
            if tix_full is not None and not np.array_equal(sub - lo, np.arange(n)):
                rel = sub - lo
        with torch.cuda.stream(copy_stream):
            if ci >= 2:
                copy_stream.wait_event(done[ci - 2])     # the last launch that read this slot
            cur = []
            for k, src in enumerate(srcs):
                b = dbuf.get((slot, k))
                if b is None or b.shape[0] < src.shape[0]:
                    b = torch.empty((max(src.shape[0], days + 8), src.shape[1]), dtype=tdt, device=dev)
                    b.record_stream(main)
                    dbuf[(slot, k)] = b
                b[: src.shape[0]].copy_(src, non_blocking=True)
                TRANSFER_BYTES["h2d"] += src.numel() * src.element_size()
                cur.append(b)
            ready = torch.cuda.Event()
            ready.record(copy_stream)
            for ent in pin_ents:
                ent[1] = ready      # outlives this call: the next packer of the buffer waits for it
        main.wait_event(ready)
        return cur, width, rel

    with _HOST_LOCK:
        return _run_chunks(plan, T, days, stage, kind, params, n_out, variant, groups, None, doy, layout=layout)[0]


class _OffsetOut:
    """Pointer view of ``out[:, :, t0:]`` for a time-chunked launch (out_ld = total T)."""

    def __init__(self, base, t0):
        self._p = base.data_ptr() + 8 * t0
        self.base = base

    def data_ptr(self):
        return self._p


# ---------------------------------------------------------------------------
# deferred variables (`.values` of a transformed / reindexed variable)
# ---------------------------------------------------------------------------
def _to_device(v, dev):
    """Materialise a (non-deferred or daily) Variable on the device with its lazy takes applied."""
    if v.deferred is not None and v.deferred.kind == "daily":
        return daily_device(v, dev)
    a = v.physical
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
    t = t.to(dev)
    for ax, d in enumerate(v.dims):
        if d in v.takes:
            t = t.index_select(ax, torch.as_tensor(v.takes[d], device=dev))
    return t.contiguous()


def materialize_deferred(var):
    """Evaluate a deferred pointwise transform with the CUDA kernel (ctb_transform)."""
    d = var.deferred
    dev = default_device()
    if d.kind == "reindex":
        return d.params[0]()  # closure built by aggregations._pointwise_reindex
    if d.kind == "daily":
        return daily_device(var, dev).cpu().numpy()
    srcs = [_to_device(s, dev) for s in d.sources]
    if srcs[0].dtype not in _T2CTB:
        srcs = [s.to(torch.float64) for s in srcs]
    n = srcs[0].numel()
    out = torch.empty((1,) + tuple(srcs[0].shape), dtype=torch.float64, device=dev)
    pa, pp = _params_array(d.kind, d.params)
    rc = N.lib().ctb_transform(
        C.c_void_p(srcs[0].data_ptr()), C.c_void_p(srcs[1].data_ptr()) if len(srcs) > 1 else None,
        _T2CTB[srcs[0].dtype], n, _KIND[d.kind], pp, int(pa.size), 1,
        C.c_void_p(out.data_ptr()), _stream_ptr(dev))
    N.check(rc)
    return out[0].cpu().numpy()
