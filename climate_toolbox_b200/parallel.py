"""Multi-GPU: the path shards along time (every day is independent given the plan).

One process per GPU; each rank builds the (deterministic, ~7 MB) plan itself and
aggregates a contiguous block of days.  There is NO data-path collective; the only
exchange is the optional final gather of the region x time outputs (NCCL all_gather over
NVLink on GPUs, gloo in the CPU tests).  SURVEY.md section 8(e).

* :func:`shard_range` / :func:`shard_sizes`   contiguous day blocks, multiples of the 32-day tile
* :func:`all_gather_time`                     one collective + one strided copy into ``[.., T]``
* :func:`aggregate_shard_overlapped`          device level: the shard is aggregated in time pieces and
                                              the all_gather of piece k runs on a side stream while
                                              the kernel of piece k+1 runs
* :class:`PeerOutput` / :func:`aggregate_shard_p2p`   the gather fused into the kernel: the epilogue
                                              stores every result into all ranks' buffers over NVLink
                                              peer memory (CUDA IPC), no collective
* :func:`aggregate_time_sharded`              Dataset level (any leading dims)
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

__all__ = ["bind_to_gpu_numa_node", "shard_range", "shard_sizes", "all_gather_time", "aggregate_shard_overlapped",
           "aggregate_time_sharded", "PeerOutput", "aggregate_shard_p2p"]


def bind_to_gpu_numa_node(device_index):
    """Pin this process to the CPU cores next to its GPU (NVML's affinity mask) -- call it BEFORE the
    host arrays are allocated: pinned pages then live on the socket whose PCIe root the GPU hangs off,
    and the GPU-side ingest (``ctb_pull_pack``) of eight ranks does not cross the inter-socket link.
    Returns the core list, or None when NVML / the scheduler call is unavailable."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(device_index))
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = [64 * w + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return allowed
    except Exception:  # noqa: BLE001 -- best effort: no NVML, no permission, not Linux
        pass
    return None


def shard_sizes(T, world_size, align=32):
    """Days per rank: contiguous blocks, multiples of ``align`` (the kernel's time tile)
    except the last non-empty one; earlier ranks take the extra tiles."""
    tiles = (T + align - 1) // align
    base, extra = divmod(tiles, world_size)
    sizes, left = [], T
    for r in range(world_size):
        n = min(left, (base + (1 if r < extra else 0)) * align)
        sizes.append(n)
        left -= n
    return sizes


def shard_range(T, world_size, rank, align=32):
    sizes = shard_sizes(T, world_size, align)
    t0 = sum(sizes[:rank])
    return t0, t0 + sizes[rank]


def _gather_padded(block, tmax, group):
    """``block`` [M, n] (n <= tmax) from every rank -> [world, M, tmax] (columns >= n undefined)."""
    world = dist.get_world_size(group)
    M = block.shape[0]
    if block.shape[1] == tmax and block.is_contiguous():
        send = block
    else:
        send = torch.empty((M, tmax), dtype=block.dtype, device=block.device)
        send[:, : block.shape[1]] = block
    recv = torch.empty((world * M, tmax), dtype=block.dtype, device=block.device)   # concatenation along dim 0
    dist.all_gather_into_tensor(recv, send, group=group)
    return recv.view(world, M, tmax)


def _scatter_columns(full2d, recv, sizes, col0s, c0=0):
    """full2d[:, col0s[r] + c0 : col0s[r] + c0 + sizes[r]] = recv[r, :, :sizes[r]] for every rank r:
    ONE strided copy when the shards tile the row evenly, else one per rank."""
    world = len(sizes)
    pitch = full2d.shape[1] // world if world else 0
    even = world > 0 and pitch * world == full2d.shape[1] and len(set(sizes)) == 1 and \
        all(col0s[r] == r * pitch for r in range(world))
    if even and sizes[0] > 0:
        full2d.view(full2d.shape[0], world, pitch)[:, :, c0: c0 + sizes[0]].copy_(
            recv[:, :, : sizes[0]].permute(1, 0, 2))
        return
    for r, n in enumerate(sizes):
        if n > 0:
            full2d[:, col0s[r] + c0: col0s[r] + c0 + n].copy_(recv[r, :, :n])


def all_gather_time(local, T, group=None, align=32):
    """Gather per-rank ``[..., T_local]`` blocks (time LAST, any leading dims) into ``[..., T]`` on
    every rank.  Ranks may hold different T_local (ragged last shards): one collective on blocks padded
    to the largest shard, then the valid columns are copied straight into the final layout."""
    world = dist.get_world_size(group)
    sizes = shard_sizes(T, world, align)
    lead = tuple(local.shape[:-1])
    M = int(np.prod(lead)) if lead else 1
    recv = _gather_padded(local.reshape(M, local.shape[-1]), max(sizes), group)
    full = torch.empty((M, T), dtype=local.dtype, device=local.device)
    _scatter_columns(full, recv, sizes, [sum(sizes[:r]) for r in range(world)])
    return full.reshape(lead + (T,))


class _ShardBuffers:
    """Streams and buffers of :func:`aggregate_shard_overlapped`, allocated once per (plan, T, n_out,
    pieces, world): a collective must not wait for ``cudaMalloc``, and blocks that are used on a side
    stream do not come back to the caching allocator quickly."""

    def __init__(self, plan, T, n_out, pieces, world, rank, gather):
        dev = plan.device
        self.sizes = shard_sizes(T, world)
        self.col0 = [sum(self.sizes[:r]) for r in range(world)]
        self.t0, self.tl = self.col0[rank], self.sizes[rank]
        tmax = max(self.sizes)
        tiles = (tmax + 31) // 32
        pieces = max(1, min(pieces, tiles))
        # piece boundaries inside a shard: the same on every rank (relative to the largest shard), 32-aligned
        self.cuts = [min(tmax, ((tiles * k) // pieces) * 32) for k in range(pieces)] + [tmax]
        self.M = n_out * plan.R
        self.loc = [torch.empty((n_out, plan.R, self.cuts[k + 1] - self.cuts[k]), dtype=torch.float64, device=dev)
                    for k in range(pieces)]
        self.recv = [torch.empty((world * self.M, self.cuts[k + 1] - self.cuts[k]), dtype=torch.float64, device=dev)
                     for k in range(pieces)] if gather else None
        self.out = torch.empty((n_out, plan.R, T), dtype=torch.float64, device=dev) if gather else None
        self.side = torch.cuda.Stream(dev) if gather else None


def aggregate_shard_overlapped(plan, x0, x1, stride, T, kind="identity", params=(), n_out=1, group=None,
                               pieces=4, gather=True, out=None):
    """Time-sharded aggregation of device-resident TIME_MAJOR inputs with the output gather
    overlapped: this rank aggregates days ``shard_range(T)`` of ``x0`` (``[T, stride]``, every rank
    holds or views the same time axis) in ``pieces`` pieces; the ``all_gather`` of piece k runs on
    a side stream while the kernel of piece k+1 runs, and lands through one strided copy in the
    final ``[n_out, R, T]`` layout.  Returns ``(out, info)``; with ``gather=False`` only the list of
    local piece blocks.  Buffers live with the plan and are reused by the next call of the same shape
    (the returned ``out`` is overwritten then)."""
    from . import _engine as E
    from . import _native as N
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = plan.device
    cache = plan.__dict__.setdefault("_shard_buffers", {})
    key = (T, n_out, pieces, world, rank, bool(gather))
    if key not in cache:
        if len(cache) > 4:
            cache.clear()
        cache[key] = _ShardBuffers(plan, T, n_out, pieces, world, rank, gather)
    sb = cache[key]
    if gather and out is None:
        out = sb.out
    main = torch.cuda.current_stream(dev)
    if gather:
        sb.side.wait_stream(main)      # the previous call's consumers of `out` / `recv` are ordered before us
    for k in range(len(sb.loc)):
        c0, c1 = sb.cuts[k], sb.cuts[k + 1]
        n = max(0, min(c1, sb.tl) - c0)           # this rank's valid days in the piece
        loc = sb.loc[k]
        if n > 0:
            a = x0[sb.t0 + c0: sb.t0 + c0 + n]
            b = x1[sb.t0 + c0: sb.t0 + c0 + n] if x1 is not None else None
            E.aggregate_device(plan, a, b, N.LAYOUT_TIME_MAJOR, stride, None, n, kind, params, n_out,
                               out=loc, out_ld=c1 - c0)
        if gather:
            ev = torch.cuda.Event()
            ev.record(main)
            sb.side.wait_event(ev)
            with torch.cuda.stream(sb.side):
                dist.all_gather_into_tensor(sb.recv[k], loc.view(sb.M, c1 - c0), group=group)
                _scatter_columns(out.view(sb.M, T), sb.recv[k].view(world, sb.M, c1 - c0),
                                 [max(0, min(c1, s) - c0) for s in sb.sizes], sb.col0, c0)
    if not gather:
        return sb.loc, {"t0": sb.t0, "t1": sb.t0 + sb.tl, "cuts": sb.cuts}
    main.wait_stream(sb.side)
    return out, {"t0": sb.t0, "t1": sb.t0 + sb.tl, "pieces": len(sb.loc),
                 "bytes_received": int(8 * sb.M * (T - sb.tl))}


class PeerOutput:
    """``[n_out, R, T]`` float64 output buffers, one per rank of a single-node group, every one mapped
    into every rank (CUDA IPC over NVLink peer memory).  :func:`aggregate_shard_p2p` makes the
    aggregation kernel store each result to all of them: the final gather of a time-sharded job
    happens inside the kernel's epilogue -- no collective, no staging copy."""

    def __init__(self, plan, T, n_out=1, group=None):
        import ctypes as C

        from . import _native as N
        self.group, self.plan, self.T, self.n_out = group, plan, T, n_out
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > N.MAX_PEERS:
            raise ValueError("at most {} ranks".format(N.MAX_PEERS))
        self.dev_index = plan.device.index or 0
        self.shape = (n_out, plan.R, T)
        nbytes = max(8, 8 * n_out * plan.R * T)
        ptr = C.c_void_p()
        handle = (C.c_ubyte * N.IPC_HANDLE_BYTES)()
        N.check(N.lib().ctb_ipc_alloc(nbytes, self.dev_index, C.byref(ptr), handle))
        self._own = ptr.value
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=plan.device)
        allh = torch.empty((self.world, N.IPC_HANDLE_BYTES), dtype=torch.uint8, device=plan.device)
        dist.all_gather_into_tensor(allh.view(-1), mine, group=group)
        allh = allh.cpu().numpy()
        self.ptrs, self._opened = [], []
        for r in range(self.world):
            if r == self.rank:
                self.ptrs.append(self._own)
                continue
            q = C.c_void_p()
            hb = (C.c_ubyte * N.IPC_HANDLE_BYTES)(*allh[r].tolist())
            N.check(N.lib().ctb_ipc_open(hb, self.dev_index, C.byref(q)))
            self.ptrs.append(q.value)
            self._opened.append(q.value)
        # this rank's buffer as a tensor (a view: the memory belongs to this object).  Its region rows are
        # in the plan's bundle order (spatial neighbours together), not in label order: one CTA's stores
        # then stay inside a few pages per peer -- with label-ordered rows a CTA touches ~28 pages per peer
        # and tile, and at 8 peers the stores thrash the TLB (3.2 ms instead of 0.4 ms for the step)
        self.raw = _tensor_from_ptr(self._own, self.shape, plan.device, self)
        pos = plan.region_order()
        self.row_of_region = torch.as_tensor(pos, device=plan.device)                 # region -> row
        self._region_rows = self.row_of_region.to(torch.int64)

        self.rows = "bundle"          # row order of ``raw`` after the last call: "bundle" (fused) or "region" (push)

    def gathered(self):
        """The full result in the reference's region order ``[n_out, R, T]`` (one device gather after the
        fused form; the buffer itself after the push form)."""
        if self.rows == "region":
            return self.raw
        return self.raw.index_select(1, self._region_rows)

    def side_stream(self):
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(self.plan.device)
        return self._side

    def push(self, t0, n, copy_engine=False):
        """Copy columns ``[t0, t0 + n)`` of this rank's buffer into every peer's (``ctb_push_rows``)."""
        import ctypes as C

        from . import _engine as E
        from . import _native as N
        arr = (C.c_void_p * self.world)(*self.ptrs)
        N.check(N.lib().ctb_push_rows(C.c_void_p(self._own), self.T, t0, n, self.n_out * self.plan.R, self.world,
                                      arr, N.PUSH_COPY_ENGINE if copy_engine else N.PUSH_SM,
                                      E._stream_ptr(self.plan.device)))

    def close(self):
        from . import _native as N
        torch.cuda.synchronize(self.plan.device)
        if dist.is_initialized():
            dist.barrier(self.group)       # nobody still writes into a buffer that is about to go
        for q in self._opened:
            N.lib().ctb_ipc_close(q, self.dev_index)
        self._opened = []
        if self._own:
            N.lib().ctb_ipc_free(self._own, self.dev_index)
            self._own = None


def _tensor_from_ptr(ptr, shape, device, owner):
    class _Mem:
        def __init__(self):
            self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (int(ptr), False),
                                             "version": 3, "strides": None}
            self.owner = owner
    return torch.as_tensor(_Mem(), device=device)


def aggregate_shard_p2p(plan, x0, x1, stride, T, peer_out, kind="identity", params=(), n_out=1, gathered=True,
                        mode="auto", pieces=1):
    """Time-sharded aggregation whose gather needs no collective: this rank aggregates days
    ``shard_range(T)`` of ``x0`` and every rank ends with the full ``[n_out, R, T]`` result in its own
    peer-mapped buffer (``peer_out``: a :class:`PeerOutput`).

    ``mode="fused"``: the kernel's epilogue stores every region-day to column ``t`` of ALL ranks'
    buffers (rows in the plan's bundle order, ``peer_out.row_of_region``; best up to 4 ranks).
    ``mode="push"``: the kernel writes this rank's own buffer and one copy kernel
    (``ctb_push_rows``) sends the finished column block to every peer as coalesced row pieces (best
    for 8 ranks: the fused form's 256-byte pieces per region and tile are too scattered for many
    destinations).  ``pieces`` > 1 pushes piece k by DMA under the kernel of piece k+1 -- measured
    slower (2-D DMA of narrow row pieces; a copy kernel cannot share an SM with the aggregation's CTAs).
    ``"auto"`` picks by the group size.  A stream-ordered barrier ends the call;
    the result comes back in the reference's label order when ``gathered`` (else ``peer_out.raw``
    in the order ``peer_out.rows`` names)."""
    from . import _engine as E
    from . import _native as N
    world, rank = peer_out.world, peer_out.rank
    if mode == "auto":
        mode = "fused" if world <= 4 else "push"
    if mode not in ("fused", "push"):
        raise ValueError("mode must be 'auto', 'fused' or 'push'")
    t0, t1 = shard_range(T, world, rank)
    n = t1 - t0
    if n > 0:
        a = x0[t0:t1]
        b = x1[t0:t1] if x1 is not None else None
        if mode == "fused":
            ptrs = [p + 8 * t0 for p in peer_out.ptrs]
            E.aggregate_device(plan, a, b, N.LAYOUT_TIME_MAJOR, stride, None, n, kind, params, n_out,
                               out=E._OffsetOut(peer_out.raw, t0), out_ld=T, peer_ptrs=ptrs,
                               peer_row=peer_out.row_of_region)
        else:
            # in `pieces` time pieces (multiples of the kernel's 32-day tiles): the push of piece k runs
            # on a side stream under the kernel of piece k+1
            step = max(32, -(-n // max(1, pieces) // 32) * 32)
            main = torch.cuda.current_stream(plan.device)
            side = peer_out.side_stream()
            for p0 in range(0, n, step):
                m = min(step, n - p0)
                E.aggregate_device(plan, a[p0:p0 + m], None if b is None else b[p0:p0 + m], N.LAYOUT_TIME_MAJOR,
                                   stride, None, m, kind, params, n_out, out=E._OffsetOut(peer_out.raw, t0 + p0),
                                   out_ld=T)
                if p0 + m < n:
                    ev = torch.cuda.Event()
                    ev.record(main)
                    side.wait_event(ev)
                    with torch.cuda.stream(side):      # DMA: the kernel's CTAs leave no room for a copy kernel
                        peer_out.push(t0 + p0, m, copy_engine=True)
                else:
                    peer_out.push(t0 + p0, m)
            if n > step:
                ev = torch.cuda.Event()
                ev.record(side)
                main.wait_event(ev)
    peer_out.rows = "bundle" if mode == "fused" else "region"
    dist.barrier(peer_out.group)      # NCCL: stream-ordered after this rank's kernels, completes when all joined
    return peer_out.gathered() if gathered else peer_out.raw


def _shard_groups(gid, T, world):
    """First global time group and number of groups of every rank's days, from the group id of every
    day of the full axis.  A group that spans a shard boundary is counted by every rank it touches."""
    firsts, counts = [], []
    for r in range(world):
        t0, t1 = shard_range(T, world, r)
        firsts.append(int(gid[t0]) if t1 > t0 else 0)
        counts.append(int(gid[t1 - 1]) - int(gid[t0]) + 1 if t1 > t0 else 0)
    return firsts, counts


def _sum_group_blocks(full2d, recv, firsts, counts):
    """full2d[:, f_r : f_r + n_r] from recv[r, :, :n_r] of every rank r, in rank order.  A group's first
    contribution is copied and a later one (the group continues from the previous shard) is added to it,
    so a group that lies inside one shard keeps the exact bits its rank computed."""
    done = 0                                       # groups [0, done) hold a contribution
    for r, (f, n) in enumerate(zip(firsts, counts)):
        if n == 0:
            continue
        k = min(n, max(0, done - f))              # leading groups continued from an earlier shard
        if k:
            full2d[:, f: f + k] += recv[r, :, :k]
        full2d[:, f + k: f + n].copy_(recv[r, :, k:n])
        done = max(done, f + n)


def aggregate_time_sharded(ds, variable, aggwt, agglev, weights, backup_aggwt="areawt", gather=True,
                           group=None, time_dim="time", aggregate_fn=None, **engine_opts):
    """``weighted_aggregate_grid_to_regions`` over a process group: every rank aggregates its own
    contiguous block of days of ``ds`` (each rank holds, or lazily views, the same Dataset) on its
    own GPU with the replicated plan; with ``gather=True`` the region x time blocks are exchanged
    once at the end (one all_gather per variable) and every rank returns the full result, otherwise
    each rank returns its block (what a job that writes per-rank files wants: 285 MB per rank and
    year-block would otherwise cross NVLink for nothing).  Variables may carry leading dims
    (ensemble member, model): everything but ``time_dim`` rides along.

    ``time_groups=`` (``"year"``, a block length or one label per step) is resolved once on the full
    time axis, so groups are the ones the single-process call forms; each rank sums the groups its days
    touch, and the gather adds the parts of a group that spans a shard boundary, in rank order.  With
    ``gather=False`` a rank returns the sums over its own days, labelled with the global group labels:
    its first and last group may then be partial, and the sum of every rank's part is the full group.

    ``aggregate_fn`` (tests) replaces the single-GPU aggregation; it must have the signature of
    ``weighted_aggregate_grid_to_regions``.
    """
    from ._xr import Dataset, Variable, from_any
    from .aggregations.aggregations import _time_group_ids
    if aggregate_fn is None:
        from .aggregations.aggregations import weighted_aggregate_grid_to_regions as aggregate_fn
    ds = from_any(ds)
    if not (dist.is_available() and dist.is_initialized()):
        return aggregate_fn(ds, variable, aggwt, agglev, weights=weights, backup_aggwt=backup_aggwt,
                            time_dim=time_dim, **engine_opts)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    T = ds.dims[time_dim]
    t0, t1 = shard_range(T, world, rank)
    spec = engine_opts.pop("time_groups", None)
    if spec is not None:
        # every rank resolves the same groups (or raises the same error) without communicating
        gid, glabels = _time_group_ids(ds, time_dim, T, spec)
        engine_opts["time_groups"] = glabels[gid[t0:t1]]              # one global label per step of the shard
    local = aggregate_fn(ds.isel(**{time_dim: np.arange(t0, t1)}), variable, aggwt, agglev,
                         weights=weights, backup_aggwt=backup_aggwt, time_dim=time_dim, **engine_opts)
    local = from_any(local)
    if not gather:
        return local
    if spec is not None:
        firsts, counts = _shard_groups(gid, T, world)
    names = [variable] if isinstance(variable, str) else list(variable)
    backend = dist.get_backend(group)
    out = Dataset()
    for name in names:
        v = local._vars[name]
        ax_t = v.dims.index(time_dim)
        a = v.physical if isinstance(v.physical, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(v.values))
        if backend == "nccl" and not a.is_cuda:
            a = a.cuda()
        blk = a.movedim(ax_t, -1).contiguous()                            # [..., T_local]
        if spec is None:
            full = all_gather_time(blk, T, group)
        else:
            lead = tuple(blk.shape[:-1])
            M = int(np.prod(lead)) if lead else 1
            recv = _gather_padded(blk.reshape(M, blk.shape[-1]), max(counts), group)
            full = torch.empty((M, len(glabels)), dtype=blk.dtype, device=blk.device)
            _sum_group_blocks(full, recv, firsts, counts)
            full = full.reshape(lead + (len(glabels),))
        full = full.movedim(-1, ax_t)                                     # back to the variable's dim order
        out[name] = Variable(v.dims, full if full.is_cuda else full.numpy(), v.attrs)
    out._coords[agglev] = local._coords[agglev]
    for d, c in ds._coords.items():
        if d in ("lat", "lon") or "lat" in c.dims or "lon" in c.dims:
            continue
        if spec is not None and time_dim in c.dims:      # the time axis is now one step per group
            if d == time_dim:
                out._coords[d] = Variable((d,), np.asarray(glabels))
            continue
        out._coords[d] = Variable(c.dims, c.values, c.attrs)
    return out
