#!/usr/bin/env python
"""Benchmark of the grid->region aggregation hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload config2|config3|config4|config1|config5] [--no-also] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic batch of the workload
(config2: 4 x 365 days of 0.25-degree tas [1460][720][1440] f32 -> 24,378 regions, popwt).
N > 1 (torchrun, one rank per GPU): `value` is weak scaling -- every rank aggregates its OWN batch
(another GCM / scenario / block of years) with the plan replicated, no data-path collective; the
`strong` block of the same line times what north_star describes: ONE 1460-day batch sharded along
time over the ranks, compute + the final NCCL gather of the region x time outputs (overlapped).
Prints ONE JSON line on rank 0.  `also` (N = 1) carries device-timed lines of the other
BASELINE.json configs and of input variants (NaN over the ocean, annual sums).
`--dump-outputs DIR` writes rank 0's result block of the last timed step, one DIR/<output>.npy per output
(float64, [regions][days]); the inputs are seeded, so two builds run with the same arguments can be compared
output for output.  The benchmark writes nothing into the repository tree.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (deg, R, T, aggwt, kind, n_in, n_out, description)
    "config1": (1.0, 3000, 365, "areawt", "identity", 1, 1,
                "synthetic 1deg daily tas 365x180x360 f32 -> 3,000 regions, areawt"),
    "config2": (0.25, 24378, 1460, "popwt", "identity", 1, 1,
                "BCSD-shaped 0.25deg daily tas 4x365x720x1440 f32 -> 24,378 hierid regions, popwt"),
    "config3": (0.25, 24378, 1460, "popwt", "poly", 1, 4,
                "fused tas_poly orders 1-4 + aggregation, 0.25deg 1460 days -> 24,378 regions, popwt"),
    "config4": (0.25, 24378, 1460, "cropwt", "edd", 2, 2,
                "fused Snyder EDD (2 thresholds) from tasmin/tasmax, 0.25deg 1460 days -> 24,378 regions, cropwt"),
    # CMIP5-ensemble scale (21 GCMs x 2 RCPs x 95 years = 3,990 model-years): one step streams a
    # slice of YEARS_PER_STEP model-years through a pool of POOL resident year buffers
    "config5": (0.25, 24378, 365, "popwt", "identity", 1, 1,
                "ensemble streaming: model-years of 365x720x1440 f32 -> 24,378 regions, popwt; "
                "8 model-years per step and rank from a pool of 4 resident buffers (full job: 3,990 model-years, "
                "model-years dealt round-robin to the ranks)"),
}
YEARS_PER_STEP, POOL, ENSEMBLE_YEARS = 8, 4, 21 * 2 * 95
METRIC = "region-days/sec"
PARAMS = {"identity": (), "poly": (273.15, 1, 2, 3, 4), "edd": (283.15, 303.15)}
KERNEL = {"identity": "agg_stream_kernel", "poly": "agg_stream_kernel", "edd": "agg_stream_kernel"}
# --dump-outputs: one file per output of the kind (the names the e2e leg gives them)
OUTPUT_NAMES = {"identity": ("tas",), "poly": ("p1", "p2", "p3", "p4"), "edd": ("edd10", "edd30")}
DUMP_BYTES = 63_000_000          # array bytes: with the .npy headers the files stay under 64 MB
# fp64-pipe lane slots per CSR entry and day of the Snyder kernel (2 thresholds): executed DFMA + DMUL + DADD +
# DSETP warp instructions x 32 / entry-days (profiles/r2_ncu_full_agg_stream_kernel_config4.json: 690 M warp
# instructions for 3.07e8 entry-days; the zero-weight padding of the quads is overhead, not work); 64 fp64
# lanes per SM and clock
SNYDER_FP64_OPS_PER_ENTRY_DAY = 72
FP64_LANES_PER_SM_CLK = 64


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_outputs(out, kind, dirname, budget=DUMP_BYTES):
    """Write the result block ``out`` [n_out][R][n_cols] (float64) as dirname/<output>.npy, one [R][n_cols]
    array per output.  A block larger than ``budget`` keeps a fixed, seeded sample of its region rows (sorted,
    the same for every run and build of the workload) and all of its columns."""
    import torch
    n_out, R, n_cols = out.shape
    rows = min(R, max(1, budget // (8 * n_out * max(1, n_cols))))
    if rows < R:
        pick = np.sort(np.random.default_rng(0).choice(R, size=rows, replace=False))
        out = out.index_select(1, torch.from_numpy(pick).to(out.device))
    host = out.cpu().numpy()
    os.makedirs(dirname, exist_ok=True)
    for name, a in zip(OUTPUT_NAMES[kind], host):
        np.save(os.path.join(dirname, name + ".npy"), a)


def config_dict(workload, T, world):
    """The `config` object: the same keys and values in both arms (the driver compares them)."""
    deg, R, _, aggwt, kind, n_in, n_out, desc = WORKLOADS[workload]
    nlat, nlon = int(round(180 / deg)), int(round(360 / deg))
    return {"workload": desc, "T": T, "grid": [nlat, nlon], "regions": R, "aggwt": aggwt,
            "input_dtype": "f32", "accumulate": "f64", "n_in": n_in, "n_out": n_out,
            "l2": "inputs larger than L2 ({:.2f} GB per step)".format(n_in * T * nlat * nlon * 4 / 1e9),
            "per_rank": "own batch, plan replicated, outputs stay sharded"}


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.sm_max = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if mask & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.004)

    def result(self):
        self.stop_flag = True
        self.join(1.0)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(self.sm)}


# --------------------------------------------------------------------------- #
# reference arm: the restated reference (numpy/pandas oracle) on the host cores
# --------------------------------------------------------------------------- #
_REF = {}


def _ref_worker(args):
    t0, t1 = args
    import oracle
    x, lat, lon, df, aggwt = _REF["x"], _REF["lat"], _REF["lon"], _REF["df"], _REF["aggwt"]
    out = oracle.weighted_aggregate_grid_to_regions(
        x[t0:t1], ("time", "lat", "lon"), lat, lon, df, aggwt, "hierid")[0]
    return float(np.nansum(out))


class CpuReference:
    """The oracle on `days` days of the workload, time-sharded over `procs` forked workers.  The pool is
    created ONCE, outside the timed passes (the workers inherit the input by fork)."""

    def __init__(self, workload, days, procs):
        import multiprocessing as mp
        from climate_toolbox_b200 import synthetic
        deg, R, T, aggwt, kind, n_in, n_out, _ = WORKLOADS[workload]
        if kind != "identity":
            raise SystemExit("reference arm runs the headline identity workloads (config1/config2)")
        lat, lon = synthetic.grid_labels(deg)
        df = synthetic.weights_table(deg, R)
        rng = np.random.default_rng(7)
        x = np.empty((days, len(lat), len(lon)), dtype=np.float32)
        for a in range(0, days, 64):                 # in slabs: the f64 temporaries of a 6 GB draw would not fit
            b = min(days, a + 64)
            x[a:b] = 288.0 + 10.0 * rng.standard_normal((b - a, len(lat), len(lon)), dtype=np.float32)
        _REF.update(x=x, lat=lat, lon=lon, df=df, aggwt=aggwt)
        self.R, self.days, self.procs = R, days, procs
        per = max(1, -(-days // procs))
        self.chunks = [(a, min(days, a + per)) for a in range(0, days, per)]
        self.pool = mp.get_context("fork").Pool(procs) if procs > 1 else None

    def one_pass(self):
        t = time.perf_counter()
        if self.pool is None:
            for c in self.chunks:
                _ref_worker(c)
        else:
            self.pool.map(_ref_worker, self.chunks)
        return time.perf_counter() - t

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 32))
    deg, R, T, aggwt, kind, n_in, n_out, desc = WORKLOADS[args.workload]
    days = args.days or T
    # the whole step of the workload when the host has the memory for it (input + the workers' f64
    # temporaries), else the largest sample that fits
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 32 << 30
    ncell = int(round(180 / deg)) * int(round(360 / deg))
    while days > 64 and days * ncell * 4 * 1.6 > 0.6 * avail:
        days //= 2
    ref = CpuReference(args.workload, days, procs)
    try:
        for _ in range(args.warmup):
            ref.one_pass()
        ts = [ref.one_pass() for _ in range(args.steps)]
    finally:
        ref.close()
    sec = float(np.mean(ts))
    v = R * days / sec
    sample = "{} of the {} days of the workload per step ({} forked workers x {} days, time-sharded; pool created " \
             "outside the timed passes)".format(days, T, procs, -(-days // procs))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "region-days/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": config_dict(args.workload, T, 1),
        "impl_note": "restated reference (oracle/oracle.py, numpy/pandas): xarray is not installable in this "
                     "image, so the unmodified reference cannot run",
        "cpu_baseline": {"value": v, "unit": "region-days/s", "cores": procs, "kind": "port",
                         "sample": sample},
        "e2e": {"value": v, "unit": "region-days/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- #
# our arm
# --------------------------------------------------------------------------- #
class Bench:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import __graft_entry__ as G
        if G._stale() and not os.environ.get("CTB_LIBRARY"):
            # the tree may be read-only: a library missing from it or older than its sources is built in a
            # temporary directory instead, removed at exit
            tmp = tempfile.mkdtemp(prefix="ctb_bench_")
            atexit.register(shutil.rmtree, tmp, True)
            os.environ["CTB_LIBRARY"] = os.path.join(tmp, "libctb.so")
            G.compile_library(os.environ["CTB_LIBRARY"])
        from climate_toolbox_b200 import _engine as E
        from climate_toolbox_b200 import _native as N
        from climate_toolbox_b200 import synthetic
        self.torch, self.dist, self.E, self.N, self.syn = torch, dist, E, N, synthetic
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("--gpus {} needs torchrun with {} ranks".format(args.gpus, args.gpus))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.cpus = None
        if self.world > 1:   # host buffers on the GPU's own socket (the e2e leg pulls them over PCIe)
            from climate_toolbox_b200.parallel import bind_to_gpu_numa_node
            self.cpus = bind_to_gpu_numa_node(self.local)
        if self.world > 1:   # ranks share the host cores for the e2e packing
            os.environ.setdefault("CTB_PACK_THREADS", str(max(1, (3 * (os.cpu_count() or 1)) // (4 * self.world))))
            dist.init_process_group("nccl", device_id=self.dev)
        self.peak, self.peak_src = _peaks()
        self._tables = {}

    # ---- helpers ---------------------------------------------------------
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def table(self, deg, R):
        if (deg, R) not in self._tables:
            self._tables[(deg, R)] = self.syn.weights_table(deg, R)
        return self._tables[(deg, R)]

    def inputs(self, workload, T, seed_off=0, variant=None):
        """Device-resident synthetic inputs of the workload ([T, ncell] f32 views)."""
        torch = self.torch
        deg, R, _, aggwt, kind, n_in, n_out, _ = WORKLOADS[workload]
        lat, lon = self.syn.grid_labels(deg)
        g = torch.Generator(device=self.dev).manual_seed(7 + self.rank + seed_off)
        shape = (T, len(lat) * len(lon))
        tas = 288.0 + 10.0 * torch.randn(shape, generator=g, device=self.dev, dtype=torch.float32)
        if n_in == 2:
            lo = tas - (3.0 * torch.randn(shape, generator=g, device=self.dev, dtype=torch.float32)).abs()
            hi = tas + (3.0 * torch.randn(shape, generator=g, device=self.dev, dtype=torch.float32)).abs()
            return [lo, hi]
        if variant in ("bcsd_like", "nan2pct"):
            df = self.table(deg, R)
            ii = np.searchsorted(lat, df["lat"].values)
            jj = np.searchsorted(lon, df["lon"].values)
            land = np.zeros(len(lat) * len(lon), dtype=bool)
            land[ii * len(lon) + jj] = True
            if variant == "bcsd_like":      # NaN over every gridcell no weights row references (ocean)
                tas[:, torch.from_numpy(~land).to(self.dev)] = float("nan")
            else:                           # 2 % of the referenced gridcells are NaN on every day
                cells = np.flatnonzero(land)
                pick = np.random.default_rng(3).choice(cells, size=len(cells) // 50, replace=False)
                tas[:, torch.from_numpy(pick).to(self.dev)] = float("nan")
        return [tas]

    def timed(self, fn, steps, warmup):
        torch = self.torch
        for _ in range(max(warmup, 3)):
            fn()
        self.barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = self.E.launch_count()
        self.barrier()
        e0.record()
        for a, b in evs:
            a.record()
            fn()
            b.record()
        e1.record()
        self.barrier()
        launches = self.E.launch_count() - n0
        total_ms = self.max_over_ranks(e0.elapsed_time(e1))
        kern_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
        return total_ms / steps, kern_ms, launches

    def roofline(self, workload, plan, T, kern_ms, traffic=None):
        deg, R, _, aggwt, kind, n_in, n_out, _ = WORKLOADS[workload]
        balg = plan.algorithmic_bytes(T, n_in, 4, n_out)
        achieved = balg / (kern_ms * 1e-3) / 1e9
        hbm = {"bound": "hbm", "achieved": achieved, "peak": self.peak, "unit": "GB/s",
               "frac": achieved / self.peak, "traffic": traffic,
               "traffic_ratio": (traffic / balg) if traffic else None, "peak_source": self.peak_src,
               "kernel": KERNEL[kind], "algorithmic_bytes_per_launch": balg,
               "bytes_per_region_day": balg / (plan.R * T), "launch_ms": kern_ms,
               "frac_of_8TBs_nominal": achieved / 8000.0}
        if kind != "edd":
            return hbm
        # Snyder: max(HBM time, fp64 time) bounds the kernel (SURVEY 7.3-5 / 8d); the fp64 side is larger
        clocks_hz = 1.965e9
        peak_ops = FP64_LANES_PER_SM_CLK * 148 * clocks_hz
        ops = SNYDER_FP64_OPS_PER_ENTRY_DAY * plan.info["nnz"] * T
        ach = ops / (kern_ms * 1e-3)
        return {"bound": "fp64", "achieved": ach / 1e12, "peak": peak_ops / 1e12, "unit": "Tinstr/s (fp64 pipe, lane-ops)",
                "frac": ach / peak_ops, "traffic": traffic, "kernel": KERNEL[kind], "launch_ms": kern_ms,
                "peak_source": "nominal: 64 fp64 lanes/SM/clk x 148 SMs x 1.965 GHz (no measured fp64 figure in MEASURED_PEAKS.json)",
                "fp64_ops_per_entry_day": SNYDER_FP64_OPS_PER_ENTRY_DAY, "entry_days": plan.info["nnz"] * T,
                "hbm": hbm}

    # ---- one workload, device-resident ------------------------------------------------
    def device_run(self, workload, steps, warmup, T=None, variant=None, groups_period=None):
        torch, E, N = self.torch, self.E, self.N
        deg, R, T0, aggwt, kind, n_in, n_out, desc = WORKLOADS[workload]
        T = T or T0
        lat, lon = self.syn.grid_labels(deg)
        df = self.table(deg, R)
        xs = self.inputs(workload, T, variant=variant)
        ncell = len(lat) * len(lon)
        t_plan = time.perf_counter()
        plan = E.get_plan(E.GridSpec(lat, lon), df, aggwt, "hierid", stage_bytes=4 * n_in, device=self.dev,
                          compact=(variant == "packed"))
        torch.cuda.synchronize()
        plan_ms = (time.perf_counter() - t_plan) * 1e3
        pack_ms = None
        if variant == "packed":
            # device-side compaction of the archive into packed planes [T][n_packed_cells] (only the
            # referenced 16-byte pieces, runs aligned to 64 bytes): paid once, reused by every later
            # aggregation of the same footprint (other weights, poly orders, ensemble members)
            import ctypes as C
            width = plan.info["n_packed_cells"]
            packed = torch.empty((T, width), dtype=torch.float32, device=self.dev)

            def pack():
                N.check(N.lib().ctb_pull_pack(plan._h, C.c_void_p(xs[0].data_ptr()), N.F32, ncell, None, 0, T,
                                              C.c_void_p(packed.data_ptr()), E._stream_ptr(self.dev)))
            _, pack_ms, _ = self.timed(pack, 5, 3)
            xs = [packed]
            ncell = width
        groups = None
        n_cols = T
        if groups_period:
            groups = E.get_time_groups(np.arange(T) // groups_period, self.dev)
            n_cols = groups.n_groups
        out = torch.empty((n_out, plan.R, n_cols), dtype=torch.float64, device=self.dev)
        ws = E._workspace(plan, T, n_out, N.LAYOUT_TIME_MAJOR, N.VARIANT_AUTO, groups, None)
        streaming = workload == "config5"
        years = YEARS_PER_STEP if streaming else 1
        params = PARAMS[kind]
        if streaming:
            pool = [xs[0]] + [self.inputs(workload, T, seed_off=100 * (k + 1))[0] for k in range(POOL - 1)]
            chk = torch.zeros((), dtype=torch.float64, device=self.dev)

        def step():
            if streaming:
                for y in range(YEARS_PER_STEP):
                    E.aggregate_device(plan, pool[y % POOL], None, N.LAYOUT_TIME_MAJOR, ncell, None, T, kind,
                                       params, n_out, out=out, workspace=ws)
                    chk.add_(out.sum())
                return
            E.aggregate_device(plan, xs[0], xs[1] if n_in == 2 else None, N.LAYOUT_TIME_MAJOR, ncell,
                               None, T, kind, params, n_out, out=out, workspace=ws, groups=groups)

        ms_step, kern_ms, launches = self.timed(step, steps, warmup)
        if streaming:
            kern_ms = ms_step / years
        res = {"plan": plan, "xs": xs, "out": out, "T": T, "ms_per_step": ms_step, "kern_ms": kern_ms, "pack_ms": pack_ms,
               "launches": launches, "years": years, "plan_ms": plan_ms,
               "value": self.world * plan.R * T * years / (ms_step * 1e-3),
               "checksum": float(torch.nansum(out).item())}
        return res

    def summary(self, workload, r, traffic=None, extra=None):
        """Compact entry of the `also` block."""
        info = r["plan"].info
        d = {"workload": WORKLOADS[workload][7], "T": r["T"], "ms_per_launch": r["kern_ms"],
             "region_days_per_s": r["value"], "roofline": self.roofline(workload, r["plan"], r["T"], r["kern_ms"], traffic),
             "bundles": info["n_bundles"], "gpu_launches": r["launches"], "checksum": r["checksum"]}
        d["roofline"].pop("peak_source", None)
        if extra:
            d.update(extra)
        return d


def run_ours(args):
    B = Bench(args)
    torch, dist, E, N = B.torch, B.dist, B.E, B.N
    from climate_toolbox_b200 import DataArray, Dataset
    from climate_toolbox_b200.aggregations.aggregations import weighted_aggregate_grid_to_regions
    from climate_toolbox_b200.transformations.transformations import snyder_edd
    rank, world, dev = B.rank, B.world, B.dev
    deg, R, T, aggwt, kind, n_in, n_out, desc = WORKLOADS[args.workload]
    if args.days:
        T = args.days
    lat, lon = B.syn.grid_labels(deg)
    df = B.table(deg, R)
    ncell = len(lat) * len(lon)
    traffic_all = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        traffic_all = json.load(open(tp))

    sampler = ClockSampler(B.local)
    sampler.start()
    head = B.device_run(args.workload, args.steps, args.warmup, T=T)
    clocks = sampler.result()
    plan, xs, out = head["plan"], head["xs"], head["out"]
    if args.dump_outputs and rank == 0:
        dump_outputs(out, kind, args.dump_outputs)
    info = plan.info
    roofline = B.roofline(args.workload, plan, T, head["kern_ms"], traffic_all.get(args.workload))
    streaming = args.workload == "config5"

    # ---- end to end through the public API with HOST buffers ----
    e2e = None
    if not args.no_e2e and not streaming:
        # every rank pins its own host copy of the batch: keep the node's total under 40 % of the
        # free host memory (8 ranks x 6 GB would not fit a small host) by shortening the e2e batch
        Te = T
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 32 << 30
        need = world * len(xs) * T * ncell * 4
        if need > 0.4 * avail:
            Te = max(64, int(T * 0.4 * avail / need) // 32 * 32)
        if world > 1:
            tmin = torch.tensor([Te], device=dev, dtype=torch.int64)
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
            Te = int(tmin.item())
        shape = (Te, len(lat), len(lon))
        host = [torch.empty(shape, dtype=torch.float32, pin_memory=True) for _ in xs]
        for h, x in zip(host, xs):
            h.copy_(x[:Te].view(shape))
        torch.cuda.synchronize()
        coords = {"time": np.arange(Te), "lat": lat, "lon": lon}
        dims = ("time", "lat", "lon")

        def make_ds(arrays):
            if kind == "identity":
                return Dataset({"tas": (dims, arrays[0])}, coords=coords), "tas"
            if kind == "poly":
                from climate_toolbox_b200._xr import Deferred, Variable
                src = Variable(dims, arrays[0])
                ds = Dataset(coords=coords)
                names = ["p1", "p2", "p3", "p4"]
                for p, nme in zip((1, 2, 3, 4), names):
                    ds._vars[nme] = Variable(dims, None, None, None, Deferred("poly", (273.15, float(p)), (src,)))
                return ds, names
            tn = DataArray(arrays[0], dims=dims, coords=coords, attrs={"units": "K"})
            tx = DataArray(arrays[1], dims=dims, coords=coords, attrs={"units": "K"})
            ds = Dataset(coords=coords)
            ds["edd10"] = snyder_edd(tn, tx, 283.15, check=False)
            ds["edd30"] = snyder_edd(tn, tx, 303.15, check=False)
            return ds, ["edd10", "edd30"]

        def measure(ds, names, steps, min_warm=3, warm_s=2.5, **opts):
            # warm-up: pinned staging/result blocks come from pools, and the host needs a moment after a
            # multi-GB pinned source was allocated and filled -- at least 3 calls and 2.5 s
            t_w, n_w = time.perf_counter(), 0
            while n_w < min_warm or (time.perf_counter() - t_w < warm_s and n_w < 30):
                r = weighted_aggregate_grid_to_regions(ds, names, aggwt, "hierid", weights=df, **opts)
                n_w += 1
            B.barrier()
            E.TRANSFER_BYTES.update(h2d=0, d2h=0)
            t0 = time.perf_counter()
            step_ms = []
            for _ in range(steps):
                ts = time.perf_counter()
                r = weighted_aggregate_grid_to_regions(ds, names, aggwt, "hierid", weights=df, **opts)
                step_ms.append(round((time.perf_counter() - ts) * 1e3, 1))      # returns host arrays: synchronous
            torch.cuda.synchronize()
            B.barrier()
            dt = B.max_over_ranks((time.perf_counter() - t0) / steps)
            first = names if isinstance(names, str) else names[0]
            return {"value": world * plan.R * Te / dt, "ms_per_step": dt * 1e3, "step_ms": step_ms,
                    "h2d_bytes_per_step": int(E.TRANSFER_BYTES["h2d"] // steps),
                    "d2h_bytes_per_step": int(E.TRANSFER_BYTES["d2h"] // steps), "warmup_calls": n_w,
                    "checksum": float(np.nansum(r[first].values))}

        e2e_steps = max(2, min(args.steps, 10))
        ds, names = make_ds([h.numpy() for h in host])
        m = measure(ds, names, e2e_steps)
        e2e = {"value": m["value"], "unit": "region-days/s", "h2d_bytes_per_step": m["h2d_bytes_per_step"],
               "d2h_bytes_per_step": m["d2h_bytes_per_step"],
               "host_input_bytes_per_step": int(sum(h.numel() * 4 for h in host)),
               "ms_per_step": m["ms_per_step"], "days_per_step": Te, "step_ms": m["step_ms"],
               "warmup_calls": m["warmup_calls"], "steps": e2e_steps,
               "pinned_result_blocks_allocated": int(sum(E._RESULT_OUT.values())),
               "api": "weighted_aggregate_grid_to_regions(ds[numpy over pinned host memory], ...) -> Dataset[numpy]: "
                      "GPU pull of the referenced gridcells from pinned host memory (ctb_pull_pack) in time chunks + fused kernel + chunked 2-D D2H into pinned memory",
               "checksum": m["checksum"],
               "rank0_cpu_affinity": (len(B.cpus) if B.cpus else None)}
        if kind == "identity":
            # the step after the path fused in (annual sums): the result block shrinks 365x
            my = measure(ds, names, max(2, e2e_steps // 2), min_warm=2, warm_s=0.5, time_groups=365)
            e2e["annual_sums"] = {k: my[k] for k in ("value", "ms_per_step", "step_ms", "h2d_bytes_per_step",
                                                     "d2h_bytes_per_step")}
        if world == 1 and kind == "identity" and not args.no_pageable:
            # a load_bcsd user holds PAGEABLE memory: same call on a plain numpy copy of a 365-day block
            Tp = min(Te, 365)
            pag = [np.array(h.numpy()[:Tp]) for h in host]
            coords_p = dict(coords, time=np.arange(Tp))
            dsp = Dataset({"tas": (dims, pag[0])}, coords=coords_p)
            keep_Te, Te = Te, Tp
            mp_ = measure(dsp, "tas", max(2, e2e_steps // 2), min_warm=2, warm_s=0.5)
            Te = keep_Te
            e2e["pageable_source"] = {"days_per_step": Tp, **{k: mp_[k] for k in ("value", "ms_per_step", "step_ms",
                                                                                  "h2d_bytes_per_step")}}
            del pag, dsp
        del host, ds

    # ---- strong scaling: ONE batch sharded along time, compute + final gather (north_star) ----
    strong = None
    if world > 1 and not streaming and kind == "identity":
        from climate_toolbox_b200.parallel import (PeerOutput, aggregate_shard_overlapped, aggregate_shard_p2p,
                                                   shard_sizes)
        x = xs[0]

        def run(gather, pieces):
            def f():
                aggregate_shard_overlapped(plan, x, None, ncell, T, kind, PARAMS[kind], n_out, pieces=pieces,
                                           gather=gather)
            return f

        s_steps = max(3, min(args.steps, 10))
        comp_ms, _, _ = B.timed(run(False, 1), s_steps, 3)
        seq_ms, _, _ = B.timed(run(True, 1), s_steps, 3)
        ovl_ms, _, _ = B.timed(run(True, 4), s_steps, 3)
        sizes = shard_sizes(T, world)
        # the gather fused into the kernel: the epilogue stores every region-day into all ranks' buffers
        # over NVLink peer memory (CUDA IPC) -- no collective, no staging copy
        p2p_ms = push_ms = p2p_err = same = same_push = None
        try:
            po = PeerOutput(plan, T, n_out)
            ref, _ = aggregate_shard_overlapped(plan, x, None, ncell, T, kind, PARAMS[kind], n_out, pieces=1)
            ref = torch.nan_to_num(ref)

            def p2p(mode, pieces=1):
                return lambda: aggregate_shard_p2p(plan, x, None, ncell, T, po, kind, PARAMS[kind], n_out, mode=mode,
                                                   pieces=pieces)
            p2p_ms, _, _ = B.timed(p2p("fused"), s_steps, 3)
            torch.cuda.synchronize()
            same = bool(torch.equal(torch.nan_to_num(po.gathered()), ref))
            # ... and as a push: the kernel writes its own buffer, one copy kernel sends the finished
            # column block to every peer as coalesced row pieces
            po.raw.zero_()
            torch.cuda.synchronize()
            dist.barrier()
            push_ms, _, _ = B.timed(p2p("push", 1), s_steps, 3)
            torch.cuda.synchronize()
            same_push = bool(torch.equal(torch.nan_to_num(po.gathered()), ref))
            del ref
            po.close()
        except Exception as ex:  # noqa: BLE001 -- IPC may be closed to the container: report, keep the NCCL numbers
            p2p_err = repr(ex)[:200]
        best = min(m for m in (seq_ms, ovl_ms, p2p_ms, push_ms) if m)
        strong = {"what": "one {}-day batch sharded along time over {} ranks (plan replicated); every rank ends with "
                          "the full [R][T] block".format(T, world),
                  "days_per_rank": sizes, "compute_ms": comp_ms,
                  "nccl_compute_plus_gather_ms": seq_ms, "nccl_overlapped_4_pieces_ms": ovl_ms,
                  "nccl_gather_ms": seq_ms - comp_ms,
                  "p2p_fused_kernel_ms": p2p_ms, "p2p_equal_to_nccl_result": same,
                  "p2p_push_ms": push_ms, "p2p_push_equal_to_nccl_result": same_push, "p2p_error": p2p_err,
                  "bytes_received_per_rank": int(8 * n_out * plan.R * (T - min(sizes))),
                  "value": plan.R * T / (best * 1e-3), "value_compute_only": plan.R * T / (comp_ms * 1e-3),
                  "unit": "region-days/s", "scaling": "strong",
                  "limiter": "NVLink: every rank receives (N-1)/N of the 285 MB fp64 output; the fused kernel hides "
                             "it behind the aggregation's own stores (best at N=2 and 4), the push kernel sends it as "
                             "coalesced row pieces after the aggregation (best at N=8), the NCCL path adds an "
                             "all_gather and a strided copy"}
        plan.__dict__.pop("_shard_buffers", None)

    # ---- the other configs and input variants (N = 1: device-timed, 10 steps each) ----
    also = None
    if world == 1 and not args.no_also and args.workload == "config2" and not args.days:
        also = {}
        del xs
        head["xs"] = None
        torch.cuda.empty_cache()
        st = max(5, min(args.steps, 10))
        for name, wl, kw in (("config2_packed_planes", "config2", {"variant": "packed"}),
                             ("config2_bcsd_like", "config2", {"variant": "bcsd_like"}),
                             ("config2_nan_2pct_of_land", "config2", {"variant": "nan2pct"}),
                             ("config2_annual_sums", "config2", {"groups_period": 365}),
                             ("config3", "config3", {}), ("config4", "config4", {}),
                             ("config1", "config1", {}), ("config5", "config5", {})):
            r = B.device_run(wl, st, 3, **kw)
            extra = None
            if wl == "config5":
                extra = {"model_years_per_step": r["years"], "pool_buffers": POOL,
                         "full_job_model_years": ENSEMBLE_YEARS,
                         "full_job_seconds_extrapolated": ENSEMBLE_YEARS / r["years"] * r["ms_per_step"] * 1e-3}
            if name == "config2_annual_sums":
                extra = {"note": "fused time reduction: output [R][4 years] instead of [R][1460 days]"}
            if name == "config2_packed_planes":
                extra = {"pack_ms_one_shot": r["pack_ms"], "one_shot_total_ms": r["pack_ms"] + r["kern_ms"],
                         "note": "archive compacted on the device (ctb_pull_pack on a device source) into packed planes; "
                                 "ms_per_launch is the amortised cost of every aggregation after the first"}
            also[name] = B.summary(wl, r, traffic_all.get(name), extra)
            del r
            torch.cuda.empty_cache()

    # ---- ensemble (config 5) at N ranks: model-years dealt round-robin, outputs stay with their owner ----
    ensemble = None
    if streaming:
        ensemble = {"model_years_per_step_per_rank": head["years"], "pool_buffers": POOL,
                    "full_job_model_years": ENSEMBLE_YEARS, "ranks": world,
                    "full_job_seconds_extrapolated": ENSEMBLE_YEARS / (head["years"] * world) * head["ms_per_step"] * 1e-3,
                    "note": "outputs are summed into a checksum and discarded; e2e is not measured for this "
                            "workload (6 TB of input do not exist on the host)"}

    # ---- CPU baseline: the oracle on a bounded sample, rank 0, N = 1 only ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and kind == "identity":
        days = 365
        ref = CpuReference(args.workload, days, 1)
        sec = ref.one_pass()
        cpu = {"value": plan.R * days / sec, "unit": "region-days/s", "cores": 1, "kind": "port",
               "sample": "{} days of the workload, single process (the reference is single-threaded "
                         "eager numpy), {:.1f} s; host has {} cores".format(days, sec, os.cpu_count())}

    if rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": "region-days/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": config_dict(args.workload, T, world),
            "plan": {"U": info["n_cells_distinct"], "nnz": info["nnz"], "bundles": info["n_bundles"],
                     "staged_pieces": info["n_pieces"], "distinct_pieces": info["n_pieces_distinct"],
                     "quads": info["n_quads"], "quads_with_bank_conflict": info["n_quads_conflict"],
                     "plan_build_ms": head["plan_ms"]},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(head["launches"]),
            "clocks": clocks, "checksum": head["checksum"],
        }
        for k, v in (("strong", strong), ("also", also), ("ensemble", ensemble)):
            if v is not None:
                line[k] = v
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--days", type=int, default=0, help="override T (debug)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the device-timed lines of the other configs")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs as DIR/<output>.npy (float64, at most 64 MB in all: "
                         "a fixed, seeded sample of regions when the block is larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    sys.dont_write_bytecode = True          # nothing lands in the tree, which may be read-only
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
