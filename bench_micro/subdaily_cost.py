"""What does the daily reduction of sub-daily data cost when it is fused into the packing (ctb_pull_pack_daily),
next to what a user does today (a full-grid daily reduction on the device, then the public aggregation)?

Device-resident case: config 2 shapes (0.25 degree, 24,378 regions, popwt), hourly f32 (S = 24) over DAYS days
(60 days = 6.0 GB, far beyond the 126 MB of L2).  Each reduce-pack call is timed with CUDA events; the median
of ROUNDS calls is reported, for the mean (float64 planes, plan of 8-byte elements) and for min + max from one
read (f32 planes), then the aggregation of the packed planes (identity of the mean; Snyder EDD of min / max).
The bytes the kernel must read are the referenced 16-byte pieces x S steps per day; their rate is set against
the 6,537 GB/s copy peak of DESIGN.md section 5.  Then two public calls, alternated in one process (host clock
around a call that ends with the result on the host): resample_daily(ds, "mean") aggregated, against the daily
mean computed on the whole grid by torch followed by the public aggregation of that daily array.

Pinned-host case: the same grid, PINNED_DAYS days in pinned host memory; the reduce-pack of the mean reads the
referenced pieces over PCIe, and its rate is set against the 47.6 GB/s of ctb_pull_pack (DESIGN.md section 5).

    python bench_micro/subdaily_cost.py [--days 60] [--pinned-days 8] [--rounds 20]"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import torch  # noqa: E402

from climate_toolbox_b200 import Dataset, synthetic  # noqa: E402
from climate_toolbox_b200 import _engine as E, _native as N  # noqa: E402
from climate_toolbox_b200.aggregations.aggregations import weighted_aggregate_grid_to_regions  # noqa: E402
from climate_toolbox_b200.utils.utils import resample_daily  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--days", type=int, default=60)
ap.add_argument("--pinned-days", type=int, default=8)
ap.add_argument("--rounds", type=int, default=20)
ap.add_argument("--public-calls", type=int, default=6)
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True)
print("gpu (name, power limit):", smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "nvidia-smi failed")

S, D = 24, args.days
lat, lon = synthetic.grid_labels(0.25)
ncell = len(lat) * len(lon)
df = synthetic.weights_table(0.25, 24378)
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(7)
x = 288.0 + 10.0 * torch.randn((D * S, ncell), generator=g, device=dev, dtype=torch.float32)
grid = E.GridSpec(lat, lon)
p8 = E.get_plan(grid, df, "popwt", "hierid", stage_bytes=8, compact=True, elem_bytes=8, device=dev)
p4 = E.get_plan(grid, df, "popwt", "hierid", stage_bytes=8, compact=True, elem_bytes=4, device=dev)
width = p8.info["n_packed_cells"]
pieces = p8.info["n_pieces_distinct"]
print("input: {} days x {} steps x {} cells f32 = {:.2f} GB; referenced pieces {} of {}; packed cells {}".format(
    D, S, ncell, D * S * ncell * 4 / 1e9, pieces, ncell // 4, width))
mean = torch.empty((D, width), dtype=torch.float64, device=dev)
mn = torch.empty((D, width), dtype=torch.float32, device=dev)
mx = torch.empty((D, width), dtype=torch.float32, device=dev)
L = N.lib()


def pull(plan, src, days, ops, dm=None, dn=None, dx=None):
    N.check(L.ctb_pull_pack_daily(plan._h, C.c_void_p(src), N.F32, ncell, S, None, 0, days, ops,
                                  C.c_void_p(dm.data_ptr()) if dm is not None else None,
                                  C.c_void_p(dn.data_ptr()) if dn is not None else None,
                                  C.c_void_p(dx.data_ptr()) if dx is not None else None,
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)))


def timed(fn, rounds):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


need = D * S * pieces * 16
kernels = {
    "reduce-pack mean": lambda: pull(p8, x.data_ptr(), D, N.DAILY_MEAN, dm=mean),
    "reduce-pack min+max": lambda: pull(p4, x.data_ptr(), D, N.DAILY_MIN | N.DAILY_MAX, dn=mn, dx=mx),
    "aggregate mean planes (identity)": lambda: E.aggregate_device(p8, mean, None, N.LAYOUT_TIME_MAJOR, width, None, D),
    "aggregate min/max planes (Snyder EDD 290)": lambda: E.aggregate_device(
        p4, mn, mx, N.LAYOUT_TIME_MAJOR, width, None, D, "edd", (290.0,), 1),
}
for name, fn in kernels.items():
    med, lo, hi = timed(fn, args.rounds)
    line = "{:44s} {:8.3f} ms  (min {:.3f}, max {:.3f})".format(name, med, lo, hi)
    if name.startswith("reduce-pack"):
        line += "  {:.2f} GB read, {:,.0f} GB/s = {:.2f} of the 6,537 GB/s copy peak".format(
            need / 1e9, need / med / 1e6, need / med / 1e6 / 6537)
    print(line)

# public calls, alternated
times = pd.date_range("2001-01-01", periods=D * S, freq="h").values
ds = Dataset({"tas": (("time", "lat", "lon"), x.view(D * S, len(lat), len(lon)))},
             coords={"time": times, "lat": lat, "lon": lon})
days = pd.date_range("2001-01-01", periods=D, freq="D").values


def fused():
    return weighted_aggregate_grid_to_regions(resample_daily(ds, "mean"), "tas", "popwt", "hierid", weights=df)


def today():
    daily = torch.nanmean(x.view(D, S, ncell), dim=1).view(D, len(lat), len(lon))
    d1 = Dataset({"tas": (("time", "lat", "lon"), daily)}, coords={"time": days, "lat": lat, "lon": lon})
    return weighted_aggregate_grid_to_regions(d1, "tas", "popwt", "hierid", weights=df)


res = {"fused": [], "full-grid reduction + aggregation": []}
for fn in (fused, today):
    fn()
torch.cuda.synchronize()
for _ in range(args.public_calls):
    for key, fn in (("fused", fused), ("full-grid reduction + aggregation", today)):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        res[key].append((time.perf_counter() - t0) * 1e3)
for key, v in res.items():
    print("public call, {:36s} median {:8.2f} ms  (min {:.2f}, max {:.2f})".format(key, np.median(v), min(v), max(v)))
a, b = fused()["tas"].values, today()["tas"].values
print("fused vs full-grid float32 nanmean path: max |diff| {:.3e} K (the full-grid path sums in float32)".format(
    np.nanmax(np.abs(a - b))))
del x, ds, mean, mn, mx
torch.cuda.empty_cache()

# pinned host source
PD = args.pinned_days
host = torch.empty((PD * S, ncell), dtype=torch.float32, pin_memory=True)
host.normal_(288.0, 10.0)
out = torch.empty((PD, width), dtype=torch.float64, device=dev)
med, lo, hi = timed(lambda: pull(p8, host.data_ptr(), PD, N.DAILY_MEAN, dm=out), max(5, args.rounds // 2))
bus = PD * S * pieces * 16
print("pinned host, {} days ({:.2f} GB pinned): reduce-pack mean {:.3f} ms (min {:.3f}, max {:.3f}), {:.2f} GB of "
      "referenced pieces = {:.1f} GB/s against the 47.6 GB/s of ctb_pull_pack".format(
          PD, host.numel() * 4 / 1e9, med, lo, hi, bus / 1e9, bus / med / 1e6))
