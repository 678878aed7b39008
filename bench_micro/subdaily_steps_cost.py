"""What do per-step transforms of sub-daily data cost when they are computed while the referenced gridcells are
packed (ctb_pull_pack_daily_steps), next to the daily mean of the same read and to the route a user has without
them (a per-step transform on the full grid, then resample_daily(..., "mean"), then the aggregation)?

Config 2 shapes (0.25 degree, 24,378 regions, popwt), hourly f32 (S = 24) over DAYS days on the device (60 days =
6.0 GB, far beyond the 126 MB of L2).  Each reduce-pack call is timed with CUDA events; the median of ROUNDS calls
is reported for the daily mean, EDD with 1, 2 and 4 thresholds, GDD with 4 pairs and 4 bins, then the identity
aggregation of one packed float64 plane (a fused request adds one per output).  For each case the bytes the
kernel must read (referenced 16-byte pieces x S steps per day) are set against the 6,537 GB/s copy peak of
DESIGN.md section 5, and the float64 adds and subtractions it must issue (2 per referenced cell-step and output
for EDD and GDD; bins count in integers) against the nominal float64 issue rate: 64 lanes per SM x 148 SMs x the
maximum SM clock nvidia-smi reports (an assumption about the card, not a measurement).
Then two public routes for 4 EDD thresholds with annual sums (time_groups="year"), alternated in one process
(host clock around a call that ends with the result on the host): subdaily_edd x 4 aggregated together, and the
manual route, one threshold at a time so that its float64 full-grid array fits: torch computes
max(x - e, 0) in float64 over the whole grid, resample_daily(..., "mean") reduces it, the public call aggregates it.

    python bench_micro/subdaily_steps_cost.py [--days 60] [--rounds 20] [--public-calls 4]"""
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
from climate_toolbox_b200.transformations.transformations import subdaily_edd  # noqa: E402
from climate_toolbox_b200.utils.utils import resample_daily  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--days", type=int, default=60)
ap.add_argument("--rounds", type=int, default=20)
ap.add_argument("--public-calls", type=int, default=4)
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True)
card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "nvidia-smi failed"
print("gpu (name, power limit, max SM clock):", card)
try:
    sm_mhz = float(card.split(",")[2].split()[0])
except (IndexError, ValueError):
    sm_mhz = float("nan")
fp64_rate = 64 * 148 * sm_mhz * 1e6          # nominal float64 adds per second

S, D = 24, args.days
lat, lon = synthetic.grid_labels(0.25)
ncell = len(lat) * len(lon)
df = synthetic.weights_table(0.25, 24378)
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(7)
x = 288.0 + 10.0 * torch.randn((D * S, ncell), generator=g, device=dev, dtype=torch.float32)
p8 = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", stage_bytes=8, compact=True, elem_bytes=8, device=dev)
width = p8.info["n_packed_cells"]
pieces = p8.info["n_pieces_distinct"]
print("input: {} days x {} steps x {} cells f32 = {:.2f} GB; referenced pieces {} of {}; packed cells {}".format(
    D, S, ncell, D * S * ncell * 4 / 1e9, pieces, ncell // 4, width))
planes = [torch.empty((D, width), dtype=torch.float64, device=dev) for _ in range(4)]
L = N.lib()
stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731


def mean():
    N.check(L.ctb_pull_pack_daily(p8._h, C.c_void_p(x.data_ptr()), N.F32, ncell, S, None, 0, D, N.DAILY_MEAN,
                                  C.c_void_p(planes[0].data_ptr()), None, None, stream()))


def steps(op, params, n_out):
    prm = (C.c_double * len(params))(*params)
    dst = (C.c_void_p * n_out)(*[p.data_ptr() for p in planes[:n_out]])
    return lambda: N.check(L.ctb_pull_pack_daily_steps(p8._h, C.c_void_p(x.data_ptr()), N.F32, ncell, S, None, 0, D,
                                                       op, prm, len(params), n_out, dst, stream()))


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
cell_steps = D * S * pieces * 4
cases = [("reduce-pack mean", mean, 0),
         ("reduce-pack EDD x1", steps(N.STEP_EDD, [290.0], 1), 2),
         ("reduce-pack EDD x2", steps(N.STEP_EDD, [290.0, 300.0], 2), 4),
         ("reduce-pack EDD x4", steps(N.STEP_EDD, [283.15, 290.0, 295.5, 300.0], 4), 8),
         ("reduce-pack GDD x4", steps(N.STEP_GDD, [283.15, 303.15, 280.0, 290.0, 290.0, 300.0, 300.0, 310.0], 4), 8),
         ("reduce-pack bins x4", steps(N.STEP_BINS, [-np.inf, 280.0, 290.0, 300.0, np.inf], 4), 0),
         ("aggregate one plane (identity)", lambda: E.aggregate_device(p8, planes[0], None, N.LAYOUT_TIME_MAJOR, width,
                                                                       None, D), -1)]
base = None
for name, fn, ops in cases:
    med, lo, hi = timed(fn, args.rounds)
    line = "{:32s} {:8.3f} ms  (min {:.3f}, max {:.3f})".format(name, med, lo, hi)
    if ops >= 0:
        base = base or med
        bw = need / med / 1e6
        line += "  {:.2f} GB read, {:,.0f} GB/s = {:.2f} of the copy peak".format(need / 1e9, bw, bw / 6537)
        if ops:
            line += "; {:.2e} fp64 adds/s = {:.2f} of nominal".format(cell_steps * ops / med * 1e3,
                                                                        cell_steps * ops / med * 1e3 / fp64_rate)
        line += "; x{:.2f} the mean".format(med / base)
    print(line)

# public routes, 4 EDD thresholds, annual sums
THR = (283.15, 290.0, 295.5, 300.0)
times = pd.date_range("2001-01-01", periods=D * S, freq="h").values
grid3 = x.view(D * S, len(lat), len(lon))
tas = Dataset({"tas": (("time", "lat", "lon"), grid3)}, coords={"time": times, "lat": lat, "lon": lon}).tas
tas.attrs["units"] = "K"
names = ["e{}".format(k) for k in range(4)]


def fused():
    das = [subdaily_edd(tas, e) for e in THR]
    d = Dataset(dict(zip(names, das)), coords=das[0]._coords)
    return weighted_aggregate_grid_to_regions(d, names, "popwt", "hierid", weights=df, time_groups="year")


def manual():
    out = {}
    for n, e in zip(names, THR):
        f = torch.clamp(grid3.double() - e, min=0.0)
        hourly = Dataset({n: (("time", "lat", "lon"), f)}, coords={"time": times, "lat": lat, "lon": lon})
        r = weighted_aggregate_grid_to_regions(resample_daily(hourly, "mean"), n, "popwt", "hierid", weights=df,
                                               time_groups="year")
        out[n] = r[n].values
        del f, hourly
    return out


res = {"subdaily_edd x4 fused": [], "manual: torch full grid + resample_daily": []}
a, b = fused(), manual()
print("fused vs manual: max |diff| {:.3e} degree days (annual sums; the torch subtraction rounds like the "
      "kernel's, the sums differ in order)".format(max(np.nanmax(np.abs(a[n].values - b[n])) for n in names)))
torch.cuda.synchronize()
for _ in range(args.public_calls):
    for key, fn in zip(res, (fused, manual)):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        res[key].append((time.perf_counter() - t0) * 1e3)
for key, v in res.items():
    print("public call, time_groups='year', {:42s} median {:8.2f} ms  (min {:.2f}, max {:.2f})".format(
        key, np.median(v), min(v), max(v)))
print("peak memory allocated through torch: {:.1f} GB".format(torch.cuda.max_memory_allocated() / 1e9))
