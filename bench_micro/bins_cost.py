"""What does a temperature-bins launch cost next to the identity and the 4-output polynomial launch?

Config 2 shapes (0.25 degree, 1460 days f32 -> 24,378 regions, popwt, device-resident, the synthetic field of
bench.py).  The three launches alternate in one process, each timed with CUDA events around one launch; the
median of ROUNDS launches per kind is reported.  Then one public call: tas_bins with 12 bins over 365 days,
time_groups="year", device-resident (host clock around the call, which ends with the result on the host).

    python bench_micro/bins_cost.py [--rounds 30]
CTB_LIBRARY selects another build of the library (e.g. one compiled with -DCTB_BINS34_THREADS=512)."""
import argparse
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
from climate_toolbox_b200.transformations.transformations import tas_bins  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=30)
ap.add_argument("--public-calls", type=int, default=10)
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True)
print("gpu (name, power limit):", smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "nvidia-smi failed")
print("library:", os.environ.get("CTB_LIBRARY", "libctb.so"))

T = 1460
lat, lon = synthetic.grid_labels(0.25)
df = synthetic.weights_table(0.25, 24378)
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(7)
tas = 288.0 + 10.0 * torch.randn((T, len(lat) * len(lon)), generator=g, device=dev, dtype=torch.float32)
plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", device=dev)
R = plan.R
KINDS = {   # name: (kind, params, n_out)
    "identity": ("identity", (), 1),
    "poly 1-4": ("poly", (273.15, 1, 2, 3, 4), 4),
    "bins x4": ("bins", (273.15, 5.0, 10.0, 15.0, 20.0, 25.0), 4),
}
outs = {k: torch.empty((n, R, T), dtype=torch.float64, device=dev) for k, (_, _, n) in KINDS.items()}


def launch(name):
    kind, params, n_out = KINDS[name]
    E.aggregate_device(plan, tas, None, N.LAYOUT_TIME_MAJOR, tas.shape[1], None, T, kind, params, n_out,
                       out=outs[name])


for _ in range(5):
    for name in KINDS:
        launch(name)
torch.cuda.synchronize()
ms = {name: [] for name in KINDS}
for _ in range(args.rounds):
    for name in KINDS:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        launch(name)
        b.record()
        b.synchronize()
        ms[name].append(a.elapsed_time(b))
print("config 2 shapes: T={} days, R={} regions, nnz={}, U={} gridcells; median of {} alternating launches each"
      .format(T, R, plan.info["nnz"], plan.info["n_cells_distinct"], args.rounds))
for name, (kind, params, n_out) in KINDS.items():
    m = float(np.median(ms[name]))
    alg = plan.algorithmic_bytes(T, 1, 4, n_out)
    print("  {:9s} n_out={}: {:.3f} ms (min {:.3f}, max {:.3f})  {:.2e} region-days/s  {:,.0f} algorithmic GB/s"
          .format(name, n_out, m, min(ms[name]), max(ms[name]), R * T / (m * 1e-3), alg / (m * 1e-3) / 1e9))
b = outs["bins x4"]
frac = float(torch.nanmean(b.sum(0)))
ref = float(torch.nanmean(((tas - 273.15 >= 5.0) & (tas - 273.15 < 25.0)).double()))
print("  check: mean over region-days of the 4 bins' sum {:.4f} (share of gridcell-days in [5, 25) C: {:.4f})"
      .format(frac, ref))
del outs, b

# ---- public call: 12 bins over one year, annual sums -----------------------------------------------
T1 = 365
tas1 = tas[:T1].view(T1, len(lat), len(lon))
ds = Dataset({"tas": (("time", "lat", "lon"), tas1)},
             coords={"time": pd.date_range("2001-01-01", periods=T1), "lat": lat, "lon": lon})
edges = [-np.inf, -10.0, -5.0, 0.0, 5.0, 10.0, 15.0, 20.0, 25.0, 30.0, 35.0, 40.0, np.inf]
ds1 = tas_bins(ds, edges, "b")
names = list(ds1.data_vars)
for _ in range(3):
    out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df, time_groups="year")
torch.cuda.synchronize()
n0 = E.launch_count()
wall = []
for _ in range(args.public_calls):
    t0 = time.perf_counter()
    out = weighted_aggregate_grid_to_regions(ds1, names, "popwt", "hierid", weights=df, time_groups="year")
    torch.cuda.synchronize()
    wall.append((time.perf_counter() - t0) * 1e3)
launches = (E.launch_count() - n0) // args.public_calls
days = sum(out[n].values for n in names)
m = float(np.median(wall))
print("public tas_bins, 12 bins x 365 days, time_groups='year', device-resident: {:.2f} ms per call (median of {}, "
      "min {:.2f}), {} kernel launches per call, {:.2e} region-days/s".format(
          m, args.public_calls, min(wall), launches, R * T1 / (m * 1e-3)))
print("  check: days per year over the 12 bins, median over regions {:.2f} (NaN-free data: 365)".format(
    float(np.nanmedian(days))))
