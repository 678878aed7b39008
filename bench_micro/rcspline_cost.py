"""What does a restricted-cubic-spline launch cost next to the identity and the 4-output polynomial launch, and
does fusing four spline terms into one pass beat two passes of two?

Config 2 shapes (0.25 degree, 1460 days f32 TIME_MAJOR -> 24,378 regions, popwt, device-resident, the synthetic
field of bench.py), leap days removed through a time index as behind tas_poly: the field holds 1461 day planes
(a leap year's Feb 29 included) and the launches read 1460 of them.  The launches alternate in one process, each
timed with CUDA events around one launch; the median of ROUNDS launches per kind is reported.  The spline
launches use 5 knots (4 terms): all four in one launch (first = 0, output 0 the linear term), and the same four
as two launches of two (first = 0 and first = 2).  Then one public call: tas_rcspline with 7 knots (6 terms,
launches of 4 + 2) over 365 days, time_groups="year", device-resident (host clock around the call, which ends
with the result on the host).

    python bench_micro/rcspline_cost.py [--rounds 30] [--libraries build/libctb_rcs384.so ...]
--libraries: builds of the library compiled with another -DCTB_RCS34_THREADS (the CTA size of the 3- and 4-term
spline kernels); each is timed on the 4-term launch in a child process, alternating with the default build."""
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
from climate_toolbox_b200.transformations.transformations import tas_rcspline  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=30)
ap.add_argument("--public-calls", type=int, default=10)
ap.add_argument("--libraries", nargs="*", default=[])
ap.add_argument("--only-rcs4", action="store_true", help=argparse.SUPPRESS)   # child runs of --libraries
args = ap.parse_args()

if not args.only_rcs4:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True)
    print("gpu (name, power limit):", smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "nvidia-smi failed")
print("library:", os.environ.get("CTB_LIBRARY", "libctb.so"))

T = 1460
KNOTS5 = (-5.0, 5.0, 12.0, 20.0, 28.0)
lat, lon = synthetic.grid_labels(0.25)
df = synthetic.weights_table(0.25, 24378)
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(7)
tas = 288.0 + 10.0 * torch.randn((T + 1, len(lat) * len(lon)), generator=g, device=dev, dtype=torch.float32)
tix = np.delete(np.arange(T + 1), 365 + 59)          # day planes of 2001..2004, without 2004-02-29
plan = E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", device=dev)
R = plan.R
KINDS = {   # name: [(kind, params, n_out), ...] launched back to back
    "identity": [("identity", (), 1)],
    "poly 1-4": [("poly", (273.15, 1, 2, 3, 4), 4)],
    "rcs x4": [("rcspline", (273.15, 0.0) + KNOTS5, 4)],
    "rcs 2+2": [("rcspline", (273.15, 0.0) + KNOTS5, 2), ("rcspline", (273.15, 2.0) + KNOTS5, 2)],
}
if args.only_rcs4:
    KINDS = {k: KINDS[k] for k in ("identity", "rcs x4")}
outs = {k: torch.empty((4, R, T), dtype=torch.float64, device=dev) for k in KINDS}


def launch(name):
    j = 0
    for kind, params, n_out in KINDS[name]:
        E.aggregate_device(plan, tas, None, N.LAYOUT_TIME_MAJOR, tas.shape[1], tix, T, kind, params, n_out,
                           out=outs[name][j:j + n_out])
        j += n_out


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
print("config 2 shapes, time index: T={} days, R={} regions, nnz={}, U={} gridcells; median of {} alternating "
      "rounds each".format(T, R, plan.info["nnz"], plan.info["n_cells_distinct"], args.rounds))
for name, launches in KINDS.items():
    m = float(np.median(ms[name]))
    n_out = sum(n for _, _, n in launches)
    alg = sum(plan.algorithmic_bytes(T, 1, 4, n) for _, _, n in launches)
    print("  {:9s} {} launch(es), {} outputs: {:.3f} ms (min {:.3f}, max {:.3f})  {:.2e} region-days/s  "
          "{:,.0f} algorithmic GB/s".format(name, len(launches), n_out, m, min(ms[name]), max(ms[name]),
                                            R * T / (m * 1e-3), alg / (m * 1e-3) / 1e9))
if "rcs 2+2" in outs:
    d = float((outs["rcs x4"] - outs["rcs 2+2"]).abs().max())
    print("  check: fused and split spline launches differ by at most {:.3g}".format(d))
print("  check: term means over region-days", [float(torch.nanmean(outs["rcs x4"][j])) for j in range(4)])
del outs
if args.only_rcs4:
    sys.exit(0)

# ---- other CTA sizes of the 3- and 4-term spline kernels: child processes, alternating with the default --------
for lib in args.libraries:
    for env_lib in (None, lib):
        env = dict(os.environ)
        if env_lib:
            env["CTB_LIBRARY"] = os.path.abspath(env_lib)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--only-rcs4", "--rounds", str(args.rounds)],
                           env=env, capture_output=True, text=True)
        print("  [child]", (r.stdout + r.stderr).strip().replace("\n", "\n  [child] "))

# ---- public call: a 7-knot basis over one year, annual sums -----------------------------------------------
T1 = 365
tas1 = tas[:T1].view(T1, len(lat), len(lon))
ds = Dataset({"tas": (("time", "lat", "lon"), tas1)},
             coords={"time": pd.date_range("2001-01-01", periods=T1), "lat": lat, "lon": lon})
ds1 = tas_rcspline(ds, (-10.0, 0.0, 5.0, 10.0, 15.0, 20.0, 30.0), "s")
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
m = float(np.median(wall))
print("public tas_rcspline, 7 knots (6 terms) x 365 days, time_groups='year', device-resident: {:.2f} ms per call "
      "(median of {}, min {:.2f}), {} kernel launches per call, {:.2e} region-days/s".format(
          m, args.public_calls, min(wall), launches, R * T1 / (m * 1e-3)))
print("  check: yearly sum of the linear term, median over regions {:.1f} C-days".format(
    float(np.nanmedian(out["s_0"].values))))
