"""What does a CF-packed int16 source (io.decode_packed) cost against float32 and float64 sources that hold the same
decoded values?

1. Config 2 shapes (0.25 degree, 24,378 regions, popwt), 1460 daily planes in pinned host memory.  The int16 source is
   packed with float32 attributes, so the decoded type is float32 and the float32 source holds exactly the decoded
   values (the float64 source holds them widened).  Reported: the public call (weighted_aggregate_grid_to_regions,
   host clock around a call that ends with the result on the host; the three sources alternate in one process), the
   bytes it moved across PCIe (_engine.TRANSFER_BYTES), the pack kernel alone over all days (CUDA events; the
   decode-pack for int16, ctb_pull_pack for the floats) from pinned memory and from device memory, and the 64-byte
   units of a source plane that the referenced pieces touch per day, counted on the CPU from plan.row_cells().
2. Hourly (S = 24), config 2 shapes, 60 days, device-resident: the reduce-pack of the daily mean and of EDD x 4, int16
   against float32 holding the same decoded values, alternated; compare with 0.434 / 0.857 ms of
   profiles/micro/r3_subdaily_steps_cost.log.

    python bench_micro/packed_cost.py [--days 1460] [--hourly-days 60] [--rounds 20] [--public-calls 5]"""
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
from climate_toolbox_b200.io import decode_packed  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--days", type=int, default=1460)
ap.add_argument("--hourly-days", type=int, default=60)
ap.add_argument("--rounds", type=int, default=20)
ap.add_argument("--public-calls", type=int, default=5)
args = ap.parse_args()

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True)
print("gpu (name, power limit, max SM clock):", smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else
      "nvidia-smi failed")

lat, lon = synthetic.grid_labels(0.25)
nlat, nlon = len(lat), len(lon)
ncell = nlat * nlon
df = synthetic.weights_table(0.25, 24378)
dev = torch.device("cuda", 0)
L = N.lib()
stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
SCALE, OFFSET = np.float32(0.0016), np.float32(265.0)
DEC32 = N.Decode(float(SCALE), float(OFFSET), N.F32, 1, (C.c_int16 * 4)(-32767))


def raw_int16(T, seed):
    """[T, ncell] int16 on the device: a smooth field plus noise, 0.1 % fill values."""
    g = torch.Generator(device=dev).manual_seed(seed)
    r = torch.randn((T, ncell), generator=g, device=dev) * 8000.0
    r = r.clamp(-32766, 32767).round().to(torch.int16)
    r[torch.rand((T, ncell), generator=g, device=dev) < 1e-3] = -32767
    return r


def decoded(r, dtype):
    y = r.to(torch.float32) * torch.tensor(SCALE, device=dev) + torch.tensor(OFFSET, device=dev)
    y[r == -32767] = float("nan")
    return y.to(dtype)


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


def pinned_copy(t):
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t)
    return h


# ---------------------------------------------------------------------------------------------------------------
# 1. daily, pinned host, 1460 days
# ---------------------------------------------------------------------------------------------------------------
T = args.days
r_dev = raw_int16(T, 7)
srcs = {"int16": r_dev, "float32": decoded(r_dev, torch.float32), "float64": decoded(r_dev, torch.float64)}
host = {k: pinned_copy(v) for k, v in srcs.items()}
torch.cuda.synchronize()
print("1. daily: {} days x {} cells; source bytes: {}".format(
    T, ncell, ", ".join("{} {:.2f} GB".format(k, v.numel() * v.element_size() / 1e9) for k, v in host.items())))

cells = np.unique(E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", device=dev).row_cells())
pieces = np.unique(cells // 4)
for k, es in (("int16", 2), ("float32", 4), ("float64", 8)):
    units = np.unique(pieces * 4 * es // 64).size
    print("   {:8s} referenced pieces {:,}: {:.2f} GB over {} days; 64-byte units touched per day {:,} of {:,} "
          "({:.2f} GB over {} days)".format(k, pieces.size, pieces.size * 4 * es * T / 1e9, T, units,
                                             ncell * es // 64, units * 64 * T / 1e9, T))

times = pd.date_range("2001-01-01", periods=T, freq="D").values
ds = {}
for k, h in host.items():
    arr = h.numpy().reshape(T, nlat, nlon)
    if k == "int16":
        d = Dataset({"tas": (("time", "lat", "lon"), arr, {"scale_factor": SCALE, "add_offset": OFFSET,
                                                             "_FillValue": np.int16(-32767)})},
                    coords={"time": times, "lat": lat, "lon": lon})
        ds[k] = decode_packed(d)
    else:
        ds[k] = Dataset({"tas": (("time", "lat", "lon"), arr)}, coords={"time": times, "lat": lat, "lon": lon})


def public(k):
    return weighted_aggregate_grid_to_regions(ds[k], "tas", "popwt", "hierid", weights=df)["tas"].values


ref = public("float32")
for k in ("int16", "float64"):
    got = public(k)
    same = np.array_equal(got.view(np.int64), ref.view(np.int64))
    print("   public call {} vs float32: bit identical {}".format(k, same))
res = {k: [] for k in ds}
moved = {}
torch.cuda.synchronize()
for _ in range(args.public_calls):
    for k in ds:
        b0 = E.TRANSFER_BYTES["h2d"]
        t0 = time.perf_counter()
        public(k)
        torch.cuda.synchronize()
        res[k].append((time.perf_counter() - t0) * 1e3)
        moved[k] = E.TRANSFER_BYTES["h2d"] - b0
for k, v in res.items():
    print("   public call, pinned {:8s} median {:8.2f} ms (min {:.2f}, max {:.2f}); h2d {:.3f} GB = {:.1f} GB/s at the "
          "median".format(k, np.median(v), min(v), max(v), moved[k] / 1e9, moved[k] / np.median(v) / 1e6))

p = {es: E.get_plan(E.GridSpec(lat, lon), df, "popwt", "hierid", stage_bytes=es, compact=True, elem_bytes=es,
                    device=dev) for es in (4, 8)}
width = p[4].info["n_packed_cells"]
dst = torch.empty((T, width), dtype=torch.float64, device=dev)


def pack(k, where):
    x = host[k] if where == "pinned" else srcs[k]
    if k == "int16":
        return lambda: N.check(L.ctb_pull_pack_decode(p[4]._h, C.c_void_p(x.data_ptr()), ncell, C.byref(DEC32), None,
                                                      0, T, C.c_void_p(dst.data_ptr()), stream()))
    es = 4 if k == "float32" else 8
    return lambda: N.check(L.ctb_pull_pack(p[es]._h, C.c_void_p(x.data_ptr()), N.F32 if es == 4 else N.F64, ncell,
                                           None, 0, T, C.c_void_p(dst.data_ptr()), stream()))


for where, rounds in (("pinned", max(3, args.rounds // 4)), ("device", args.rounds)):
    for k in srcs:
        med, lo, hi = timed(pack(k, where), rounds)
        nbytes = pieces.size * 4 * {"int16": 2, "float32": 4, "float64": 8}[k] * T
        print("   pack kernel, {:6s} {:8s} {:8.3f} ms (min {:.3f}, max {:.3f}); referenced {:.2f} GB = {:,.0f} GB/s"
              .format(where, k, med, lo, hi, nbytes / 1e9, nbytes / med / 1e6))
del srcs, host, ds, dst, r_dev
torch.cuda.empty_cache()

# ---------------------------------------------------------------------------------------------------------------
# 2. hourly, device-resident, 60 days
# ---------------------------------------------------------------------------------------------------------------
S, D = 24, args.hourly_days
r = raw_int16(D * S, 11)
x32 = decoded(r, torch.float32)
p8 = p[8]
width = p8.info["n_packed_cells"]
planes = [torch.empty((D, width), dtype=torch.float64, device=dev) for _ in range(4)]
print("2. hourly: {} days x {} steps, device: int16 {:.2f} GB, float32 {:.2f} GB; referenced {:.2f} / {:.2f} GB".format(
    D, S, r.numel() * 2 / 1e9, x32.numel() * 4 / 1e9, D * S * pieces.size * 8 / 1e9, D * S * pieces.size * 16 / 1e9))
EDD = (C.c_double * 4)(283.15, 290.0, 295.5, 300.0)
dsts = (C.c_void_p * 4)(*[q.data_ptr() for q in planes])


def mean(k):
    if k == "int16":
        return lambda: N.check(L.ctb_pull_pack_daily_decode(p8._h, C.c_void_p(r.data_ptr()), ncell, C.byref(DEC32), S,
                                                            None, 0, D, N.DAILY_MEAN, C.c_void_p(planes[0].data_ptr()),
                                                            None, None, stream()))
    return lambda: N.check(L.ctb_pull_pack_daily(p8._h, C.c_void_p(x32.data_ptr()), N.F32, ncell, S, None, 0, D,
                                                 N.DAILY_MEAN, C.c_void_p(planes[0].data_ptr()), None, None, stream()))


def edd4(k):
    if k == "int16":
        return lambda: N.check(L.ctb_pull_pack_daily_steps_decode(p8._h, C.c_void_p(r.data_ptr()), ncell,
                                                                  C.byref(DEC32), S, None, 0, D, N.STEP_EDD, EDD, 4, 4,
                                                                  dsts, stream()))
    return lambda: N.check(L.ctb_pull_pack_daily_steps(p8._h, C.c_void_p(x32.data_ptr()), N.F32, ncell, S, None, 0, D,
                                                       N.STEP_EDD, EDD, 4, 4, dsts, stream()))


for name, make in (("daily mean", mean), ("EDD x4", edd4)):
    out = {}
    for k in ("int16", "float32"):
        make(k)()
        torch.cuda.synchronize()
        out[k] = [q.clone() for q in planes]
    same = all(torch.equal(a.view(torch.int64), b.view(torch.int64)) for a, b in zip(out["int16"], out["float32"]))
    ts = {"int16": [], "float32": []}
    for _ in range(args.rounds):
        for k in ts:
            ts[k].append(timed(make(k), 1)[0])
    print("   reduce-pack {:10s} int16 median {:.3f} ms (min {:.3f}), float32 median {:.3f} ms (min {:.3f}); "
          "planes bit identical {}".format(name, np.median(ts["int16"]), min(ts["int16"]), np.median(ts["float32"]),
                                           min(ts["float32"]), same))
print("peak memory allocated through torch: {:.1f} GB".format(torch.cuda.max_memory_allocated() / 1e9))
