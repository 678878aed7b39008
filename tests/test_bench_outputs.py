"""bench.py --dump-outputs: what the timed path computed in its last step, sampled the same way on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import oracle
from conftest import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_samples_a_large_block_the_same_way_every_time(tmp_path):
    import torch
    R, T = 500, 40
    out = torch.arange(4 * R * T, dtype=torch.float64).view(4, R, T)     # value = (k * R + row) * T + day
    budget = 4 * 8 * 100 * T                                             # room for 100 of the 500 rows
    bench.dump_outputs(out, "poly", str(tmp_path / "full"))
    bench.dump_outputs(out, "poly", str(tmp_path / "a"), budget=budget)
    bench.dump_outputs(out, "poly", str(tmp_path / "b"), budget=budget)
    assert sorted(os.listdir(tmp_path / "a")) == ["p1.npy", "p2.npy", "p3.npy", "p4.npy"]
    for k, name in enumerate(bench.OUTPUT_NAMES["poly"]):
        full = np.load(tmp_path / "full" / (name + ".npy"))
        assert full.dtype == np.float64 and np.array_equal(full, out[k].numpy())
        a = np.load(tmp_path / "a" / (name + ".npy"))
        assert a.dtype == np.float64 and a.shape == (100, T)
        np.testing.assert_array_equal(a, np.load(tmp_path / "b" / (name + ".npy")))
        rows = (a[:, 0] / T - k * R).astype(np.int64)
        assert np.all(np.diff(rows) > 0)                                 # sorted, distinct region rows
        np.testing.assert_array_equal(a, full[rows])                     # whole rows, every day
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget + 4 * 256


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_result(tmp_path):
    """Config 1 (1 degree, 3,000 regions, 365 days): the dumped block is the aggregation of bench.py's seeded
    input, checked against the oracle on three days; --steps sets the number of timed steps."""
    import torch
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "config1", "--steps", "3",
                        "--warmup", "1", "--no-e2e", "--no-cpu", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] > 0 and line["gpu_launches"] % 3 == 0
    assert os.listdir(tmp_path) == ["tas.npy"]
    got = np.load(tmp_path / "tas.npy")
    from climate_toolbox_b200 import synthetic
    deg, R, T, aggwt = bench.WORKLOADS["config1"][:4]
    lat, lon = synthetic.grid_labels(deg)
    df = synthetic.weights_table(deg, R)
    g = torch.Generator(device="cuda").manual_seed(7)                   # bench.Bench.inputs, rank 0
    x = 288.0 + 10.0 * torch.randn((T, len(lat) * len(lon)), generator=g, device="cuda", dtype=torch.float32)
    days = [0, 181, 364]
    sl = x[days].cpu().numpy().reshape(len(days), len(lat), len(lon))
    ref, dims, labels = oracle.weighted_aggregate_grid_to_regions(sl, ("time", "lat", "lon"), lat, lon, df, aggwt,
                                                                  "hierid")
    scale = oracle.weighted_aggregate_grid_to_regions(np.abs(sl), ("time", "lat", "lon"), lat, lon, df, aggwt,
                                                      "hierid")[0]
    assert got.dtype == np.float64 and got.shape == (len(labels), T)
    assert rel_err(got[:, days].T, ref, scale) <= 1e-9
