"""o3r_cloud_register timings on one GPU -> profiles/register_1gpu.jsonl (or argv[1]): time per call and iterations used for
10 k / 100 k / 1 M source points against maps of about 0.4 M and 10 M cells, and the host driver's cycle time with and
without --register_map.  The card's name and power limit are read in the same run and written with every record."""
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import register_model as reg  # noqa: E402
from online_3d_reconstruction_b200 import abi  # noqa: E402
from online_3d_reconstruction_b200.pose import Pose  # noqa: E402

V = 1.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit": q[1] if len(q) > 1 else "unknown"}


def map_cells(side, h):
    """side x side cells of 1 m, 4 points each at the terrain height of the cell centre."""
    g = np.arange(side, dtype=np.float64) - side / 2 + 0.5
    x, y = np.meshgrid(g, g)
    x, y = x.ravel(), y.ravel()
    z = h(x, y)
    c = np.zeros(x.size, dtype=abi.CELL)
    i, j = np.floor(x).astype(np.int64), np.floor(y).astype(np.int64)
    import reduce_model as rm
    c["key"] = rm.cell_keys(i, j, np.zeros_like(i))
    c["n"] = 4
    c["sx"], c["sy"], c["sz"] = (4 * x).astype(np.float32), (4 * y).astype(np.float32), (4 * (z + 500.0)).astype(np.float32)
    return c[np.argsort(c["key"])]


def source(n, half, h, rng):
    x, y = rng.uniform(-half, half, n), rng.uniform(-half, half, n)
    p = np.zeros(n, dtype=abi.POINT)
    p["x"], p["y"], p["z"] = x.astype(np.float32), y.astype(np.float32), h(x, y).astype(np.float32)
    return reg.transform_points(p, reg.rigid(yaw_deg=1.0, roll_deg=0.5, t=(0.3, 0.3, 0.3)))


def driver_cycles(flag):
    from test_host_driver_register import _write_same_frames
    with tempfile.TemporaryDirectory() as d:
        _write_same_frames(os.path.join(d, "data"), 40, 720, 1280, lifted=set(range(10, 40)))
        r = subprocess.run([os.path.join(ROOT, "host", "pose"), "100", "139", "--seq_len", "10", "--jump_pixels", "1",
                            "--voxel_size", "0.05", "--only_MAVLink", "--data_root", os.path.join(d, "data"),
                            "--output", os.path.join(d, "out")] + flag, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        return [float(v) for v in re.findall(r"Cycle time: ([0-9.eE+-]+) sec", r.stdout)]


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "register_1gpu.jsonl")
    info = card()
    h = reg._terrain(7)
    rng = np.random.default_rng(5)
    recs = []
    for side in (632, 3162):
        cells = map_cells(side, h)
        with Pose(abi.make_params(voxel_size=V, merge_mode=abi.MERGE_ACCUMULATE)) as P:
            P.importCells(cells)
            for n in (10_000, 100_000, 1_000_000):
                src = source(n, min(side / 2 - 5, 150.0), h, rng)
                P.registerCloud(src)   # warm-up (module load, staging buffer)
                ts = []
                for _ in range(5):
                    t0 = time.perf_counter()
                    _, st = P.registerCloud(src)
                    ts.append(time.perf_counter() - t0)
                recs.append({**info, "what": "o3r_cloud_register", "map_cells": int(len(cells)), "points": n,
                             "ms_per_call_median": 1e3 * float(np.median(ts)), "ms_per_call_min": 1e3 * min(ts),
                             "iterations": st["iterations"], "converged": st["converged"], "n_inliers": st["n_inliers"]})
                print(recs[-1], flush=True)
    for flag in ([], ["--register_map"]):
        c = driver_cycles(flag)
        recs.append({**info, "what": "host/pose cycle time, 720x1280, 10 frames per cycle, 4 cycles",
                     "flags": " ".join(flag) or "(none)", "cycle_s": c, "cycle_s_after_first_median": float(np.median(c[1:]))})
        print(recs[-1], flush=True)
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
