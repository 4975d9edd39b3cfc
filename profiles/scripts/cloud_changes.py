#!/usr/bin/env python
"""What change tracking costs and saves on one GPU.

    python profiles/scripts/cloud_changes.py [--out profiles/cloud_changes_1gpu.jsonl] [--cycles 12]

Workloads (bench.py's definitions, FUSED merge, device-resident frames, the images reused along bench.py's lawnmower
trajectory so the resident map keeps growing cycle after cycle):
  - config2_semidense_720p (BASELINE.json configs[1]): 50 frames of 1280x720 per cycle, voxel 0.05;
  - config5_4k_u16_v001: 10 frames of 3840x2160 u16 per cycle, voxel 0.01.

Three contexts per workload see the same frames in every cycle: `off` (tracking off), `on_host` and `on_dev` (tracking on,
read by o3r_cloud_changes and o3r_cloud_changes_dev after every cycle).  Per cycle, after one untimed warm-up cycle:
  - step time (o3r_frames_cloud_dev, CUDA events on o3r_stream) of `off` and `on_host`, the two run alternately;
  - read time, host wall clock to return (every read ends in a stream sync): o3r_cloud_changes (query + fill) on
    `on_host`, o3r_cloud_changes_dev on `on_dev`, o3r_cloud_downsample (query + fill) and o3r_cloud_downsample_dev on `off`;
  - records returned against resident cells, and launches per cycle of `off` and `on_host`.
At the end the consumer's map of `on_host` (every result upserted by key) must equal its o3r_cloud_downsample bit for bit.
Writes one JSON line per workload, with the GPU name, power limit and SM clock read in the same run (read-only queries).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402
from online_3d_reconstruction_b200 import abi  # noqa: E402
from online_3d_reconstruction_b200.pose import Pose  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        v = [x.strip() for x in q.strip().split(",")]
        info["power_limit_w"], info["sm_mhz"], info["sm_max_mhz"] = float(v[0]), float(v[1]), float(v[2])
    except Exception as e:   # reported, never guessed
        info["power_limit_w"] = f"unavailable ({e})"
    return info


def frames_dev(disp, bgr, Ts, dev):
    d = [torch.from_numpy(a).to(dev) for a in disp]
    b = [torch.from_numpy(a).to(dev) for a in bgr]
    arr = (abi.Frame * len(Ts))()
    for i, T in enumerate(Ts):
        arr[i].disp, arr[i].disp_step = d[i].data_ptr(), disp[i].strides[0]
        arr[i].bgr, arr[i].bgr_step = b[i].data_ptr(), bgr[i].strides[0]
        arr[i].T = (C.c_float * 16)(*np.asarray(T, dtype=np.float32).reshape(16))
    return arr, d + b


def step_ms(P, arr, dt):
    st = torch.cuda.ExternalStream(P.stream())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    P.createCycleClouds(arr, dt, device_pointers=True)
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b)


def wall_ms(fn):
    t = time.perf_counter()
    r = fn()
    return (time.perf_counter() - t) * 1e3, r


def run(wl, cycles):
    rows, cols, dt, J, v, mp, nd, F, seed, qs = bench.WORKLOADS[wl]
    disp, bgr, T = bench.make_data(wl, 0, 1, cycles + 1)
    dev = torch.device("cuda:0")
    p = bench.params_for(wl, 0, abi.MERGE_ACCUMULATE_FUSED)
    rec = {k: [] for k in ("step_ms_off", "step_ms_on", "changes_host_ms", "changes_dev_ms", "downsample_host_ms",
                           "downsample_dev_ms", "records_changed", "records_downsample", "resident_cells",
                           "launches_off", "launches_on")}
    with Pose(p) as off, Pose(p) as on_host, Pose(p) as on_dev:
        on_host.trackCloudChanges(True)
        on_dev.trackCloudChanges(True)
        keys_map, pts_map = np.zeros(0, np.uint64), np.zeros(0, abi.POINT)
        for c in range(cycles + 1):
            arr, keep = frames_dev(disp, bgr, T[c], dev)
            l0, l1 = off.launch_count(), on_host.launch_count()
            pair = [(off, "step_ms_off"), (on_host, "step_ms_on")]
            times = {}
            for P, name in (pair if c % 2 == 0 else pair[::-1]):
                times[name] = step_ms(P, arr, dt)
            on_dev.createCycleClouds(arr, dt, device_pointers=True)
            la, lb = off.launch_count() - l0, on_host.launch_count() - l1
            t_ch, (pts, keys, _) = wall_ms(on_host.cloudChanges)
            t_cd, (_, _, _, n_dev) = wall_ms(on_dev.cloudChangesDevice)
            t_dh, ds = wall_ms(off.downsamplePtCloud)
            t_dd, (_, n_dd) = wall_ms(off.downsamplePtCloudDevice)
            k = np.concatenate([keys, keys_map])
            q = np.concatenate([pts, pts_map])
            keys_map, first = np.unique(k, return_index=True)
            pts_map = q[first]
            del keep
            if c == 0:
                continue   # warm-up (the first read is also the full state)
            for name in times:
                rec[name].append(round(times[name], 4))
            rec["changes_host_ms"].append(round(t_ch, 4)); rec["changes_dev_ms"].append(round(t_cd, 4))
            rec["downsample_host_ms"].append(round(t_dh, 4)); rec["downsample_dev_ms"].append(round(t_dd, 4))
            rec["records_changed"].append(int(len(keys))); rec["records_downsample"].append(int(len(ds)))
            rec["resident_cells"].append(int(on_host.cloudSize()))
            rec["launches_off"].append(int(la)); rec["launches_on"].append(int(lb))
            assert n_dev == len(keys) and n_dd == len(ds)
        final = on_host.downsamplePtCloud()
        parity = bool(np.array_equal(pts_map.view(np.uint32), final.view(np.uint32)))
    med = {f"median_{k}": float(np.median(v)) for k, v in rec.items() if v and k.endswith("_ms")}
    med["median_extra_launches_per_cycle"] = float(np.median(np.subtract(rec["launches_on"], rec["launches_off"])))
    med["median_changed_over_resident"] = float(np.median(np.divide(rec["records_changed"], rec["resident_cells"])))
    return {"workload": wl, "merge_mode": "fused", "frames_per_cycle": F, "frame": f"{cols}x{rows}", "voxel_size": v,
            "cycles_timed": cycles, "warmup_cycles": 1, "map_equals_downsample": parity, **med, "per_cycle": rec}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cloud_changes_1gpu.jsonl"))
    ap.add_argument("--cycles", type=int, default=12)
    ap.add_argument("--workloads", default="config2_semidense_720p,config5_4k_u16_v001")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    info = gpu_info()
    for wl in a.workloads.split(","):
        r = run(wl, a.cycles)
        r["gpu"] = info
        line = json.dumps(r)
        print(line, flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
