#!/usr/bin/env python
"""Weak scaling of the sharded RETAIN (ICP-on) mode: N ranks, one GPU each, under torch.distributed.run.

    python -m torch.distributed.run --nproc-per-node N profiles/scripts/retain_scaling.py [--out FILE] [--cycles 6]

Workload: BASELINE.json configs[1] geometry (synth.uav720-style 1280x720 u8 disparity, jump_pixels 1, voxel_size 0.05,
min_points_per_voxel 1) in O3R_MERGE_RETAIN mode, 50 device-resident frames per rank and cycle (o3r_frames_cloud_dev), each
cycle followed by o3r_cloud_transform with a small rotation + translation (pose.cpp:350-354), then one collective
o3r_cloud_downsample.  One untimed pass warms every shape up; the timed pass repeats it from an empty cloud.

Rank 0 prints ONE JSON line (and appends it to --out): the cycle step (frames + transform, CUDA events, slowest rank), the
final downsample (host wall time to its sync, slowest rank) and its split into local prep / exchange / owner reduction
(o3r_profile phases of a second, profiled downsample of the same cloud), frames/s, the weak-scaling efficiency against the
1-rank line already in --out (if any), the retained points per rank, and the GPU name and power limit read in the same run.
A parity leg first checks, at a smaller size, that the union of the shards equals single-rank RETAIN bit for bit.
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
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from online_3d_reconstruction_b200 import abi, synth  # noqa: E402
from online_3d_reconstruction_b200.pose import Pose  # noqa: E402

ROWS, COLS, VOXEL, SEED = 720, 1280, 0.05, 1002


def tf_icp(k):
    """A small rigid correction (about 0.5 degree of yaw, a few cm), different per cycle."""
    a = 0.008 + 0.001 * k
    tf = np.eye(4, dtype=np.float32)
    c, s = np.float32(np.cos(a)), np.float32(np.sin(a))
    tf[0, 0], tf[0, 1], tf[1, 0], tf[1, 1] = c, -s, s, c
    tf[:3, 3] = [0.03, -0.02, 0.01 * (k % 3)]
    return tf


def params(local):
    return abi.make_params(rows=ROWS, cols=COLS, jump_pixels=1, voxel_size=VOXEL, min_points_per_voxel=1,
                           merge_mode=abi.MERGE_RETAIN, device=local, max_batch_frames=64)


def frames_dev(disp, bgr, Ts, dev):
    """Device-resident frames (torch tensors kept alive by the caller) -> (ctypes frame array, tensors)."""
    d = [torch.from_numpy(a).to(dev) for a in disp]
    b = [torch.from_numpy(a).to(dev) for a in bgr]
    arr = (abi.Frame * len(Ts))()
    for i, T in enumerate(Ts):
        arr[i].disp, arr[i].disp_step = d[i].data_ptr(), disp[i].strides[0]
        arr[i].bgr, arr[i].bgr_step = b[i].data_ptr(), bgr[i].strides[0]
        arr[i].T = (C.c_float * 16)(*np.asarray(T, dtype=np.float32).reshape(16))
    return arr, d + b


def cell_keys(a):
    """64-bit absolute cell key of each record on the combined grid (leaf v, v, 1000 after z += 500), as the device."""
    inv = np.float32(1.0) / np.float32(VOXEL)
    i = np.floor(a["x"] * inv).astype(np.int64)
    j = np.floor(a["y"] * inv).astype(np.int64)
    k = np.floor((a["z"] + np.float32(500)) * (np.float32(1.0) / np.float32(1000.0))).astype(np.int64)
    B = 1 << 20
    return ((k + B).astype(np.uint64) << np.uint64(42)) | ((j + B).astype(np.uint64) << np.uint64(21)) | (i + B).astype(np.uint64)


def parity_leg(rank, world, local, dev, uid):
    """Two cycles of 2 frames per rank with a transform between: union of the shards == single-rank RETAIN, bit for bit."""
    per_rank, n_cyc = 2, 2
    n = per_rank * world
    seq = synth.sequence(SEED + 17, n * n_cyc, ROWS, COLS)
    tf = tf_icp(0)
    keep = []
    cyc = [seq[s * n:(s + 1) * n] for s in range(n_cyc)]
    with Pose(params(local)) as P:
        P.commInit(world, rank, uid, 1 << 16)
        for s, c in enumerate(cyc):
            if s:
                P.transformPtCloud(tf)
            mine = c[rank::world]
            arr, t = frames_dev([x[0] for x in mine], [x[1] for x in mine], [x[2] for x in mine], dev)
            keep.append(t)
            P.createCycleClouds(arr, abi.DISP_U8, device_pointers=True)
        shard = P.downsamplePtCloud()
        P.commDestroy()
    shards = [None] * world
    dist.gather_object(shard, shards if rank == 0 else None, dst=0)
    if rank != 0:
        return None
    with Pose(params(local)) as S:
        for s, c in enumerate(cyc):
            if s:
                S.transformPtCloud(tf)
            arr, t = frames_dev([x[0] for x in c], [x[1] for x in c], [x[2] for x in c], dev)
            keep.append(t)
            S.createCycleClouds(arr, abi.DISP_U8, device_pointers=True)
        single = S.downsamplePtCloud()
    union = np.concatenate(shards)
    union = union[np.argsort(cell_keys(union), kind="stable")]
    ok = bool(np.array_equal(union.view(np.uint32), single.view(np.uint32)))
    return {"frames": n * n_cyc, "cells": int(len(single)), "shards": [int(len(s)) for s in shards], "array_equal": ok}


def gpu_info(local):
    info = {"name": torch.cuda.get_device_name(local)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:   # reported, never guessed
        info["power_limit_w"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="append the JSON line here (and read the 1-rank line for the efficiency)")
    ap.add_argument("--cycles", type=int, default=6)
    ap.add_argument("--frames", type=int, default=50, help="frames per rank and cycle")
    a = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if "RANK" not in os.environ:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", RANK="0", WORLD_SIZE="1")
    dist.init_process_group("gloo")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    def new_uid():
        box = [Pose.commUniqueId() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    parity = parity_leg(rank, world, local, dev, new_uid())

    # this rank's 50 frames (the same images every cycle, new poses: rank r holds global frames i * world + r)
    F, K = a.frames, a.cycles
    seq = synth.sequence(SEED + 101 * rank, F, ROWS, COLS)
    Ts = synth.trajectory(np.random.default_rng(SEED + 7919), K * world * F)
    cyc = []
    keep = []
    for s in range(K):
        arr, t = frames_dev([x[0] for x in seq], [x[1] for x in seq], [Ts[s * world * F + i * world + rank] for i in range(F)], dev)
        cyc.append(arr)
        keep.append(t)
    torch.cuda.synchronize()
    P = Pose(params(local))
    P.commInit(world, rank, new_uid(), 1 << 16)
    stream = torch.cuda.ExternalStream(P.stream(), device=dev)

    def one_pass():
        P.clearCloud()
        step_ms = []
        for s in range(K):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            P.createCycleClouds(cyc[s], abi.DISP_U8, device_pointers=True)
            P.transformPtCloud(tf_icp(s))
            e1.record(stream)
            e1.synchronize()
            step_ms.append(e0.elapsed_time(e1))
        dist.barrier()
        t0 = time.perf_counter()
        _, m = P.downsamplePtCloudDevice()
        ds_ms = (time.perf_counter() - t0) * 1e3
        return step_ms, ds_ms, m

    one_pass()                                        # warm-up: every buffer and shape of the timed pass
    step_ms, ds_ms, m = one_pass()
    retained = P.cloudSize()
    # split of the same collective: identity transform (exact in float) drops the kept result, then a profiled downsample
    P.transformPtCloud(np.eye(4, dtype=np.float32))
    dist.barrier()
    P.profile(True)
    P.downsamplePtCloudDevice()
    prof = P.profileRead()
    P.profile(False)
    P.commDestroy()
    P.close()
    split = {k: round(prof.get(k, (0, 0.0))[1], 3) for k in ("retain_prep", "retain_exchange", "retain_reduce")}

    mine = {"rank": rank, "step_ms": step_ms, "downsample_ms": ds_ms, "cells": int(m), "retained_points": int(retained),
            "split_ms": split}
    allr = [None] * world
    dist.gather_object(mine, allr if rank == 0 else None, dst=0)
    if rank == 0:
        step_max = [max(r["step_ms"][s] for r in allr) for s in range(K)]
        ds_max = max(r["downsample_ms"] for r in allr)
        total_ms = sum(step_max) + ds_max
        fps = world * F * K / (total_ms / 1e3)
        line = {
            "metric": "retain_sharded_weak_scaling", "world": world, "frames_per_rank_per_cycle": F, "cycles": K,
            "workload": "configs[1] geometry: 1280x720 u8, jump_pixels 1, voxel_size 0.05, min_points_per_voxel 1, MERGE_RETAIN, "
                        "device-resident inputs, o3r_cloud_transform after every cycle",
            "cycle_step_ms": [round(x, 3) for x in step_max], "cycle_step_ms_mean": round(float(np.mean(step_max)), 3),
            "downsample_wall_ms": round(ds_max, 3),
            "downsample_split_ms_per_rank": [r["split_ms"] for r in allr],
            "frames_per_s": round(fps, 1),
            "retained_points_per_rank": [r["retained_points"] for r in allr],
            "cells_per_rank": [r["cells"] for r in allr],
            "parity_small_run": parity,
            "gpu": gpu_info(local),
            "timing": "cycle step: CUDA events on the context's stream, slowest rank per cycle; downsample: host wall time of "
                      "o3r_cloud_downsample_dev (ends in a sync), slowest rank; split: o3r_profile phase events of a second, "
                      "profiled downsample of the same cloud",
        }
        if a.out and os.path.exists(a.out):
            for ln in open(a.out):
                try:
                    ref = json.loads(ln)
                except ValueError:
                    continue
                if ref.get("metric") == line["metric"] and ref.get("world") == 1:
                    line["weak_scaling_efficiency"] = round(fps / (world * ref["frames_per_s"]), 3)
        print(json.dumps(line), flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(line) + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
