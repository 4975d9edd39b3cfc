#!/usr/bin/env python
"""What o3r_cloud_mesh costs on one GPU, beside o3r_cloud_downsample on the same map.

    python profiles/scripts/mesh_map.py [--out profiles/mesh_1gpu.jsonl] [--reps 5]

Workloads (bench.py's definitions, FUSED merge, device-resident frames along bench.py's lawnmower trajectory, as
map_checkpoint.py builds them):
  - config2_semidense_720p (BASELINE.json configs[1]) after 10 cycles of 50 frames: about 0.4 M cells;
  - config5_4k_u16_v001 after 8 cycles: about 10^7 cells.

Per workload, on the final map, `reps` times each and alternating: o3r_cloud_mesh (no gate) into page-locked buffers
(o3r_host_alloc) and into pageable numpy buffers, o3r_cloud_mesh_dev, and o3r_cloud_downsample into page-locked and
pageable buffers and _dev.  Every call synchronises before it returns, so a host clock around it measures the call.  Also
recorded: the vertex and triangle counts with and without a 1 m gate, and the mesh's per-kernel times from o3r_profile in
one separate call.  One JSON line per workload, with the GPU name, power limit and SM clock read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import bench  # noqa: E402
from cloud_changes import frames_dev, gpu_info  # noqa: E402
from online_3d_reconstruction_b200 import abi, lib  # noqa: E402
from online_3d_reconstruction_b200.pose import Pose  # noqa: E402


def ok(rc, P):
    if rc != 0:
        raise lib.O3RError(rc, P._L.o3r_last_error(P.handle).decode())


def wall_ms(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3


def pinned(L, nbytes, keep):
    ptr = L.o3r_host_alloc(max(nbytes, 1))
    assert ptr, "o3r_host_alloc failed"
    keep.append(ptr)
    return np.ctypeslib.as_array((C.c_uint8 * max(nbytes, 1)).from_address(ptr))


def run(wl, cycles, reps):
    L = lib.load()
    rows, cols, dt, J, v, mp, nd, F, seed, qs = bench.WORKLOADS[wl]
    disp, bgr, T = bench.make_data(wl, 0, 1, cycles)
    dev = torch.device("cuda:0")
    p = bench.params_for(wl, 0, abi.MERGE_ACCUMULATE_FUSED)
    calls = ("mesh_pinned", "mesh_pageable", "mesh_dev", "downsample_pinned", "downsample_pageable", "downsample_dev")
    rec = {k + "_ms": [] for k in calls}
    held = []
    with Pose(p) as A:
        for c in range(cycles):
            arr, keep = frames_dev(disp, bgr, T[c], dev)
            A.createCycleClouds(arr, dt, device_pointers=True)
            del keep
        A.sync()
        cells = A.cloudSize()
        inf = float("inf")
        nv, nt = C.c_size_t(0), C.c_size_t(0)
        ok(L.o3r_cloud_mesh(A.handle, inf, None, None, 0, C.byref(nv), None, 0, C.byref(nt)), A)
        nv, nt = nv.value, nt.value
        bufs = {
            "pinned": (pinned(L, nv * 16, held), pinned(L, nv * 12, held), pinned(L, nt * 12, held)),
            "pageable": (np.empty(nv * 16, np.uint8), np.empty(nv * 12, np.uint8), np.empty(nt * 12, np.uint8)),
        }
        dsb = {"pinned": pinned(L, nv * 16, held), "pageable": np.empty(nv * 16, np.uint8)}
        m1, m2 = C.c_size_t(0), C.c_size_t(0)
        pv, pn, pt = C.c_void_p(), C.c_void_p(), C.c_void_p()

        def mesh(kind):
            vb, nb, tb = bufs[kind]
            ok(L.o3r_cloud_mesh(A.handle, inf, vb.ctypes.data, nb.ctypes.data, nv, C.byref(m1), tb.ctypes.data, nt,
                                C.byref(m2)), A)

        def mesh_dev():
            ok(L.o3r_cloud_mesh_dev(A.handle, inf, C.byref(pv), C.byref(pn), C.byref(m1), C.byref(pt), C.byref(m2)), A)

        def ds(kind):
            ok(L.o3r_cloud_downsample(A.handle, dsb[kind].ctypes.data, nv, C.byref(m1)), A)

        def ds_dev():
            ok(L.o3r_cloud_downsample_dev(A.handle, C.byref(pv), C.byref(m1)), A)

        fns = {"mesh_pinned": lambda: mesh("pinned"), "mesh_pageable": lambda: mesh("pageable"), "mesh_dev": mesh_dev,
               "downsample_pinned": lambda: ds("pinned"), "downsample_pageable": lambda: ds("pageable"),
               "downsample_dev": ds_dev}
        for f in fns.values():   # warm-up: buffers are allocated and modules loaded here
            f()
        for r in range(reps):
            for k in (calls if r % 2 == 0 else calls[::-1]):
                rec[k + "_ms"].append(round(wall_ms(fns[k]), 4))
        assert bufs["pinned"][0].tobytes() == dsb["pinned"].tobytes() == bufs["pageable"][0].tobytes()
        assert bufs["pinned"][2].tobytes() == bufs["pageable"][2].tobytes()
        gated = A.meshCloud(1.0)
        A.profile(True)
        mesh_dev()
        prof = {k: round(v[1], 4) for k, v in A.profileRead().items()}
        A.profile(False)
    for ptr in held:
        L.o3r_host_free(ptr)
    med = {f"median_{k}": float(np.median(x)) for k, x in rec.items()}
    return {"workload": wl, "merge_mode": "fused", "frames_per_cycle": F, "frame": f"{cols}x{rows}", "voxel_size": v,
            "cycles": cycles, "cells": int(cells), "vertices": nv, "triangles": nt, "triangles_gate_1m": int(len(gated[2])),
            "mesh_bytes_d2h": nv * 28 + nt * 12, "reps": reps, **med, "mesh_dev_kernel_ms": prof, "per_rep": rec}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mesh_1gpu.jsonl"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="config2_semidense_720p:10,config5_4k_u16_v001:8")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    info = gpu_info()
    for item in a.workloads.split(","):
        wl, cycles = item.split(":")
        r = run(wl, int(cycles), a.reps)
        r["gpu"] = info
        line = json.dumps(r)
        print(line, flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
