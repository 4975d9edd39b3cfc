#!/usr/bin/env python
"""What a map checkpoint costs on one GPU: o3r_cloud_export_cells and o3r_cloud_import_cells at two map sizes.

    python profiles/scripts/map_checkpoint.py [--out profiles/map_checkpoint_1gpu.jsonl] [--reps 5]

Workloads (bench.py's definitions, FUSED merge, device-resident frames along bench.py's lawnmower trajectory, so the map
grows cycle after cycle):
  - config2_semidense_720p (BASELINE.json configs[1]) after 10 cycles: about 0.4 M cells (15 MB of records);
  - config5_4k_u16_v001 after 8 cycles: about 10^7 cells (400 MB of records).

Per workload, on the final map: export_cells (fill only, the size is known) into a page-locked buffer (o3r_host_alloc) and
into a pageable numpy buffer, then import_cells of those records into a fresh context from each kind of buffer, `reps`
times each, the two buffer kinds alternating.  Every call synchronises before it returns, so a host clock around it
measures the call.  The first import into a fresh context also allocates the resident buffers; that is part of what a
resume costs, so every import is timed into a new context.  Checked in the same run: the map exported two cycles before
the end, imported into a new context that then runs the last two cycles, downsamples to the uninterrupted run's cloud
within the FUSED contract (same cells in the same order, colours exact, centroids within 1e-5 relative), and bit for bit
whenever the resumed context served the remaining cycles with the same engines (both are recorded); the fused
mode picks the engine, and whether to pre-reduce, from the context's own batch history, which a checkpoint does not carry.
Writes one JSON line per workload, with the GPU name and power limit read in the same run.
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


def wall_ms(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3


def run(wl, cycles, reps):
    L = lib.load()
    rows, cols, dt, J, v, mp, nd, F, seed, qs = bench.WORKLOADS[wl]
    disp, bgr, T = bench.make_data(wl, 0, 1, cycles)
    dev = torch.device("cuda:0")
    p = bench.params_for(wl, 0, abi.MERGE_ACCUMULATE_FUSED)
    rec = {k: [] for k in ("export_pinned_ms", "export_pageable_ms", "import_pinned_ms", "import_pageable_ms")}
    engines, engines_resumed = [], []
    with Pose(p) as A:
        for c in range(cycles):
            arr, keep = frames_dev(disp, bgr, T[c], dev)
            A.createCycleClouds(arr, dt, device_pointers=True)
            engines.append(A.lastCycleEngine())
            if c == cycles - 3:
                mid = A.exportCells()
            del keep
        A.sync()
        n = A.cloudSize()
        full_ds = A.downsamplePtCloud()
        nbytes = n * abi.CELL.itemsize
        ptr = L.o3r_host_alloc(nbytes)
        assert ptr, "o3r_host_alloc failed"
        try:
            pinned = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr)).view(abi.CELL)
            pageable = np.empty(n, dtype=abi.CELL)
            bufs = {"pinned": pinned, "pageable": pageable}
            m = C.c_size_t(0)
            A.exportCells()   # warm-up: the pack buffer is allocated here
            for r in range(reps):
                for kind in (("pinned", "pageable") if r % 2 == 0 else ("pageable", "pinned")):
                    b = bufs[kind]
                    rec[f"export_{kind}_ms"].append(round(wall_ms(lambda: lib_ok(L.o3r_cloud_export_cells(
                        A.handle, b.ctypes.data, n, C.byref(m)), A)), 4))
                    assert m.value == n
            assert pinned.tobytes() == pageable.tobytes()
            for r in range(reps):
                for kind in (("pinned", "pageable") if r % 2 == 0 else ("pageable", "pinned")):
                    b = bufs[kind]
                    with Pose(p) as Q:
                        rec[f"import_{kind}_ms"].append(round(wall_ms(lambda: lib_ok(L.o3r_cloud_import_cells(
                            Q.handle, b.ctypes.data, n), Q)), 4))
                        if r == 0:
                            assert Q.exportCells().tobytes() == pinned.tobytes(), "import is not a bit copy"
        finally:
            L.o3r_host_free(ptr)
    # resume two cycles before the end: the same frames, the same result
    with Pose(p) as B:
        B.importCells(mid)
        for c in range(cycles - 2, cycles):
            arr, keep = frames_dev(disp, bgr, T[c], dev)
            B.createCycleClouds(arr, dt, device_pointers=True)
            engines_resumed.append(B.lastCycleEngine())
            del keep
        resumed = B.downsamplePtCloud()
    resumed_bitwise = bool(np.array_equal(resumed.view(np.uint32), full_ds.view(np.uint32)))
    assert resumed.shape == full_ds.shape and np.array_equal(resumed["rgb"], full_ds["rgb"]), "the resumed run has other cells"
    rel = 0.0
    for f, sh in (("x", 0.0), ("y", 0.0), ("z", 500.0)):
        a, b = resumed[f].astype(np.float64) + sh, full_ds[f].astype(np.float64) + sh
        rel = max(rel, float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-3), initial=0.0)))
    assert rel <= 1e-5, f"resumed centroids differ by {rel:.3g} relative"
    assert resumed_bitwise or engines_resumed != engines[-2:], "same engines after the resume, yet not bit for bit"
    med = {f"median_{k}": float(np.median(x)) for k, x in rec.items()}
    gbps = {f"{k[7:-3]}_GB_per_s": round(nbytes / (med[k] * 1e-3) / 1e9, 3) for k in med}
    return {"workload": wl, "merge_mode": "fused", "frames_per_cycle": F, "frame": f"{cols}x{rows}", "voxel_size": v,
            "cycles": cycles, "cells": int(n), "record_bytes": int(nbytes), "reps": reps,
            "resumed_bitwise_equal": resumed_bitwise, "resumed_max_centroid_rel": rel,
            "engines": engines, "engines_resumed": engines_resumed, "mid_checkpoint_cells": int(len(mid)), **med, **gbps,
            "per_rep": rec}


def lib_ok(rc, P):
    if rc != 0:
        raise lib.O3RError(rc, P._L.o3r_last_error(P.handle).decode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "map_checkpoint_1gpu.jsonl"))
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
