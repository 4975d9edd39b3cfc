#!/usr/bin/env python
"""bench.py — frames/s of the disparity -> voxel-cloud hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--dump-outputs DIR]

A "step" is one reconstruction cycle of the reference (pose.cpp:361-434 + :527-531): seq_len = 50 accepted
frames go through createAndTransformPtCloud (validity mask, Q reprojection, rigid transform, per-frame
VoxelGrid at voxel_size/5), are merged into the global cloud, and the combined VoxelGrid cloud
(voxel_size, min_points_per_voxel) is produced.  Workload at N = 1 is BASELINE.json configs[1]:
1280x720 u8 disparity, --jump_pixels 1 --voxel_size 0.05 --min_points_per_voxel 1, synthetic uav720(seed=1002).
StatisticalOutlierRemoval (pose_functions.cpp:1673-1686) is excluded on both the GPU and the CPU side
(SURVEY §8f-1, not built yet).

Prints ONE JSON line (rank 0).  `value` times the cycle with inputs resident in HBM; `e2e` times the same
cycle through the host-pointer C-ABI call from pinned host memory (H2D of every frame and D2H of the
result inside the timed region); `roofline` is the dominant kernel's algorithmic bytes / its CUDA-event
time; `cpu_baseline` is the CPU oracle (a port of the reference path) on the box's host cores.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from online_3d_reconstruction_b200 import abi, synth  # noqa: E402

# (workload, kernel) -> dram__bytes_read.sum + dram__bytes_write.sum per launch, from the COMMITTED `ncu --set full` capture of
# the same command (profiles/r02_ncu_full.txt) — a constant of that capture, not a property of this run (roofline.traffic_source)
NCU_TRAFFIC = {
    ("config2_semidense_720p", "k_tv"): 181.9e6,
}
NCU_TRAFFIC_SOURCE = "profiles/r02_ncu_full.txt (ncu --set full --clock-control none, cold caches, one launch)"
# smsp__inst_executed.sum of the same capture: warp instructions one launch of the kernel executes (a property of the build and
# the workload, not of the run) — the numerator of the instruction-issue view below
NCU_WARP_INST = {
    ("config2_semidense_720p", "k_tv"): 702.7e6,
}

WORKLOADS = {
    # name: (rows, cols, disp_type, J, voxel_size, min_pts, dont_downsample, frames/step, seed, Q scale)
    "config2_semidense_720p": (720, 1280, abi.DISP_U8, 1, 0.05, 1, False, 50, 1002, 1.0),
    "config3_dont_downsample_720p": (720, 1280, abi.DISP_U8, 1, 0.05, 1, True, 50, 1003, 1.0),
    "config4_sweep_720p_v002": (720, 1280, abi.DISP_U8, 1, 0.02, 1, False, 50, 1004, 1.0),
    "config5_4k_u16_v001": (2160, 3840, abi.DISP_U16, 1, 0.01, 1, False, 10, 1005, 3.0),
    "config1_sparse_720p": (720, 1280, abi.DISP_U8, 15, 0.05, 1, False, 50, 1001, 1.0),
    # configs[1] with the reference's StatisticalOutlierRemoval(50, 1.0) in front of the per-frame VoxelGrid
    # (pose_functions.cpp:1673-1686) — the full per-frame composition of the reference, SURVEY 8f-1
    "config2_semidense_720p_sor": (720, 1280, abi.DISP_U8, 1, 0.05, 1, False, 50, 1002, 1.0),
}
SOR_MEAN_K = {"config2_semidense_720p_sor": 50}
# configs[1] with the reference's live blur (cv::bilateralFilter(k, 2k, k/2), README's --blur_kernel 30) / the median
# north_star names (odd kernel) in front of the scan: row F of SURVEY 8a on the books
WORKLOADS["config2_semidense_720p_blur30"] = WORKLOADS["config2_semidense_720p"]
WORKLOADS["config2_semidense_720p_median31"] = WORKLOADS["config2_semidense_720p"]
BLUR = {"config2_semidense_720p_blur30": (30, abi.BLUR_BILATERAL), "config2_semidense_720p_median31": (31, abi.BLUR_MEDIAN)}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.time()  # NVML start-up holds driver locks: let it finish before anything is timed
            while not self.rows and time.time() - t0 < 10:
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax = float(r[2])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        hi = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(hi)) if hi else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_data(wl, rank, world, n_steps_total):
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    seq = synth.sequence(seed + 101 * rank, F, rows, cols, disp_type=dt)
    disp = [s[0] for s in seq]
    bgr = [s[1] for s in seq]
    # global cycle of world*F frames per step, frame j -> rank j % world: trajectory index s*world*F + j
    Ts = synth.trajectory(np.random.default_rng(seed + 7919), n_steps_total * world * F)
    T = [[Ts[s * world * F + (i * world + rank)] for i in range(F)] for s in range(n_steps_total)]
    return disp, bgr, T


MERGE_MODES = {"fused": abi.MERGE_ACCUMULATE_FUSED, "tiled": abi.MERGE_ACCUMULATE_TILED, "accumulate": abi.MERGE_ACCUMULATE}
MERGE_MODE = "fused"   # set from --merge-mode
ENGINE_NAMES = {0: "sort", 1: "bucket", 2: "tile"}


def params_for(wl, device, merge_mode=None):
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    if merge_mode is None:
        merge_mode = MERGE_MODES[MERGE_MODE]
    bk, bm = BLUR.get(wl, (1, abi.BLUR_MEDIAN))
    return abi.make_params(rows=rows, cols=cols, jump_pixels=J, voxel_size=v, min_points_per_voxel=mp,
                           dont_downsample=nd, Q=synth.q_scaled(qs), device=device, max_batch_frames=F,
                           merge_mode=merge_mode, sor_mean_k=SOR_MEAN_K.get(wl, 0), blur_kernel=bk, blur_mode=bm)


def static_config(wl, world):
    """The workload description both arms print (the driver compares the two config objects)."""
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    bk, bm = BLUR.get(wl, (1, abi.BLUR_MEDIAN))
    return {"workload": wl, "frames_per_step": F, "frames_per_step_is": "per GPU (weak scaling)", "frame": f"{cols}x{rows}",
            "jump_pixels": J, "voxel_size": v, "min_points_per_voxel": mp, "dont_downsample": nd, "seq_len": F,
            "blur_kernel": bk, "blur": {abi.BLUR_BILATERAL: "bilateral", abi.BLUR_MEDIAN: "median", abi.BLUR_BOX: "box"}[bm] if bk > 1 else "off",
            "synthetic_seed": seed,
            "l2": "inputs and intermediates of a step exceed the 126 MB L2 (184 MB of input planes per 50-frame 720p step)",
            "sor": ("StatisticalOutlierRemoval(50, 1.0) applied per frame on both the GPU and the CPU side" if wl in SOR_MEAN_K
                    else "north_star path: StatisticalOutlierRemoval not applied on either side (sor_mean_k = 0); "
                         "--workload config2_semidense_720p_sor runs the reference's full per-frame composition")}


def frames_array(disp_ptrs, disp_step, bgr_ptrs, bgr_step, Ts):
    n = len(Ts)
    arr = (abi.Frame * n)()
    for i in range(n):
        arr[i].disp, arr[i].disp_step = disp_ptrs[i], disp_step
        arr[i].bgr, arr[i].bgr_step = bgr_ptrs[i], bgr_step
        arr[i].T = (C.c_float * 16)(*Ts[i].reshape(16))
    return arr


# per-kernel algorithmic bytes of one step (what the kernel must read + write once), keyed by profile name.
# n_valid = points after the mask, n_vox = per-frame voxels of the cycle, np1 / np2 = radix passes of the per-frame
# index sort / the combined-grid key sort (7-8 bit digits: 28-bit index -> 4, 20-bit key -> 3).
def algorithmic_bytes(wl, n_valid, n_vox, n_cells_cycle, bd, np1=4, np2=3, n_part=0):
    """n_part = tile partial cells of the cycle (O3R_MERGE_ACCUMULATE_TILED / _FUSED): the merge then sorts and reduces those
    40-byte records instead of the n_vox per-frame voxels.  np1 = radix passes of the per-frame leaf-index sort that actually
    ran (0 when the frame path is the bucket / tile engine or every frame is a PCL pass-through), np2 = passes of the
    combined-grid key sort; the caller derives both from the launches the library counted, not from constants."""
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    p = params_for(wl, 0)
    ny, nx = abi.scan_dims(p)
    npix = ny * nx * F
    m, item = (n_part, 40) if n_part else (n_vox, 16)   # records the merge works on, bytes per gathered record
    return {
        "k_pre": npix * bd,
        "k_emit": npix * bd + npix * 3 + n_valid * (16 + (0 if nd else 4)),
        "k_rs_ghist_u32": n_valid * 4,
        # first pass reads keys only (values are the element index), every pass writes key + value
        "k_rs_onesweep_u32": (n_valid * (4 + 8) + (np1 - 1) * n_valid * 16 if np1 > 0 else 0) + np2 * m * 16,
        "k_vg_heads": n_valid * 4,
        "k_vg_reduce_w": n_valid * (4 + 4 + 16) + n_vox * 16,
        "k_cell_prereduce": n_vox * 16 + n_part * 40,
        # the fused bucket engine (csrc/bucket.cuh): histogram reads the disparity, the scatter reads disparity + colour and
        # writes 16 B point + 4 B scan position, the reduce reads those and writes the partial cells
        "k_bk_hist": npix * bd,
        "k_bk_scatter": npix * bd + npix * 3 + n_valid * 20,
        "k_bk_reduce": n_valid * 20 + n_part * 40,
        # the fused tile engine (csrc/tile.cuh): SURVEY 8d's fused A+B figure — every input plane read once, 20 B per per-frame
        # voxel (which this kernel never materialises: they live and die in shared memory) — the compaction copies the records
        "k_tv": F * (rows * cols * bd + 3 * ny * nx) + 20 * n_vox,
        "k_tv_compact": 2 * 40 * n_part,
        "k_acc_key": m * (item + 8),
        "k_acc_heads": m * 4,
        "k_acc_reduce": m * (4 + 4 + item) + n_cells_cycle * 40,
    }


def _cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(local_rank):
    """Multi-rank runs: keep the rank's host thread — and with it, by first touch, the pinned staging buffers it is about to
    allocate — on the NUMA node the rank's GPU hangs off, so that N ranks' H2D copies read N different memory controllers
    instead of crossing the socket link.  Returns a short description for the JSON line (None when nothing was bound:
    no sysfs entry, a single node, or the node's CPUs are outside this process's allowed set)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = _cpulist(f.read()) & os.sched_getaffinity(0)
        if not cpus or cpus == os.sched_getaffinity(0):
            return None
        os.sched_setaffinity(0, cpus)
        return f"node {node}, {len(cpus)} cpus"
    except Exception:   # binding is an optimisation, never a requirement
        return None


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from online_3d_reconstruction_b200 import exchange as xchg
    from online_3d_reconstruction_b200.lib import O3RError
    from online_3d_reconstruction_b200.pose import Pose

    wl = args.workload
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    W, K = args.warmup, args.steps
    disp, bgr, T = make_data(wl, rank, world, W + K + 1)
    bd = disp[0].dtype.itemsize
    p = params_for(wl, local_rank)
    P = Pose(p)
    # inputs resident in HBM
    d_disp = [torch.from_numpy(a).to(dev) for a in disp]
    d_bgr = [torch.from_numpy(a).to(dev) for a in bgr]
    # pinned host copies for the end-to-end leg
    # (the cycle's frames sit back to back in ONE pinned arena per plane type — a ring buffer of page-locked image slots, what
    #  o3r_host_alloc is for — so the library can move groups of adjacent planes with one 3-D copy each)
    h_disp_all = torch.from_numpy(np.stack(disp)).pin_memory()
    h_bgr_all = torch.from_numpy(np.stack(bgr)).pin_memory()
    h_disp = [h_disp_all[i] for i in range(len(disp))]
    h_bgr = [h_bgr_all[i] for i in range(len(bgr))]
    torch.cuda.synchronize()
    fr_dev = [frames_array([t.data_ptr() for t in d_disp], disp[0].strides[0], [t.data_ptr() for t in d_bgr],
                           bgr[0].strides[0], T[s]) for s in range(W + K + 1)]
    fr_host = [frames_array([t.data_ptr() for t in h_disp], disp[0].strides[0], [t.data_ptr() for t in h_bgr],
                            bgr[0].strides[0], T[s]) for s in range(W + K + 1)]
    stream = torch.cuda.ExternalStream(P.stream(), device=dev)
    ny, nx = abi.scan_dims(p)
    cell_cap = F * ny * nx
    out_pin = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()   # pinned result buffer of the e2e leg (grown if the cloud outgrows it)
    stats = {}

    if world > 1:
        # the library's own exchange (o3r_exchange_cycle: the cycle is pre-reduced on the combined grid, then grouped
        # ncclSend/ncclRecv of fixed-size slots inside libo3r.so).  Slot size: twice what one rank sends to one owner in a
        # cycle = the distinct cells of a probe cycle / world (the largest over the ranks).
        P.createCycleClouds(fr_dev[0], dt, device_pointers=True)
        probe = max(P.cloudSize(), 1)
        t = torch.tensor([probe], device=dev, dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        slot_cells = int(2 * int(t.item()) // world + 4096)
        P.clearCloud()
        box = [Pose.commUniqueId() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0, device=dev)
        P.commInit(world, rank, box[0], slot_cells)
        stats["exchange_slot_cells"] = slot_cells

    # bytes the library's copies move per step: exactly the scan ROI of every plane (groups of up to 16 adjacent frames move as
    # one 3-D copy per plane type whose extent is the ROIs)
    roi_w, roi_h = cols - p.bounding_box - p.cols_start_aft_cutout, rows - 2 * p.bounding_box
    h2d_bytes = F * roi_h * roi_w * (bd + 3)

    def exchange():
        P.exchangeCycle()

    def step(s, host):
        """One cycle (pose.cpp:361-434) + the combined downsample of the global cloud (pose.cpp:527-531 / :645).
        host=True: inputs come from pinned host memory and the combined cloud is read back to the host."""
        nonlocal out_pin
        counts = P.createCycleClouds(fr_host[s] if host else fr_dev[s], dt, device_pointers=not host)
        if world > 1:
            exchange()
        stats["counts"] = counts
        stats["n_vox"] = int(counts.sum())
        stats["n_part"] = P.lastCyclePartials()
        stats["engine"] = P.lastCycleEngine()
        if nd:   # --dont_downsample: cloud_small = cloud_big, nothing to compute; it is saved once at exit
            stats["n_out"] = 0
            return
        if host:
            try:
                out = P.downsamplePtCloud(out_pin.numpy().view(abi.POINT))
            except O3RError:   # the cloud outgrew the pinned result buffer: grow it and read again
                need = P.cloudSize() * abi.POINT.itemsize
                out_pin = torch.empty((int(need * 4) + 15) // 16 * 16, dtype=torch.uint8).pin_memory()
                out = P.downsamplePtCloud(out_pin.numpy().view(abi.POINT))
            stats["n_out"] = len(out)
        else:
            stats["out_dev"] = P.downsamplePtCloudDevice()
            stats["n_out"] = stats["out_dev"][1]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(host):
        """host=True: every timed step issues one 50-frame H2D copy from pinned host memory and one D2H read of the
        combined cloud, all inside the timed region.  The copies are pipelined one cycle ahead (o3r_frames_prefetch,
        double-buffered staging): step s starts the copy of cycle s+1, then computes cycle s, so the timed region holds
        K copies (cycles W+1 .. W+K) and K computes (cycles W .. W+K-1); the closing barrier waits for the last copy
        too, and the end-to-end time is the WALL time of the region."""
        P.clearCloud()
        if host:
            P.prefetchCycle(fr_host[0], dt)
        for s in range(W):
            if host:
                P.prefetchCycle(fr_host[s + 1], dt)
            step(s, host)
        barrier()
        l0 = P.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for s in range(W, W + K):
            if host:
                P.prefetchCycle(fr_host[s + 1], dt)
            step(s, host)
        e1.record(stream)
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms, wall], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = t.tolist()
        return ms, wall, P.launch_count() - l0

    def h2d_ceiling():
        """Plain pinned -> device copies of one step's input volume, as two halves on two streams (the library stages on two copy
        streams as well), all ranks at once: what the host link gives each GPU.  Best of 6 on one GPU, median of 6 when several
        ranks share the link."""
        nbytes = int(h2d_bytes)
        half = nbytes // 2
        src = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        src.zero_()
        dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        sa, sb = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

        def once():
            with torch.cuda.stream(sa):
                dst[:half].copy_(src[:half], non_blocking=True)
            with torch.cuda.stream(sb):
                dst[half:].copy_(src[half:], non_blocking=True)
            torch.cuda.synchronize()

        once()
        barrier()
        times = []
        for _ in range(6):
            t0 = time.perf_counter()
            once()
            times.append(time.perf_counter() - t0)
        dt_s = min(times) if world == 1 else sorted(times)[3]
        if world > 1:
            t = torch.tensor([dt_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt_s = float(t.item())
        return nbytes / dt_s / 1e9, dt_s * 1e3

    def last_step_outputs():
        """What the last step of the timed device-resident leg returned to its caller: the per-frame counts and the combined
        cloud, or with --dont_downsample (nothing is downsampled) the points the cycle appended.  The combined cloud is read
        from the context's device result buffer, valid until the next call on the context (the leg ends with nothing but a
        read of the launch counter)."""
        out = {"frame_counts": stats["counts"]}
        if nd:
            out["cycle_points"] = P.lastCyclePoints()
            return out
        ptr, n = stats["out_dev"]
        out["cloud"] = np.zeros(0, abi.POINT)
        if n:
            class DevArr:
                __cuda_array_interface__ = {"shape": (n * abi.POINT.itemsize,), "typestr": "|u1", "data": (ptr, False), "version": 2}
            out["cloud"] = torch.as_tensor(DevArr(), device=dev).cpu().numpy().view(abi.POINT)
        return out

    h2d_gbs, h2d_ms = h2d_ceiling()
    timed(host=False)  # untimed pass: every buffer reaches its steady-state size
    clocks = ClockSampler(local_rank)
    clocks.start()
    ms, wall, launches = timed(host=False)
    clk = clocks.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step_outputs(), rank, world)
    cells_after_value = P.cloudSize()
    ms_e2e_ev, ms_e2e, _ = timed(host=True)   # end to end = wall time of the region (copy stream included)
    d2h = stats["n_out"] * 16 + F * 4

    # per-kernel CUDA-event pass for the roofline
    P.clearCloud()
    for s in range(W):
        step(s, False)
    P.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    cells_before = P.cloudSize()
    for s in range(W, W + K):
        step(s, False)
    e1.record(stream)
    prof = P.profileRead()
    ms_prof = e0.elapsed_time(e1)
    P.profile(False)
    new_cells_per_step = (P.cloudSize() - cells_before) / K

    n_valid = int(sum(int((a[p.bounding_box:rows - p.bounding_box, p.cols_start_aft_cutout:cols - p.bounding_box][::J, ::J].astype(np.float64)
                           / (p.disp_divisor if dt == abi.DISP_U16 else 1.0) > p.min_disparity).sum()) for a in disp))
    # radix passes from the launches the library counted (a planned-out pass still launches and exits at once, so these are
    # upper bounds of the passes that moved data): the per-frame leaf-index sort only exists in the sort engine
    sort_launches = prof.get("k_rs_onesweep_u32", (0, 0.0))[0] / K
    engine = stats.get("engine", 0)
    np1 = 0 if engine else min(4, int(round(sort_launches)))
    np2 = max(0, int(round(sort_launches)) - np1)
    # sort engine: whether a launched pass moved data is decided on the device (k_rs_plan); only configs[1]'s plan is known
    # here (28-bit leaf index -> 4 passes, 20-bit compact cell key -> 3), so the radix kernel gets a figure on that workload only
    passes_known = bool(engine) or (v == 0.05 and rows == 720 and dt == abi.DISP_U8 and J == 1)
    alg = algorithmic_bytes(wl, n_valid, stats["n_vox"], max(new_cells_per_step, 1), bd, np1=np1, np2=np2,
                            n_part=stats.get("n_part", 0))
    if not passes_known:
        alg.pop("k_rs_onesweep_u32", None)
    peak, peak_src = peaks()
    kern = sorted(prof.items(), key=lambda kv: -kv[1][1])
    total_kernel_ms = sum(v[1] for v in prof.values())
    top_name, (top_n, top_ms) = kern[0]
    per_launch_ms = top_ms / top_n
    roof = {"bound": "hbm", "kernel": top_name, "peak": peak, "unit": "GB/s", "peak_source": peak_src,
            "launches_per_step": top_n / K, "avg_launch_ms": per_launch_ms,
            "share_of_kernel_time": top_ms / total_kernel_ms, "traffic": None}
    if top_name in alg:
        # launches that exit at once (planned-out radix passes) are included in the count: the per-launch figure
        # is total algorithmic bytes of the kernel in a step / its launches in a step
        per_launch_bytes = alg[top_name] / (top_n / K)
        roof["achieved"] = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9
        roof["frac"] = roof["achieved"] / peak
        roof["algorithmic_bytes_per_launch"] = per_launch_bytes
    else:
        roof["achieved"] = roof["frac"] = None
    roof["per_kernel_frac_of_peak"] = {k: round(alg[k] / (v[1] / K * 1e-3) / 1e9 / peak, 4) for k, v in kern if k in alg}
    # dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed ncu --set full
    # capture of this workload (profiles/), when one exists for this kernel
    roof["traffic"] = NCU_TRAFFIC.get((wl, top_name))
    roof["traffic_source"] = NCU_TRAFFIC_SOURCE if roof["traffic"] is not None else None
    # The kernel that dominates is not HBM-bound (its DRAM traffic is a few percent of what the HBM could move in its run time), so
    # the HBM fraction above says little about it.  What bounds it is instruction issue: warp instructions of one launch (committed
    # ncu capture) / (SMs x 4 schedulers x 1 instruction per clock x the SM clock measured during the timed region) = the time the
    # same instruction stream would need at 100 % issue; `frac` = that time / the launch's measured time.
    try:
        if (wl, top_name) in NCU_WARP_INST and clk.get("sm_mhz"):
            n_sm = torch.cuda.get_device_properties(local_rank).multi_processor_count
            peak_ips = n_sm * 4 * clk["sm_mhz"] * 1e6
            t_min_ms = NCU_WARP_INST[(wl, top_name)] / peak_ips * 1e3
            roof["issue_view"] = {"warp_instructions_per_launch": NCU_WARP_INST[(wl, top_name)],
                                  "source": "smsp__inst_executed.sum, " + NCU_TRAFFIC_SOURCE,
                                  "peak_warp_instructions_per_s": peak_ips, "min_launch_ms_at_full_issue": round(t_min_ms, 4),
                                  "frac": round(t_min_ms / per_launch_ms, 4),
                                  "note": "complementary to the HBM roofline above, which the contract asks for"}
    except Exception as exc:   # an optional view must never cost the line
        roof["issue_view"] = {"error": repr(exc)}
    roof["radix_passes_counted"] = {"per_frame_index_sort": np1, "combined_key_sort": np2}
    # whole-step view: compulsory bytes of the fused pipeline (SURVEY §8d) / step time
    ny, nx = abi.scan_dims(p)
    step_alg = F * (rows * cols * bd + 3 * ny * nx) + (16 * n_valid if nd else 20 * stats["n_vox"] + 2 * 32 * new_cells_per_step)
    roof["pipeline_algorithmic_bytes_per_step"] = step_alg
    roof["pipeline_frac_of_peak"] = step_alg / (ms / K * 1e-3) / 1e9 / peak
    roof["kernels_ms_per_step"] = {k: round(v[1] / K, 4) for k, v in kern[:12]}
    roof["profiled_step_ms"] = ms_prof / K

    frames_total = world * F * K
    res = {
        "metric": "frames_per_sec", "value": frames_total / (ms * 1e-3), "unit": "frames/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": {abi.DISP_U8: "u8", abi.DISP_U16: "u16", abi.DISP_F32: "f32"}[dt] + "->f64->f32",
        "data": "synthetic", "mpoints_per_sec": world * n_valid * K / (ms * 1e-3) / 1e6,
        "config": static_config(wl, world),
        "run": {"valid_points_per_step_per_gpu": n_valid, "per_frame_voxels_per_step_per_gpu": stats["n_vox"],
                "partial_cells_per_step_per_gpu": stats.get("n_part", 0),
                "merge_mode": "ACCUMULATE_" + MERGE_MODE.upper() if MERGE_MODE != "accumulate" else "ACCUMULATE",
                "engine": ENGINE_NAMES.get(stats.get("engine"), str(stats.get("engine"))),
                "resident_cells_after_timed_region": cells_after_value,
                "parallelism": f"frames f mod {world}; grouped ncclSend/ncclRecv of hash-partitioned cells inside libo3r.so" if world > 1 else "single GPU"},
        "clocks": clk, "wall_ms_per_step": wall / K,
        "e2e": {"value": frames_total / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e / K,
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h),
                "h2d_note": ("only the scan ROI of each frame crosses PCIe (x in [cols/8, cols-20), y in [20, rows-20)); the frames of a cycle "
                             "sit back to back in one pinned arena, so up to 16 adjacent planes move as one 3-D copy whose extent is exactly "
                             "their ROIs"),
                "h2d_ceiling_gbs_per_gpu": round(h2d_gbs, 2), "h2d_floor_ms_per_step": round(h2d_ms, 3),
                "h2d_ceiling_note": f"a step's input bytes as two contiguous pinned->device copies on two streams, {world} rank(s) at once, slowest rank",
                "compute_stream_ms_per_step": ms_e2e_ev / K, "timing": "wall clock around K steps incl. final sync",
                "api": "o3r_frames_prefetch(next cycle) + o3r_frames_cloud(host pinned) + o3r_cloud_downsample(host pinned)"},
        "gpu_launches": int(launches), "roofline": roof,
    }
    if world > 1:
        res["run"]["exchange_slot_cells"] = stats.get("exchange_slot_cells")
    P.close()
    if world == 1 and args.parity_steps > 0:
        res["parity"] = parity_leg(wl, local_rank, fr_dev, disp, bgr, T, args.parity_steps)
    return res, (disp, bgr, T)


def parity_leg(wl, device, fr_dev, disp, bgr, T, n_cycles):
    """After the timed regions: the first n_cycles cycles of the SAME workload through a fresh context (device-resident inputs,
    the mode that was timed) and through the CPU oracle (tests/oracle_binding.py, the checker), compared the way
    tests/test_gpu_fused.py does: per-frame voxel counts, the combined cloud's cells / order / colours exactly, centroids
    relative to where the sums live (z + 500)."""
    import oracle_binding as ob
    from online_3d_reconstruction_b200.pose import Pose
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    p = params_for(wl, device)
    threads = os.cpu_count() or 1
    keep, cloud, n, counts_equal = [], None, 0, True
    t0 = time.perf_counter()
    with Pose(p) as P:
        at = 0
        for s in range(n_cycles):
            frames = [abi.make_frame(disp[i], bgr[i], T[s][i], keep=keep) for i in range(F)]
            at = n
            cloud, n, counts = ob.run_cycle(p, frames, dt, threads, cloud, n)
            got_counts = P.createCycleClouds(fr_dev[s], dt, device_pointers=True)
            counts_equal = counts_equal and bool(np.array_equal(got_counts, counts))
        if nd:   # --dont_downsample: the cloud itself, bit for bit
            got = P.lastCyclePoints()
            exp = cloud[at:n]
        else:
            got = P.downsamplePtCloud()
            exp = ob.downsample_pt_cloud(p, cloud[:n], True)
    out = {"checked_steps": n_cycles, "frames_checked": n_cycles * F, "against": "CPU oracle (oracle/o3r_oracle.cpp), same frames",
           "per_frame_counts_equal": counts_equal, "records": int(len(got)), "records_equal": bool(len(got) == len(exp))}
    if len(got) == len(exp):
        inv = np.float32(1.0) / np.float32(v)
        out["keys_equal"] = bool(nd or all(np.array_equal(np.floor(got[f] * inv), np.floor(exp[f] * inv)) for f in ("x", "y")))
        out["colours_equal"] = bool(np.array_equal(got["rgb"], exp["rgb"]))
        rel = 0.0
        for f, shift in (("x", 0.0), ("y", 0.0), ("z", 500.0)):
            a, b = got[f].astype(np.float64) + shift, exp[f].astype(np.float64) + shift
            if len(a):
                rel = max(rel, float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-3))))
        out["max_centroid_rel"] = rel
        out["bitwise_equal"] = bool(np.array_equal(got, exp))
    # per-cell point counts are probed by tests/ through min_points_per_voxel = 1, 2, 5 (not visible in a cloud at min 1)
    out["counts_equal"] = counts_equal and out.get("colours_equal", False)
    out["seconds"] = round(time.perf_counter() - t0, 1)
    return out


CPU_PHASES = {}   # split of the last cpu_cycle call


def cpu_cycle(wl, disp, bgr, Ts, threads):
    """One step on the CPU oracle (port of the reference path): cycle + combined downsample. -> seconds"""
    import oracle_binding as ob
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    p = params_for(wl, 0)
    keep = []
    frames = [abi.make_frame(disp[i], bgr[i], Ts[i], keep=keep) for i in range(len(Ts))]
    t0 = time.perf_counter()
    cloud, n, counts = ob.run_cycle(p, frames, dt, threads)
    t1 = time.perf_counter()
    if not nd:
        ob.downsample_pt_cloud(p, cloud[:n], True)
    t2 = time.perf_counter()
    CPU_PHASES["per_frame_path_s"], CPU_PHASES["combined_downsample_s"] = t1 - t0, t2 - t1
    return t2 - t0


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path (the oracle port; the reference itself cannot be built
    here: PCL/OpenCV/Boost/VTK absent) on all host cores.  Rank 0 only."""
    if rank != 0:
        return None
    wl = args.workload
    rows, cols, dt, J, v, mp, nd, F, seed, qs = WORKLOADS[wl]
    W, K = args.warmup, args.steps
    sample_frames = min(F, args.ref_frames)
    disp, bgr, T = make_data(wl, 0, 1, W + K + 1)
    threads = os.cpu_count() or 1
    for s in range(min(W, 1)):
        cpu_cycle(wl, disp[:sample_frames], bgr[:sample_frames], T[s][:sample_frames], threads)
    t = 0.0
    for s in range(W, W + K):
        t += cpu_cycle(wl, disp[:sample_frames], bgr[:sample_frames], T[s][:sample_frames], threads)
    fps = sample_frames * K / t
    return {"impl": "reference", "metric": "frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": t / K * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8->f64->f32", "data": "synthetic",
            "config": static_config(wl, world),
            "run": {"frames_per_cpu_step": sample_frames, "note": "CPU port of the reference path (oracle/, g++ -O2; the reference "
                    "was built with no -O flag); " + ("with SOR" if wl in SOR_MEAN_K else "no SOR")},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": f"{K} cycles of {sample_frames} frames + combined downsample each"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# points of one dump over all ranks (each rank writes at most DUMP_MAX_POINTS // world): 12 B of xyz + 8 B of rgb + 8 B of
# sample index each, so a dump stays under 64 MB
DUMP_MAX_POINTS = 1_500_000


def dump_outputs(out_dir, arrays, rank=0, world=1):
    """Writes every array as <out_dir>/<name>.npy (<name>_rank<r>.npy when several ranks share the directory): counts as
    float64; a point cloud as <name>_xyz (n x 3 float32) and <name>_rgb (n float64: the whole packed 32-bit colour word,
    0x00RRGGBB).  A cloud of more than DUMP_MAX_POINTS // world points is cut to a fixed sample (seed 0, ascending, so two
    builds that agree pick the same points) whose indices go to <name>_index (float64)."""
    suffix = f"_rank{rank}" if world > 1 else ""
    max_points = DUMP_MAX_POINTS // world
    os.makedirs(out_dir, exist_ok=True)

    def save(name, a):
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)

    for name, a in arrays.items():
        if a.dtype != abi.POINT:
            save(name, a.astype(np.float64))
            continue
        if len(a) > max_points:
            idx = np.sort(np.random.default_rng(0).choice(len(a), max_points, replace=False))
            save(name + "_index", idx.astype(np.float64))
            a = a[idx]
        save(name + "_xyz", np.stack([a["x"], a["y"], a["z"]], 1).astype(np.float32))
        save(name + "_rgb", a["rgb"].astype(np.float64))


def emit(res, real_stdout):
    os.write(real_stdout, (json.dumps(res) + "\n").encode())


def main():
    # Libraries (NCCL prints its version banner) write to stdout: keep fd 1 for the ONE JSON line only.
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2_semidense_720p", choices=sorted(WORKLOADS))
    ap.add_argument("--ref-frames", type=int, default=50, help="frames per CPU-reference step (bounded sample)")
    ap.add_argument("--cpu-baseline-frames", type=int, default=50)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--merge-mode", default="fused", choices=sorted(MERGE_MODES))
    ap.add_argument("--parity-steps", type=int, default=-1,
                    help="cycles compared with the CPU oracle after the timed regions (default 2; 1 at 4K; 0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (per-frame counts, combined cloud) "
                         "as DIR/<name>.npy, to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    global MERGE_MODE
    MERGE_MODE = args.merge_mode
    if args.parity_steps < 0:
        args.parity_steps = 1 if WORKLOADS[args.workload][0] > 1000 else 2
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        res = run_reference(args, rank, world)
        if res is not None:
            emit(res, real_stdout)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    allowed = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    res, (disp, bgr, T) = run_ours(args, rank, world, local_rank)
    os.sched_setaffinity(0, allowed)
    res["run"]["host_numa_binding"] = numa
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        wl = args.workload
        n = min(len(disp), args.cpu_baseline_frames)
        threads = os.cpu_count() or 1
        cpu_cycle(wl, disp[:4], bgr[:4], T[0][:4], threads)  # warm
        t = cpu_cycle(wl, disp[:n], bgr[:n], T[args.warmup][:n], threads)
        phases = {k: round(x, 3) for k, x in CPU_PHASES.items()}
        phases["note"] = (f"per-frame path (pose.cpp:356-429) on {threads} threads; the combined downsample (pose.cpp:527-531) is one "
                          "thread, as in the reference (a single pcl::VoxelGrid call)")
        n7 = min(n, 14)   # the reference's own fan-out is 7 boost::threads per batch (pose.cpp:392-413): two batches of 7
        t7 = cpu_cycle(wl, disp[:n7], bgr[:n7], T[args.warmup][:n7], 7) if wl not in SOR_MEAN_K else None
        res["cpu_baseline"] = {"value": n / t, "unit": "frames/s", "cores": threads, "kind": "port",
                               "value_7_threads": (n7 / t7) if t7 else None, "phases": phases,
                               "sample": f"1 cycle of {n} frames + combined downsample, {t:.2f} s, " + ("with SOR" if wl in SOR_MEAN_K else "no SOR")}
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(res, real_stdout)


if __name__ == "__main__":
    main()
