"""Launches and kernel time of one steady-state fused cycle of bench.py's default workload (configs[1]: 720p u8, 50 frames,
O3R_MERGE_ACCUMULATE_FUSED, device-resident inputs), step as bench.py times it: o3r_frames_cloud_dev + the combined
downsample.  Prints launch_count() per cycle, then every kernel name with its launches and CUDA-event ms per cycle (the
profile pass; its events serialise the launches, so its times are an upper bound of what the kernels take in a timed step).

    python profiles/scripts/cycle_launches.py [--steps K] [--warmup W] [--workload NAME] [--json OUT]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload tables and the frame set-up bench.py times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="config2_semidense_720p")
    ap.add_argument("--json", metavar="OUT", help="also write the result as JSON")
    args = ap.parse_args()

    import torch
    from online_3d_reconstruction_b200.pose import Pose

    wl, W, K = args.workload, args.warmup, args.steps
    rows, cols, dt, J, v, mp, nd, F, seed, qs = bench.WORKLOADS[wl]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    disp, bgr, T = bench.make_data(wl, 0, 1, W + K)
    d_disp = [torch.from_numpy(a).to(dev) for a in disp]
    d_bgr = [torch.from_numpy(a).to(dev) for a in bgr]
    torch.cuda.synchronize()
    fr = [bench.frames_array([t.data_ptr() for t in d_disp], disp[0].strides[0], [t.data_ptr() for t in d_bgr],
                             bgr[0].strides[0], T[s]) for s in range(W + K)]
    P = Pose(bench.params_for(wl, 0))

    def step(s):
        P.createCycleClouds(fr[s], dt, device_pointers=True)
        if not nd:
            P.downsamplePtCloudDevice()

    def cycles(profile):
        P.clearCloud()
        for s in range(W):
            step(s)
        P.sync()
        per = []
        if profile:
            P.profile(True)
        for s in range(W, W + K):
            l0 = P.launch_count()
            step(s)
            per.append(P.launch_count() - l0)
        prof = P.profileRead() if profile else {}
        if profile:
            P.profile(False)
        return per, prof

    cycles(False)   # every buffer reaches its steady-state size
    per, _ = cycles(False)
    _, prof = cycles(True)
    kern = sorted(prof.items(), key=lambda kv: -kv[1][1])
    out = {"workload": wl, "steps": K, "warmup": W, "engine": P.lastCycleEngine(),
           "device": torch.cuda.get_device_name(0),
           "launch_count_per_cycle": per, "launches_per_cycle_max": max(per),
           "kernels": {k: {"launches_per_cycle": n / K, "ms_per_cycle": round(ms / K, 4)} for k, (n, ms) in kern},
           "kernel_ms_per_cycle": round(sum(ms for _, ms in prof.values()) / K, 4)}
    print(f"{wl}: engine {out['engine']}, launch_count() per steady-state cycle {sorted(set(per))} "
          f"(max {out['launches_per_cycle_max']}), profiled kernel time {out['kernel_ms_per_cycle']:.4f} ms per cycle")
    print(f"{'kernel':28s} {'launches':>9s} {'ms':>8s}")
    for k, (n, ms) in kern:
        print(f"{k:28s} {n / K:9.2f} {ms / K:8.4f}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)
    P.close()


if __name__ == "__main__":
    main()
