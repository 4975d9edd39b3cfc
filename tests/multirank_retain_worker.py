"""Worker of tests/test_gpu_multirank_retain.py: one process per GPU under torch.distributed.run.

Sharded RETAIN (ICP-on) mode: every rank reconstructs the frames f with f mod world == rank and keeps their points, all
ranks apply the same tf_icp between cycles (o3r_cloud_transform stays local), and o3r_cloud_downsample is the collective
that moves each point to the owner of its combined-grid cell.  Rank 0 checks the shards against the single-rank RETAIN
cloud and the CPU oracle bit for bit.  gloo is only the host channel for the NCCL id and for collecting the shards."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import oracle_binding as ob  # noqa: E402
from online_3d_reconstruction_b200 import abi, exchange, synth  # noqa: E402
from online_3d_reconstruction_b200.pose import Pose  # noqa: E402


def keys_of(a, voxel):
    sh = a.copy()
    sh["z"] += np.float32(500)
    leaf = (voxel, voxel, 1000.0)
    return np.array([ob.cell_key(q["x"], q["y"], q["z"], leaf) for q in sh], dtype=np.uint64)


def tf_icp():
    tf = np.eye(4, dtype=np.float32)
    c, s = np.float32(np.cos(0.01)), np.float32(np.sin(0.01))
    tf[0, 0], tf[0, 1], tf[1, 0], tf[1, 1] = c, -s, s, c
    tf[:3, 3] = [0.03, -0.02, 0.01]
    return tf


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("gloo")
    torch.cuda.set_device(local)
    rows, cols = 128, 256
    per_cycle = [5, 3, 1]   # the last cycle leaves every rank but rank 0 without a frame (n = 0 calls)
    keep = []
    seq = synth.sequence(4343, sum(per_cycle), rows, cols)
    frames = [abi.make_frame(d, img, T, keep=keep) for d, img, T in seq]
    cycles, at = [], 0
    for n in per_cycle:
        cycles.append(frames[at:at + n])
        at += n
    tf = tf_icp()
    cases = [("retain", dict(voxel_size=0.05, min_points_per_voxel=1)), ("retain", dict(voxel_size=0.05, min_points_per_voxel=3)),
             ("passthrough", dict(voxel_size=2e-5, min_points_per_voxel=1)), ("dont_downsample", dict(dont_downsample=True))]
    for kind, kw in cases:
        p = abi.make_params(rows=rows, cols=cols, jump_pixels=1, merge_mode=abi.MERGE_RETAIN, device=local, **kw)
        box = [Pose.commUniqueId() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        counts = []
        with Pose(p) as P:
            P.commInit(world, rank, box[0], 1 << 16)
            for s, cyc in enumerate(cycles):
                if s:
                    P.transformPtCloud(tf)
                counts.append(P.createCycleClouds(cyc[rank::world]))
                P.exchangeCycle()   # a no-op in RETAIN mode: one driver loop serves every mode
            shard = P.downsamplePtCloud()
            again = P.downsamplePtCloud()   # unchanged cloud: the kept result, no communication
            assert np.array_equal(shard, again)
            P.commDestroy()
        got = [None] * world
        dist.gather_object((shard, counts), got if rank == 0 else None, dst=0)
        if rank == 0:
            shards = [g[0] for g in got]
            with Pose(p) as S:
                for s, cyc in enumerate(cycles):
                    if s:
                        S.transformPtCloud(tf)
                    S.createCycleClouds(cyc)
                single = S.downsamplePtCloud()
            cloud, n = None, 0
            for s, cyc in enumerate(cycles):
                if s:
                    cloud[:n] = ob.transform_pt_cloud(cloud[:n], tf)
                cloud, n, _ = ob.run_cycle(p, cyc, abi.DISP_U8, 4, cloud, n)
            exp = cloud[:n] if p.dont_downsample else ob.downsample_pt_cloud(p, cloud[:n], True)   # (pose.cpp:535)
            if kind != "passthrough":   # (on a pass-through grid the single-GPU path returns the points as stored, the oracle
                assert np.array_equal(single, exp), "single-rank RETAIN differs from the oracle"   # after its z + 500 - 500)
            assert len(single) == len(exp)
            if kind == "retain":
                union = np.concatenate(shards)
                ku = keys_of(union, p.voxel_size)
                assert np.array_equal(exchange.owner_of(ku, world), np.repeat(np.arange(world), [len(s) for s in shards])), \
                    "a cell sits on a rank the owner hash does not name"
                order = np.argsort(ku, kind="stable")
                union, ku = union[order], ku[order]
                assert len(np.unique(ku)) == len(ku), "ownership is not disjoint"
                for f in ("x", "y", "z", "rgb"):
                    assert np.array_equal(union[f].view(np.uint32), single[f].view(np.uint32)), f
                assert min(len(s) for s in shards) > 0.3 * len(single) / world
            else:   # every rank returns its own points: interleaved back into frame order they are the single-rank output
                merged = exchange.unshard_points(shards, [g[1] for g in got], world)
                assert np.array_equal(merged.view(np.uint32), single.view(np.uint32)), "unsharded points differ"
            print(f"{kind} {kw}: {world} ranks, shards {[len(s) for s in shards]} == single {len(single)}", flush=True)
        dist.barrier()
    if rank == 0:
        print("MULTIRANK RETAIN OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
