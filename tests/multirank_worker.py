"""Worker of tests/test_gpu_multirank.py: one process per GPU under torch.distributed.run.

Every rank reconstructs the frames f with f mod world == rank, calls the library's own exchange (o3r_exchange_cycle: NCCL
grouped send/recv inside libo3r.so) after each cycle, and rank 0 checks the union of the shards against the single-rank
result and against the CPU oracle.  gloo is only the host channel for the NCCL id and for collecting the shards."""
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


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("gloo")
    torch.cuda.set_device(local)
    rows, cols, voxel = 128, 256, 0.05
    n_cycles, per_cycle = 3, 6
    for mode in (abi.MERGE_ACCUMULATE_FUSED, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE):
        keep = []
        seq = synth.sequence(4242, n_cycles * per_cycle, rows, cols)
        frames = [abi.make_frame(d, img, T, keep=keep) for d, img, T in seq]
        cycles = [frames[c * per_cycle:(c + 1) * per_cycle] for c in range(n_cycles)]
        p = abi.make_params(rows=rows, cols=cols, jump_pixels=1, voxel_size=voxel, min_points_per_voxel=1, merge_mode=mode,
                            device=local)
        box = [Pose.commUniqueId() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        with Pose(p) as P:
            P.commInit(world, rank, box[0], 1 << 16)
            for cyc in cycles:
                P.createCycleClouds(cyc[rank::world])
                P.exchangeCycle()
            shard = P.downsamplePtCloud()
            P.commDestroy()
        shards = [None] * world
        dist.gather_object(shard, shards if rank == 0 else None, dst=0)
        if rank == 0:
            with Pose(p) as S:
                for cyc in cycles:
                    S.createCycleClouds(cyc)
                single = S.downsamplePtCloud()
            union = np.concatenate(shards)
            ku, ks = keys_of(union, voxel), keys_of(single, voxel)
            # every rank holds exactly the cells the host mirror of the device's owner hash assigns to it
            assert np.array_equal(exchange.owner_of(ku, world), np.repeat(np.arange(world), [len(s) for s in shards])), \
                "a cell sits on a rank the owner hash does not name"
            order = np.argsort(ku, kind="stable")
            union, ku = union[order], ku[order]
            assert len(np.unique(ku)) == len(ku), "ownership is not disjoint"
            assert np.array_equal(ku, ks), "cell sets differ"
            assert np.array_equal(union["rgb"], single["rgb"]), "colours differ"
            for f, sh in (("x", 0.0), ("y", 0.0), ("z", 500.0)):
                a, b = union[f].astype(np.float64) + sh, single[f].astype(np.float64) + sh
                assert np.all(np.abs(a - b) <= 1e-5 * np.maximum(np.abs(b), 1e-3)), f
            assert min(len(s) for s in shards) > 0.3 * len(single) / world
            # and against the oracle's one-shot voxelisation of everything (pose.cpp:527-531)
            cloud, n = None, 0
            for cyc in cycles:
                cloud, n, _ = ob.run_cycle(p, cyc, abi.DISP_U8, 4, cloud, n)
            exp = ob.downsample_pt_cloud(p, cloud[:n], True)
            assert np.array_equal(keys_of(exp, voxel), ku) and np.array_equal(exp["rgb"], union["rgb"])
            print(f"mode {mode}: {world} ranks, shards {[len(s) for s in shards]} == single {len(single)} cells", flush=True)
        dist.barrier()
    if rank == 0:
        print("MULTIRANK OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
