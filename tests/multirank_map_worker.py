"""Worker of tests/test_gpu_multirank_map.py: one process per GPU under torch.distributed.run.

Each rank builds its shard of the map through the library's exchange, checkpoints it after two of three cycles and at the
end.  Checked: the union of the ranks' exports, imported into one single-GPU context, downsamples to the union of the
ranks' downsamples bit for bit; a rank refuses a cell another rank owns; and every rank that reloads its own checkpoint
into a new communicator and runs the last cycle ends bit for bit where the uninterrupted run ended."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from online_3d_reconstruction_b200 import abi, exchange, lib, synth  # noqa: E402
from online_3d_reconstruction_b200.pose import Pose  # noqa: E402


def uid(rank):
    box = [Pose.commUniqueId() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("gloo")
    torch.cuda.set_device(local)
    rows, cols, min_pts = 128, 256, 2
    n_cycles, per_cycle = 3, 6
    for mode in (abi.MERGE_ACCUMULATE_FUSED, abi.MERGE_ACCUMULATE):
        keep = []
        seq = synth.sequence(5151, n_cycles * per_cycle, rows, cols)
        frames = [abi.make_frame(d, img, T, keep=keep) for d, img, T in seq]
        cycles = [frames[c * per_cycle:(c + 1) * per_cycle] for c in range(n_cycles)]
        p = abi.make_params(rows=rows, cols=cols, jump_pixels=1, voxel_size=0.05, min_points_per_voxel=min_pts,
                            merge_mode=mode, device=local)
        with Pose(p) as P:
            P.commInit(world, rank, uid(rank), 1 << 16)
            for i, cyc in enumerate(cycles):
                P.createCycleClouds(cyc[rank::world])
                P.exchangeCycle()
                if i == n_cycles - 2:
                    mid = P.exportCells()
            cells, ds = P.exportCells(), P.downsamplePtCloud()
            assert np.all(exchange.owner_of(cells["key"], world) == rank)
            # a cell of another rank's shard is refused, and the shard stays as it was
            mids = [None] * world
            dist.all_gather_object(mids, mid)
            foreign = mids[(rank + 1) % world][:1]
            try:
                P.importCells(foreign)
                raise AssertionError("a cell owned by another rank was imported")
            except lib.O3RError as e:
                assert e.code == abi.O3R_ERR_INVALID and "another rank" in str(e), str(e)
            assert P.exportCells().tobytes() == cells.tobytes()
            P.commDestroy()
        # every rank reloads its own shard into a new communicator of the same size and runs the last cycle
        with Pose(p) as Q:
            Q.commInit(world, rank, uid(rank), 1 << 16)
            Q.importCells(mid)
            Q.createCycleClouds(cycles[-1][rank::world])
            Q.exchangeCycle()
            assert Q.exportCells().tobytes() == cells.tobytes(), "the resumed shard differs"
            assert Q.downsamplePtCloud().tobytes() == ds.tobytes()
            Q.commDestroy()
        gathered = [None] * world
        dist.gather_object((cells, ds), gathered if rank == 0 else None, dst=0)
        if rank == 0:
            union_cells = np.concatenate([g[0] for g in gathered])
            keys = np.concatenate([g[0]["key"][g[0]["n"] >= min_pts] for g in gathered])
            union_ds = np.concatenate([g[1] for g in gathered])[np.argsort(keys, kind="stable")]
            with Pose(p) as S:
                S.importCells(union_cells)
                single = S.downsamplePtCloud()
            assert single.tobytes() == union_ds.tobytes(), "the single-GPU import differs from the union of the shards"
            print(f"mode {mode}: {world} ranks, shards {[len(g[0]) for g in gathered]} cells, union reloads on one GPU",
                  flush=True)
        dist.barrier()
    if rank == 0:
        print("MULTIRANK MAP OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
