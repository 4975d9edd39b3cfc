"""Multi-GPU equivalence on REAL ranks (SURVEY 8e): N processes, N GPUs, the library's own NCCL exchange
(o3r_exchange_cycle), union of the shards == the single-rank cloud == the oracle's cells.  Needs >= 2 devices; the
single-device test below drives the same exchange path at world size 1."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi
from online_3d_reconstruction_b200.pose import Pose
from test_gpu_parity import SMALL4, _close, _eq, _frames

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 4])
def test_n_ranks_equal_one_rank_through_the_library_exchange(world):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multirank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MULTIRANK OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE_FUSED, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE])
def test_exchange_cycle_world_1_equals_the_plain_merge(mode):
    """The library exchange at world size 1 (own communicator, the slot goes to the rank itself): same cells, counts and
    colours as the direct merge, centroids within 1e-5; bit-identical from run to run.  After commDestroy the context
    merges its cycles itself again: the last cycle runs without an exchange and still reaches the cloud."""
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=2, merge_mode=mode, **geom)
    cycles = [_frames(500, 5, geom["rows"], geom["cols"], keep=keep), _frames(501, 5, geom["rows"], geom["cols"], keep=keep, traj_start=5),
              _frames(503, 5, geom["rows"], geom["cols"], keep=keep, traj_start=10)]
    with Pose(p) as S:
        for c in cycles:
            S.createCycleClouds(c)
        plain = S.downsamplePtCloud()
    outs = []
    for _ in range(2):
        with Pose(p) as P:
            P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
            for c in cycles[:2]:
                P.createCycleClouds(c)
                P.exchangeCycle()
            P.commDestroy()
            P.createCycleClouds(cycles[2])
            outs.append(P.downsamplePtCloud())
    _eq(outs[0], outs[1])
    _close(outs[0], plain)


def test_exchange_slot_overflow_is_reported():
    from online_3d_reconstruction_b200.lib import O3RError
    keep = []
    geom = SMALL4
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, merge_mode=abi.MERGE_ACCUMULATE_FUSED, **geom)
    with Pose(p) as P:
        P.commInit(1, 0, Pose.commUniqueId(), 16)   # far too small a slot
        P.createCycleClouds(_frames(502, 3, geom["rows"], geom["cols"], keep=keep))
        P.exchangeCycle()
        with pytest.raises(O3RError):
            P.downsamplePtCloud()
