"""Sharded RETAIN (ICP-on) mode at world size 1: a communicator of one rank runs the collective downsample's plumbing on one
device (bbox all-reduce, counts and buffer agreements, the copy to itself, the tag sort, engine 1 on the global grid, the kept
result).  Its output must be the plain RETAIN output bit for bit, centroids included, and the CPU oracle's one-shot
voxelisation.  At world 1 every point's owner is rank 0 and the records already arrive in tag order, so a wrong owner hash, a
wrong global frame index in the tag or a mis-ordered merge of several sources cannot show here: tests/test_gpu_multirank_retain.py
(2 and 4 ranks) covers those."""
import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi
from online_3d_reconstruction_b200.lib import O3RError
from online_3d_reconstruction_b200.pose import Pose
from test_gpu_parity import SMALL4, _eq, _frames

pytestmark = pytest.mark.gpu


def _tf_icp(angle=0.01, t=(0.03, -0.02, 0.01)):
    tf = np.eye(4, dtype=np.float32)
    c, s = np.float32(np.cos(angle)), np.float32(np.sin(angle))
    tf[0, 0], tf[0, 1], tf[1, 0], tf[1, 1] = c, -s, s, c
    tf[:3, 3] = t
    return tf


@pytest.fixture(scope="module")
def cycles():
    keep = []
    g = SMALL4
    out = [_frames(700, 4, g["rows"], g["cols"], keep=keep), _frames(701, 3, g["rows"], g["cols"], keep=keep, traj_start=4),
           _frames(702, 4, g["rows"], g["cols"], keep=keep, traj_start=7)]
    yield out
    del keep


def _params(**kw):
    kw.setdefault("voxel_size", 0.05)
    return abi.make_params(jump_pixels=1, merge_mode=abi.MERGE_RETAIN, **SMALL4, **kw)


def _run(p, cycles, tf, world1=False):
    """Cycles with transformPtCloud(tf) between them (pose.cpp:350-354), then the combined downsample."""
    with Pose(p) as P:
        if world1:
            P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        for i, c in enumerate(cycles):
            if i:
                P.transformPtCloud(tf)
            P.createCycleClouds(c)
        return P.downsamplePtCloud()


def _oracle(p, cycles, tf):
    cloud, n = None, 0
    for i, c in enumerate(cycles):
        if i:
            cloud[:n] = ob.transform_pt_cloud(cloud[:n], tf)
        cloud, n, _ = ob.run_cycle(p, c, abi.DISP_U8, 4, cloud, n)
    return cloud[:n]


@pytest.mark.parametrize("min_pts", [1, 3])
def test_sharded_retain_world_1_is_bit_identical(cycles, min_pts):
    p = _params(min_points_per_voxel=min_pts)
    tf = _tf_icp()
    plain = _run(p, cycles, tf)
    exp = ob.downsample_pt_cloud(p, _oracle(p, cycles, tf), True)
    a = _run(p, cycles, tf, world1=True)
    b = _run(p, cycles, tf, world1=True)
    assert len(exp) > 100
    _eq(a, plain)
    _eq(a, exp)
    _eq(a, b)


def test_query_then_fill_and_a_later_cycle(cycles):
    p = _params()
    tf = _tf_icp()
    with Pose(p) as S:
        S.createCycleClouds(cycles[0])
        plain0 = S.downsamplePtCloud()
        S.transformPtCloud(tf)
        S.createCycleClouds(cycles[1])
        plain1 = S.downsamplePtCloud()
    with Pose(p) as P:
        P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        P.createCycleClouds(cycles[0])
        first = P.downsamplePtCloud()              # size query (cap 0), then the fill: one collective
        again = P.downsamplePtCloud()              # unchanged cloud: the kept result
        ptr, n = P.downsamplePtCloudDevice()
        assert ptr and n == len(first)
        P.transformPtCloud(tf)
        P.createCycleClouds(cycles[1])
        later = P.downsamplePtCloud()
    _eq(first, plain0)
    _eq(again, plain0)
    _eq(later, plain1)


@pytest.mark.parametrize("kind", ["passthrough", "dont_downsample"])
def test_passthrough_grid_and_dont_downsample_equal_the_plain_context(cycles, kind):
    p = _params(voxel_size=2e-5) if kind == "passthrough" else _params(dont_downsample=True)
    tf = _tf_icp()
    plain = _run(p, cycles, tf)
    got = _run(p, cycles, tf, world1=True)
    if kind == "passthrough":   # PCL's int32 guard tripped on the combined grid: every point comes back, one per record
        assert len(got) == len(_oracle(p, cycles, tf))
    assert len(got) > 1000
    _eq(got, plain)


def test_empty_cycle_append_exchange_destroy_and_init_rules(cycles):
    p = _params()
    tf = _tf_icp()
    plain = _run(p, cycles[:2], tf)
    with Pose(p) as P:
        P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        P.createCycleClouds(cycles[0])
        P.exchangeCycle()                          # a no-op in RETAIN mode
        n0 = P.cloudSize()
        assert len(P.createCycleClouds([])) == 0   # n = 0: a cycle without frames on this rank
        assert P.cloudSize() == n0
        P.transformPtCloud(tf)
        P.createCycleClouds(cycles[1])
        P.exchangeCycle()
        with pytest.raises(O3RError):
            P.appendPoints(np.zeros(4, dtype=abi.POINT))
        _eq(P.downsamplePtCloud(), plain)
        P.commDestroy()                            # local again: the same cloud, downsampled by the single-GPU path
        _eq(P.downsamplePtCloud(), plain)
        P.transformPtCloud(tf)
        P.createCycleClouds(cycles[2])
        local = P.downsamplePtCloud()
    _eq(local, _run(p, cycles, tf))
    with Pose(p) as P:
        P.createCycleClouds(cycles[0])
        with pytest.raises(O3RError):
            P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)   # a sharded retained cloud starts empty
        P.clearCloud()
        P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        P.createCycleClouds(cycles[0])
        _eq(P.downsamplePtCloud(), _run(p, cycles[:1], tf))
