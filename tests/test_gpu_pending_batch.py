"""The last batch is what the last frame-path call (o3r_frame_cloud / o3r_frames_cloud[_dev]) produced: the stand-alone calls
o3r_voxel_grid, o3r_sor and an accumulate-mode o3r_cloud_append stage their data in buffers of their own, so
o3r_last_batch_* and a pending o3r_exchange_cycle still see the batch that came before them."""
import numpy as np
import pytest

from online_3d_reconstruction_b200 import abi
from online_3d_reconstruction_b200.pose import Pose
from test_gpu_parity import SMALL4, _eq, _frames

pytestmark = pytest.mark.gpu
MODES = [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_FUSED]
CALLS = ["voxelGrid", "statisticalOutlierRemoval", "appendPoints"]
R, W = SMALL4["rows"], SMALL4["cols"]


@pytest.fixture(scope="module")
def keep():
    return []   # host buffers the frames point into


@pytest.fixture(scope="module")
def cycles(keep):
    return [_frames(900 + c, 3, R, W, keep=keep, traj_start=3 * c) for c in range(2)]


@pytest.fixture(scope="module")
def cloud(keep):
    """a host cloud in the scene of the cycles (one frame's points), the input of the stand-alone calls"""
    with Pose(_params(abi.MERGE_ACCUMULATE)) as P:
        pts = P.createAndTransformPtCloud(_frames(950, 1, R, W, keep=keep, traj_start=1)[0])
    assert pts.size > 1000
    return pts


def _params(mode):
    return abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=1, merge_mode=mode, **SMALL4)


def _call(P, name, pts):
    if name == "voxelGrid":
        P.voxelGrid(pts, (0.02, 0.02, 0.02))
    elif name == "statisticalOutlierRemoval":
        P.statisticalOutlierRemoval(pts, mean_k=8)
    else:
        P.appendPoints(pts)


def _same_cells(got, exp):
    assert got.shape == exp.shape, (got.shape, exp.shape)
    for f in got.dtype.names:
        assert np.array_equal(got[f].view(np.uint32) if got[f].dtype == np.float32 else got[f],
                              exp[f].view(np.uint32) if exp[f].dtype == np.float32 else exp[f]), f


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", CALLS)
def test_stand_alone_call_leaves_the_last_batch(mode, name, cycles, cloud):
    with Pose(_params(mode)) as P:
        if mode == abi.MERGE_ACCUMULATE_FUSED:
            P.setKeepFrameVoxels(True)
        P.createCycleClouds(cycles[0])
        pts, part, eng = P.lastCyclePoints(), P.lastCyclePartials(), P.lastCycleEngine()
        assert pts.size > 0
        _call(P, name, cloud)
        _eq(P.lastCyclePoints(), pts)
        assert P.lastCyclePartials() == part
        assert P.lastCycleEngine() == eng


def _exchanged(mode, cycles, between=None, before=None):
    """cycle 0 -> exchange; [before] -> cycle 1 -> [between] -> exchange, on a world-1 communicator -> exported cells"""
    with Pose(_params(mode)) as P:
        P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        P.createCycleClouds(cycles[0])
        P.exchangeCycle()
        if before:
            before(P)
        P.createCycleClouds(cycles[1])
        if between:
            between(P)
        P.exchangeCycle()
        return P.exportCells()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", CALLS[:2])
def test_stand_alone_call_between_cycle_and_exchange_changes_nothing(mode, name, cycles, cloud):
    plain = _exchanged(mode, cycles)
    assert plain.size > 0
    _same_cells(_exchanged(mode, cycles, between=lambda P: _call(P, name, cloud)), plain)


@pytest.mark.parametrize("mode", MODES)
def test_append_between_cycle_and_exchange_merges_both(mode, cycles, cloud):
    # both orders merge the appended points first (o3r_cloud_append merges at once), then the exchanged cycle
    first = _exchanged(mode, cycles, before=lambda P: P.appendPoints(cloud))
    assert first.size > 0
    _same_cells(_exchanged(mode, cycles, between=lambda P: P.appendPoints(cloud)), first)
