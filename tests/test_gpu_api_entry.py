"""The C-ABI entry guard (host_ctx.cuh: api): every call on a context selects the context's device before anything is queued or
flushed, and returns with no device fill still queued, so a fill never waits for a later call that may find another device
current."""
import pytest

from online_3d_reconstruction_b200 import abi, lib
from online_3d_reconstruction_b200.pose import Pose
from test_gpu_parity import SMALL4, _eq, _frames

pytestmark = pytest.mark.gpu


def _params(device=0):
    return abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=1, merge_mode=abi.MERGE_ACCUMULATE,
                           device=device, **SMALL4)


@pytest.fixture
def cycles():
    keep = []
    r, c = SMALL4["rows"], SMALL4["cols"]
    yield [_frames(600, 3, r, c, keep=keep), _frames(601, 3, r, c, keep=keep, traj_start=3)]


def test_clear_launches_its_fill_before_it_returns(cycles):
    with Pose(_params()) as P:
        P.createCycleClouds(cycles[0])
        P.sync()
        n0 = P.launch_count()
        P.clearCloud()   # queues the zeroing of the resident count
        assert P.launch_count() == n0 + 1
        assert P.cloudSize() == 0
        assert P.launch_count() == n0 + 1   # nothing was left for the next call to launch


def test_comm_init_launches_its_fill_before_it_returns():
    try:
        uid = Pose.commUniqueId()
    except lib.O3RError as e:
        pytest.skip(f"NCCL cannot be loaded: {e}")
    with Pose(_params()) as P:
        n0 = P.launch_count()
        P.commInit(1, 0, uid, 1 << 16)   # queues the zeroing of the exchange flags
        assert P.launch_count() == n0 + 1
        P.commDestroy()
        assert P.launch_count() == n0 + 1


def test_contexts_on_two_devices_interleaved(cycles):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    with Pose(_params(device=1)) as R:   # the sequence on context A's device, alone
        R.createCycleClouds(cycles[0])
        R.clearCloud()
        R.createCycleClouds(cycles[1])
        expect = R.downsamplePtCloud()
    assert len(expect) > 0
    with Pose(_params(device=1)) as A, Pose(_params(device=0)) as B:
        A.createCycleClouds(cycles[0])
        A.clearCloud()
        B.createCycleClouds(cycles[0])   # leaves device 0 current
        A.createCycleClouds(cycles[1])
        got = A.downsamplePtCloud()
        assert len(B.downsamplePtCloud()) > 0
    _eq(got, expect)
