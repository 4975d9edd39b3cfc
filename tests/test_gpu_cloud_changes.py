"""Change tracking of the resident cloud (o3r_cloud_track_changes / o3r_cloud_changes[_dev]): a consumer that upserts the
changed records by key holds exactly what o3r_cloud_downsample returns, and the changes are exactly the cells whose point
count grew since the last read."""
import ctypes as C

import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi, lib, synth
from online_3d_reconstruction_b200.pose import Pose
from test_gpu_parity import SMALL4, _eq, _frames

pytestmark = pytest.mark.gpu

ACC_MODES = [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE_FUSED]
#: launches one merged cycle adds while tracking is on (DESIGN.md: k_chg_part, k_chg_union_cnt, k_scan_u32, k_chg_union)
CHG_LAUNCHES_PER_CYCLE = 4


class KeyMap:
    """The consumer's copy of the combined grid: records upserted by cell key, read back in key order."""

    def __init__(self):
        self.k = np.zeros(0, np.uint64)
        self.p = np.zeros(0, abi.POINT)

    def upsert(self, pts, keys):
        assert np.all(np.diff(keys.astype(np.int64)) > 0), "keys of one result must be strictly ascending"
        k = np.concatenate([keys, self.k])
        p = np.concatenate([pts, self.p])
        self.k, first = np.unique(k, return_index=True)   # first occurrence = the new record
        self.p = p[first]

    def points(self):
        return self.p


def _cycles(seed, geom=SMALL4, keep=None):
    """>= 4 cycles: two ordinary ones, an empty one (n = 0), another, and one frame that revisits the trajectory's start."""
    r, c = geom["rows"], geom["cols"]
    return [_frames(seed, 4, r, c, keep=keep, traj_start=0), _frames(seed + 1, 3, r, c, keep=keep, traj_start=4), [],
            _frames(seed + 2, 4, r, c, keep=keep, traj_start=6), _frames(seed + 3, 1, r, c, keep=keep, traj_start=0)]


def _params(mode, min_pts, geom=SMALL4, **kw):
    return abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=min_pts, merge_mode=mode, **geom, **kw)


def _oracle_clouds(p, cycles):
    """cloud_big after every cycle (the reference's order)."""
    cloud, n, out = None, 0, []
    for frames in cycles:
        if frames:
            cloud, n, _ = ob.run_cycle(p, frames, abi.DISP_U8, 4, cloud, n)
        out.append(cloud[:n].copy() if cloud is not None else np.zeros(0, abi.POINT))
    return out


def _cell_counts(big, v):
    """{absolute cell key: points} of cloud_big on the combined grid (z + 500, leaf (v, v, 1000), min_points 0)."""
    if len(big) == 0:
        return {}
    sh = big.copy()
    sh["z"] = sh["z"] + np.float32(500.0)
    _, keys, counts, pt = ob.voxel_grid(sh, (v, v, 1000.0), 0)
    assert not pt
    return dict(zip(keys.tolist(), counts.tolist()))


def _grown(before, after, min_pts):
    return sorted(k for k, c in after.items() if c > before.get(k, 0) and c >= min_pts)


def _full(after, min_pts):
    return sorted(k for k, c in after.items() if c >= min_pts)


@pytest.mark.parametrize("mode", ACC_MODES)
@pytest.mark.parametrize("min_pts", [1, 3])
def test_upserted_changes_equal_downsample_every_cycle(mode, min_pts):
    keep = []
    with Pose(_params(mode, min_pts)) as P:
        P.trackCloudChanges(True)
        m = KeyMap()
        for frames in _cycles(200, keep=keep):
            P.createCycleClouds(frames)
            pts, keys, counts = P.cloudChanges()
            assert np.all(counts >= min_pts)
            m.upsert(pts, keys)
            _eq(m.points(), P.downsamplePtCloud())
        assert len(m.points()) > 100


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_FUSED])
@pytest.mark.parametrize("min_pts", [1, 3])
def test_changes_are_exactly_the_grown_cells(mode, min_pts):
    keep = []
    p = _params(mode, min_pts)
    cycles = _cycles(210, keep=keep)
    bigs = _oracle_clouds(p, cycles)
    with Pose(p) as P:
        P.trackCloudChanges(True)
        before = {}
        for i, frames in enumerate(cycles):
            P.createCycleClouds(frames)
            after = _cell_counts(bigs[i], 0.05)
            pts, keys, counts = P.cloudChanges()
            if i == 0:   # the key formats agree: the first result (the full state) has the oracle's keys
                assert keys.tolist() == _full(after, min_pts)
            exp = _grown(before, after, min_pts)
            assert keys.tolist() == exp, f"cycle {i}"
            assert counts.tolist() == [after[k] for k in exp]
            if not frames:
                assert len(keys) == 0
            before = after


def test_polling_every_third_cycle_returns_the_union():
    keep = []
    p = _params(abi.MERGE_ACCUMULATE, 2)
    r, c = SMALL4["rows"], SMALL4["cols"]
    cycles = [_frames(220 + i, 2, r, c, keep=keep, traj_start=2 * i) for i in range(6)]
    bigs = _oracle_clouds(p, cycles)
    with Pose(p) as A, Pose(p) as B:
        A.trackCloudChanges(True)
        B.trackCloudChanges(True)
        ma, mb = KeyMap(), KeyMap()
        before = {}
        for i, frames in enumerate(cycles):
            A.createCycleClouds(frames)
            B.createCycleClouds(frames)
            pa, ka, _ = A.cloudChanges()
            ma.upsert(pa, ka)
            if i % 3 == 2:
                after = _cell_counts(bigs[i], 0.05)
                pb, kb, cb = B.cloudChanges()
                if i > 2:   # (the first read of B is the full state)
                    assert kb.tolist() == _grown(before, after, 2)
                    assert cb.tolist() == [after[k] for k in kb.tolist()]
                mb.upsert(pb, kb)
                before = after
        _eq(ma.points(), mb.points())
        _eq(ma.points(), A.downsamplePtCloud())


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_FUSED])
def test_enable_on_non_empty_cloud_and_reenable_give_full_state(mode):
    keep = []
    p = _params(mode, 2)
    cycles = _cycles(230, keep=keep)
    bigs = _oracle_clouds(p, cycles)
    with Pose(p) as P:
        P.createCycleClouds(cycles[0])
        P.createCycleClouds(cycles[1])
        P.trackCloudChanges(True)
        pts, keys, _ = P.cloudChanges()
        assert keys.tolist() == _full(_cell_counts(bigs[1], 0.05), 2)
        _eq(pts, P.downsamplePtCloud())
        P.createCycleClouds(cycles[3])
        after = _cell_counts(bigs[3], 0.05)
        _, keys, _ = P.cloudChanges()
        assert keys.tolist() == _grown(_cell_counts(bigs[1], 0.05), after, 2)
        P.createCycleClouds(cycles[4])
        P.trackCloudChanges(True)   # re-enable: the pending cycle is folded into the full state
        pts, keys, _ = P.cloudChanges()
        assert keys.tolist() == _full(_cell_counts(bigs[4], 0.05), 2)
        _eq(pts, P.downsamplePtCloud())
        assert len(P.cloudChanges()[0]) == 0


def test_query_then_fill_semantics():
    keep = []
    L = lib.load()
    cycles = _cycles(240, keep=keep)
    with Pose(_params(abi.MERGE_ACCUMULATE, 1)) as P:
        P.trackCloudChanges(True)
        P.createCycleClouds(cycles[0])
        _ = P.cloudChanges()
        P.createCycleClouds(cycles[1])
        n1, n2 = C.c_size_t(0), C.c_size_t(0)
        assert L.o3r_cloud_changes(P.handle, None, None, None, 0, C.byref(n1)) == 0
        assert L.o3r_cloud_changes(P.handle, None, None, None, 0, C.byref(n2)) == 0
        assert n1.value == n2.value > 0
        small = np.empty(n1.value - 1, abi.POINT)
        nc = C.c_size_t(0)
        assert L.o3r_cloud_changes(P.handle, small.ctypes.data, None, None, small.size, C.byref(nc)) == -3
        assert nc.value == n1.value
        pts, keys, counts = P.cloudChanges()   # nothing was consumed: the same set
        assert len(pts) == n1.value
        assert L.o3r_cloud_changes(P.handle, None, None, None, 0, C.byref(nc)) == 0 and nc.value == 0
        # a cycle between the query and the fill: the fill returns the grown set
        P.createCycleClouds(cycles[3])
        assert L.o3r_cloud_changes(P.handle, None, None, None, 0, C.byref(n1)) == 0
        P.createCycleClouds(cycles[4])
        with Pose(_params(abi.MERGE_ACCUMULATE, 1)) as Q:   # twin: the union of both cycles in one read
            Q.createCycleClouds(cycles[0]); Q.createCycleClouds(cycles[1])
            Q.trackCloudChanges(True); Q.cloudChanges()
            Q.createCycleClouds(cycles[3]); Q.createCycleClouds(cycles[4])
            _, exp_keys, _ = Q.cloudChanges()
        cap = max(1, len(exp_keys))
        out, k = np.empty(cap, abi.POINT), np.empty(cap, np.uint64)
        assert L.o3r_cloud_changes(P.handle, out.ctypes.data, k.ctypes.data, None, cap, C.byref(nc)) == 0
        assert nc.value == len(exp_keys) > n1.value
        assert np.array_equal(k[:nc.value], exp_keys)


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_FUSED])
def test_clear_and_append(mode):
    keep = []
    p = _params(mode, 1)
    cycles = _cycles(250, keep=keep)
    with Pose(p) as P:
        P.trackCloudChanges(True)
        P.createCycleClouds(cycles[0])
        P.cloudChanges()
        P.createCycleClouds(cycles[1])
        P.clearCloud()
        pts, _, _ = P.cloudChanges()
        assert len(pts) == 0
        P.createCycleClouds(cycles[3])
        pts, keys, _ = P.cloudChanges()
        _eq(pts, P.downsamplePtCloud())
    if mode != abi.MERGE_ACCUMULATE:
        return
    with Pose(p) as P:   # o3r_cloud_append merges through the same funnel
        P.trackCloudChanges(True)
        P.createCycleClouds(cycles[0])
        m = KeyMap()
        m.upsert(*P.cloudChanges()[:2])
        extra = ob.create_and_transform_pt_cloud(p, cycles[1][0], abi.DISP_U8)
        P.appendPoints(extra)
        pts, keys, _ = P.cloudChanges()
        assert len(keys) > 0
        assert keys.tolist() == sorted(_cell_counts(extra, 0.05))
        m.upsert(pts, keys)
        _eq(m.points(), P.downsamplePtCloud())


def test_refusals():
    L = lib.load()
    keep = []
    frames = _frames(260, 2, SMALL4["rows"], SMALL4["cols"], keep=keep)
    for kw in (dict(merge_mode=abi.MERGE_RETAIN), dict(dont_downsample=True)):
        with Pose(abi.make_params(jump_pixels=1, voxel_size=0.05, **SMALL4, **kw)) as P:
            P.createCycleClouds(frames)
            n, a, b, c = C.c_size_t(0), C.c_void_p(), C.c_void_p(), C.c_void_p()
            assert L.o3r_cloud_track_changes(P.handle, 1) == -4
            assert L.o3r_cloud_changes(P.handle, None, None, None, 0, C.byref(n)) == -4
            assert L.o3r_cloud_changes_dev(P.handle, C.byref(a), C.byref(b), C.byref(c), C.byref(n)) == -4
    with Pose(_params(abi.MERGE_ACCUMULATE, 1)) as P:
        with pytest.raises(lib.O3RError) as e:
            P.cloudChanges()
        assert e.value.code == -1
        P.trackCloudChanges(True)
        P.trackCloudChanges(False)
        with pytest.raises(lib.O3RError) as e:
            P.cloudChangesDevice()
        assert e.value.code == -1


@pytest.mark.parametrize("mode", ACC_MODES)
def test_launch_counts_off_and_on(mode):
    keep = []
    p = _params(mode, 1)
    r, c = SMALL4["rows"], SMALL4["cols"]
    cycles = [_frames(270 + i, 3, r, c, keep=keep, traj_start=3 * i) for i in range(4)]

    def per_cycle(P, read):
        d = []
        for frames in cycles:
            n0 = P.launch_count()
            P.createCycleClouds(frames)
            d.append(P.launch_count() - n0)
            if read:
                P.cloudChanges()
        return d

    with Pose(p) as never, Pose(p) as toggled, Pose(p) as on:
        toggled.trackCloudChanges(True)
        toggled.trackCloudChanges(False)
        on.trackCloudChanges(True)
        on.cloudChanges()   # (the full state: from here on every merged cycle runs the union)
        base = per_cycle(never, False)
        assert per_cycle(toggled, False) == base
        assert per_cycle(on, True) == [b + CHG_LAUNCHES_PER_CYCLE for b in base]


def test_device_result_matches_host_result():
    torch = pytest.importorskip("torch")
    keep = []
    p = _params(abi.MERGE_ACCUMULATE_FUSED, 2)
    cycles = _cycles(280, keep=keep)

    def dev(ptr, n, dtype, size):
        class DevArr:
            __cuda_array_interface__ = {"shape": (n * size,), "typestr": "|u1", "data": (ptr, False), "version": 2}
        return torch.as_tensor(DevArr(), device="cuda").cpu().numpy().view(dtype)

    with Pose(p) as A, Pose(p) as B:
        A.trackCloudChanges(True)
        B.trackCloudChanges(True)
        for frames in cycles:
            A.createCycleClouds(frames)
            B.createCycleClouds(frames)
            hp, hk, hc = A.cloudChanges()
            pp, pk, pc, n = B.cloudChangesDevice()
            assert n == len(hp)
            if n:
                _eq(dev(pp, n, abi.POINT, 16), hp)
                assert np.array_equal(dev(pk, n, np.uint64, 8), hk)
                assert np.array_equal(dev(pc, n, np.uint32, 4), hc)


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_FUSED])
def test_world1_communicator(mode):
    keep = []
    p = _params(mode, 2)
    cycles = _cycles(290, keep=keep)
    with Pose(p) as X, Pose(p) as plain:
        X.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        X.trackCloudChanges(True)
        plain.trackCloudChanges(True)
        m = KeyMap()
        for frames in cycles:
            X.createCycleClouds(frames)
            X.exchangeCycle()
            plain.createCycleClouds(frames)
            pts, keys, counts = X.cloudChanges()
            _, pk, pcnt = plain.cloudChanges()
            assert np.array_equal(keys, pk) and np.array_equal(counts, pcnt)
            m.upsert(pts, keys)
            _eq(m.points(), X.downsamplePtCloud())
        X.commDestroy()


def test_full_size_720p_fused():
    """configs[1] geometry: 50 720p images reused along a lawnmower trajectory (as bench.py does), 3 cycles x 50 frames,
    then a one-frame cycle."""
    keep = []
    seq = synth.sequence(1002, 50, 720, 1280)
    Ts = synth.trajectory(np.random.default_rng(1002 + 7919), 151)
    frames = [abi.make_frame(seq[j % 50][0], seq[j % 50][1], Ts[j], keep=keep) for j in range(151)]
    p = abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=3, merge_mode=abi.MERGE_ACCUMULATE_FUSED)
    with Pose(p) as P, Pose(p) as twin:
        P.trackCloudChanges(True)
        twin.trackCloudChanges(True)
        m = KeyMap()
        for i in range(3):
            P.createCycleClouds(frames[50 * i:50 * (i + 1)])
            twin.createCycleClouds(frames[50 * i:50 * (i + 1)])
            m.upsert(*P.cloudChanges()[:2])
        _eq(m.points(), P.downsamplePtCloud())
        # the one-frame cycle's changes = the grown cells; both full states from the twin (re-enable before and after)
        twin.trackCloudChanges(True)
        _, k0, c0 = twin.cloudChanges()
        P.createCycleClouds(frames[150:])
        twin.createCycleClouds(frames[150:])
        pts, keys, counts = P.cloudChanges()
        twin.trackCloudChanges(True)
        _, k1, c1 = twin.cloudChanges()
        before = dict(zip(k0.tolist(), c0.tolist()))
        grown = [(k, c) for k, c in zip(k1.tolist(), c1.tolist()) if c > before.get(k, 0)]
        assert len(keys) > 1000
        assert keys.tolist() == [k for k, _ in grown] and counts.tolist() == [c for _, c in grown]
        m.upsert(pts, keys)
        _eq(m.points(), P.downsamplePtCloud())
