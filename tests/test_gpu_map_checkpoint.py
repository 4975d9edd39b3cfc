"""Map checkpoints (o3r_cloud_export_cells / o3r_cloud_import_cells / o3r_cloud_export_points): a map leaves its context
bit for bit and comes back, resumes as if never interrupted, merges with another flight, and refuses malformed records
without touching the map."""
import ctypes as C

import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi, exchange, lib
from online_3d_reconstruction_b200.pose import Pose
from test_gpu_parity import SMALL4, _close, _eq, _frames

pytestmark = pytest.mark.gpu
MODES = [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE_FUSED]
R, W = SMALL4["rows"], SMALL4["cols"]


def _params(mode, min_pts=1, **kw):
    return abi.make_params(jump_pixels=1, voxel_size=0.05, min_points_per_voxel=min_pts, merge_mode=mode, **SMALL4, **kw)


def _cycles(keep, seed=700, n=5, per=3, start=0):
    return [_frames(seed + c, per, R, W, keep=keep, traj_start=start + c * per) for c in range(n)]


def _code(fn, *a):
    with pytest.raises(lib.O3RError) as e:
        fn(*a)
    return e.value.code, str(e.value)


def _bytes(a):
    return np.ascontiguousarray(a).tobytes()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("min_pts", [1, 3])
def test_round_trip_is_bit_exact(mode, min_pts):
    keep = []
    cyc = _cycles(keep, 710, n=2)
    p = _params(mode, min_pts)
    with Pose(p) as P:
        for c in cyc:
            P.createCycleClouds(c)
        cells, size, ds = P.exportCells(), P.cloudSize(), P.downsamplePtCloud()
    assert len(cells) == size > 1000
    assert np.all(np.diff(cells["key"].astype(np.uint64)) > 0) and np.all(cells["pad"] == 0)
    assert np.count_nonzero(cells["n"] >= min_pts) == len(ds)
    if min_pts > 1:
        assert np.any(cells["n"] < min_pts)   # cells below the threshold are state and are exported
    with Pose(p) as Q:
        Q.importCells(cells)
        again = Q.exportCells()
        assert Q.cloudSize() == size
        _eq(Q.downsamplePtCloud(), ds)
    assert _bytes(again) == _bytes(cells)


@pytest.mark.parametrize("mode", MODES)
def test_resume_equals_uninterrupted(mode):
    keep = []
    cyc = _cycles(keep, 720)
    p = _params(mode, 3)
    with Pose(p) as A:
        for c in cyc:
            A.createCycleClouds(c)
        full_cells, full_ds = A.exportCells(), A.downsamplePtCloud()
    runs = [(cyc[:2], cyc[2:])]
    if mode == abi.MERGE_ACCUMULATE:   # in input order per point, its result does not depend on the batching
        runs.append((cyc[:2] + [cyc[2][:1]], [cyc[2][1:]] + cyc[3:]))
    for before, after in runs:
        with Pose(p) as B:
            for c in before:
                B.createCycleClouds(c)
            ck = B.exportCells()
        with Pose(p) as C2:
            C2.importCells(ck)
            for c in after:
                C2.createCycleClouds(c)
            cells, ds = C2.exportCells(), C2.downsamplePtCloud()
        assert _bytes(cells) == _bytes(full_cells)
        _eq(ds, full_ds)
        # a cell below min_points at the checkpoint crosses it after the resume
        below = ck["key"][ck["n"] < 3]
        final_n = dict(zip(cells["key"].tolist(), cells["n"].tolist()))
        assert any(final_n[k] >= 3 for k in below.tolist())


def _voxel_keys_counts(p, big):
    sh = big.copy()
    sh["z"] += np.float32(500)
    _, keys, counts, _ = ob.voxel_grid(sh, (p.voxel_size, p.voxel_size, 1000.0), 0)
    return keys, counts


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_FUSED])
def test_merging_two_flights(mode):
    keep = []
    fa = _cycles(keep, 730, n=2)
    fb = _cycles(keep, 740, n=2, start=2)   # overlaps flight A
    p = _params(mode, 2)
    cells = []
    for flight in (fa, fb):
        with Pose(p) as F:
            for c in flight:
                F.createCycleClouds(c)
            cells.append(F.exportCells())
    with Pose(p) as Q:
        Q.importCells(cells[0])
        Q.importCells(cells[1])
        merged, merged_ds = Q.exportCells(), Q.downsamplePtCloud()
    with Pose(p) as S:
        for c in fa + fb:
            S.createCycleClouds(c)
        both, both_ds = S.exportCells(), S.downsamplePtCloud()
    for f in ("key", "n", "sr", "sg", "sb"):
        assert np.array_equal(merged[f], both[f]), f
    _close(merged_ds, both_ds)
    assert len(np.intersect1d(cells[0]["key"], cells[1]["key"])) > 100
    # the oracle's cells of both flights' clouds
    big = []
    for flight in (fa, fb):
        cloud, n = None, 0
        for c in flight:
            cloud, n, _ = ob.run_cycle(p, c, abi.DISP_U8, 4, cloud, n)
        big.append(cloud[:n])
    keys, counts = _voxel_keys_counts(p, np.concatenate(big))
    assert np.array_equal(keys, merged["key"]) and np.array_equal(counts, merged["n"])


def test_duplicate_keys_in_one_import_sum_in_input_order():
    keep = []
    p = _params(abi.MERGE_ACCUMULATE)
    ex = []
    for seed in (750, 760):
        with Pose(p) as F:
            F.createCycleClouds(_frames(seed, 3, R, W, keep=keep))
            ex.append(F.exportCells())
    a, b = ex
    m = min(len(a), len(b)) // 2
    extra = b[:m].copy()
    extra["key"] = a["key"][::2][:m]       # other sums on keys already in the import
    rec = np.concatenate([a, extra, a[:50]])
    exp = {}
    for r in rec:
        k = int(r["key"])
        s = exp.setdefault(k, [np.float32(0), np.float32(0), np.float32(0), 0, 0, 0, 0])
        for i, f in enumerate(("sx", "sy", "sz")):
            s[i] = np.float32(s[i] + r[f])
        for i, f in enumerate(("n", "sr", "sg", "sb")):
            s[3 + i] += int(r[f])
    with Pose(p) as Q:
        Q.importCells(rec)
        got = Q.exportCells()
    assert np.array_equal(got["key"], np.array(sorted(exp), dtype=np.uint64))
    want = np.array([tuple(exp[k]) for k in sorted(exp)],
                    dtype=[("sx", "<f4"), ("sy", "<f4"), ("sz", "<f4"), ("n", "<u4"), ("sr", "<u4"), ("sg", "<u4"), ("sb", "<u4")])
    for f in want.dtype.names:
        assert _bytes(got[f]) == _bytes(want[f]), f


def _break(rec, reason):
    if reason == "bit63":
        rec["key"] |= np.uint64(1 << 63)
    elif reason == "field_i":
        rec["key"] &= ~np.uint64(0x1fffff)
    elif reason == "field_j":
        rec["key"] &= ~np.uint64(0x1fffff << 21)
    elif reason == "field_k":
        rec["key"] &= ~np.uint64(0x1fffff << 42)
    elif reason == "zero_n":
        rec["n"] = 0
    elif reason == "nan":
        rec["sy"] = np.float32(np.nan)
    elif reason == "inf":
        rec["sz"] = np.float32(-np.inf)
    elif reason == "colour":
        rec["sg"] = rec["n"] * 255 + 1
    elif reason == "pad":
        rec["pad"] = 1


_REASON_TEXT = {"bit63": "bit 63", "field_i": "key field", "field_j": "key field", "field_k": "key field", "zero_n": "n == 0",
                "nan": "not finite", "inf": "not finite", "colour": "colour sum", "pad": "pad != 0"}


@pytest.mark.parametrize("reason", list(_REASON_TEXT))
def test_refused_record_merges_nothing(reason):
    keep = []
    cyc = _cycles(keep, 770, n=2)
    p = _params(abi.MERGE_ACCUMULATE_FUSED, 2)
    with Pose(p) as F:
        F.createCycleClouds(_frames(780, 2, R, W, keep=keep, traj_start=3))
        imp = F.exportCells()
    bad = imp.copy()
    _break(bad[7:8], reason)
    other = "zero_n" if reason == "pad" else "pad"   # later bad records, another reason: the first index and its own reasons come back
    _break(bad[20:21], other)
    _break(bad[len(bad) - 5:len(bad) - 4], other)
    outs = []
    for with_bad in (True, False):
        with Pose(p) as P:
            P.trackCloudChanges(True)
            P.createCycleClouds(cyc[0])
            P.cloudChanges()
            P.createCycleClouds(cyc[1])
            before = P.exportCells()
            if with_bad:
                code, msg = _code(P.importCells, bad)
                assert code == abi.O3R_ERR_INVALID and "cell record 7 " in msg, msg
                assert _REASON_TEXT[reason] in msg and _REASON_TEXT[other] not in msg, msg
            assert _bytes(P.exportCells()) == _bytes(before)
            outs.append([_bytes(x) for x in P.cloudChanges()])
    assert outs[0] == outs[1]
    if reason == "colour":   # the limit itself is fine
        ok = imp.copy()
        ok["sg"][7] = ok["n"][7] * 255
        with Pose(p) as P:
            P.importCells(ok)


@pytest.mark.parametrize("rank", [0, 1])
def test_import_refuses_cells_of_another_rank(rank):
    """The ownership check on one GPU: a context attached as rank `rank` of 2 takes the cells hash64(key) % 2 names for it and
    refuses any other, naming the first one.  No collective is called, so the attached handle is never used."""
    keep = []
    p = _params(abi.MERGE_ACCUMULATE_FUSED)
    with Pose(p) as F:
        F.createCycleClouds(_frames(785, 2, R, W, keep=keep))
        cells = F.exportCells()
    own = exchange.owner_of(cells["key"], 2) == rank
    assert own.any() and not own.all()
    first_foreign = int(np.nonzero(~own)[0][0])
    L = lib.load()
    with Pose(p) as P:
        assert L.o3r_comm_attach(P.handle, C.c_void_p(1), 2, rank, 1 << 10) == 0
        code, msg = _code(P.importCells, cells)
        assert code == abi.O3R_ERR_INVALID and f"cell record {first_foreign} " in msg and "another rank" in msg, msg
        assert P.exportCells().size == 0
        P.importCells(cells[own])
        assert _bytes(P.exportCells()) == _bytes(cells[own])
        P.commDestroy()


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_FUSED])
def test_import_reports_exactly_its_cells_as_changes(mode):
    keep = []
    p = _params(mode, 2)
    with Pose(p) as F:
        F.createCycleClouds(_frames(790, 3, R, W, keep=keep, traj_start=2))
        imp = F.exportCells()
    with Pose(p) as Q:
        Q.trackCloudChanges(True)
        Q.createCycleClouds(_frames(795, 3, R, W, keep=keep))
        Q.cloudChanges()
        Q.importCells(imp)
        pts, keys, counts = Q.cloudChanges()
        cells, ds = Q.exportCells(), Q.downsamplePtCloud()
    emitted = cells[cells["n"] >= 2]
    assert len(emitted) == len(ds)
    want = np.isin(emitted["key"], imp["key"])
    assert 0 < want.sum() < len(emitted)
    assert np.array_equal(keys, emitted["key"][want]) and np.array_equal(counts, emitted["n"][want])
    _eq(pts, ds[want])


def test_large_import_with_wide_keys_round_trips():
    rng = np.random.default_rng(5)
    n = (1 << 20) + 123457
    lim = (1 << 20) - 1
    i = rng.integers(-lim, lim + 1, n)
    j = rng.integers(-lim, lim + 1, n)
    i[:4] = [-lim, lim, 0, lim]
    j[:4] = [lim, -lim, -lim, lim]
    k = rng.integers(-3, 4, n)
    B = 1 << 20
    keys = ((k + B).astype(np.uint64) << np.uint64(42)) | ((j + B).astype(np.uint64) << np.uint64(21)) | (i + B).astype(np.uint64)
    keys = np.unique(keys)
    c = np.zeros(len(keys), dtype=abi.CELL)
    c["key"] = keys
    c["n"] = rng.integers(1, 50, len(c))
    c["sx"], c["sy"] = (rng.normal(0, 1e4, len(c)).astype(np.float32) for _ in range(2))
    c["sz"] = rng.uniform(1, 1e4, len(c)).astype(np.float32)
    for ch in ("sr", "sg", "sb"):
        c[ch] = rng.integers(0, 256, len(c)) * c["n"]
    assert len(c) > 1 << 20
    rng.shuffle(perm := np.arange(len(c)))
    with Pose(_params(abi.MERGE_ACCUMULATE_FUSED)) as Q:
        Q.importCells(c[perm])   # any order in, ascending key out
        got = Q.exportCells()
        assert Q.cloudSize() == len(c)
    assert _bytes(got) == _bytes(c)


def test_retain_points_resume_with_transforms():
    keep = []
    cyc = _cycles(keep, 800, n=3)
    p = _params(abi.MERGE_RETAIN, 2)
    tf = np.eye(4, dtype=np.float32)
    cs, sn = np.float32(np.cos(0.02)), np.float32(np.sin(0.02))
    tf[0, 0], tf[0, 1], tf[1, 0], tf[1, 1] = cs, -sn, sn, cs
    tf[:3, 3] = [0.05, -0.03, 0.02]
    with Pose(p) as A:
        A.createCycleClouds(cyc[0]); A.transformPtCloud(tf)
        A.createCycleClouds(cyc[1]); A.transformPtCloud(tf)
        A.createCycleClouds(cyc[2])
        full = A.downsamplePtCloud()
    with Pose(p) as B:
        B.createCycleClouds(cyc[0]); B.transformPtCloud(tf)
        B.createCycleClouds(cyc[1])
        pts = B.exportPoints()
        assert len(pts) == B.cloudSize()
    with Pose(p) as C2:
        C2.appendPoints(pts)
        C2.transformPtCloud(tf)
        C2.createCycleClouds(cyc[2])
        _eq(C2.downsamplePtCloud(), full)


@pytest.mark.parametrize("mode", [abi.MERGE_ACCUMULATE, abi.MERGE_RETAIN])
def test_export_points_equals_dont_downsample_output(mode):
    keep = []
    p = _params(mode, dont_downsample=True)
    with Pose(p) as P:
        for c in _cycles(keep, 810, n=2):
            P.createCycleClouds(c)
        pts = P.exportPoints()
        _eq(pts, P.downsamplePtCloud())
    assert len(pts) > 1000


def test_unsupported_modes_and_query_then_fill():
    keep = []
    fr = _frames(820, 2, R, W, keep=keep)
    L = lib.load()
    cell = np.zeros(1, dtype=abi.CELL)
    for kw in (dict(mode=abi.MERGE_RETAIN), dict(mode=abi.MERGE_ACCUMULATE, dont_downsample=True),
               dict(mode=abi.MERGE_ACCUMULATE_FUSED, dont_downsample=True)):
        with Pose(_params(kw.pop("mode"), **kw)) as P:
            P.createCycleClouds(fr)
            assert _code(P.exportCells)[0] == abi.O3R_ERR_UNSUPPORTED
            assert _code(P.importCells, cell)[0] == abi.O3R_ERR_UNSUPPORTED
            n = C.c_size_t(0)
            assert L.o3r_cloud_export_points(P.handle, None, 0, C.byref(n)) == 0 and n.value == P.cloudSize() > 0
            buf = np.empty(n.value, dtype=abi.POINT)
            m = C.c_size_t(0)
            assert L.o3r_cloud_export_points(P.handle, buf.ctypes.data, n.value - 1, C.byref(m)) == abi.O3R_ERR_CAPACITY
            assert m.value == n.value
    for kw in (dict(), dict(dont_downsample=True)):   # a sharded point cloud cannot be exported
        with Pose(_params(abi.MERGE_RETAIN, **kw)) as P:
            P.commInit(1, 0, Pose.commUniqueId(), 1 << 10)
            P.createCycleClouds(fr)
            assert _code(P.exportPoints)[0] == abi.O3R_ERR_UNSUPPORTED
    for mode in MODES:
        with Pose(_params(mode)) as P:
            P.createCycleClouds(fr)
            assert _code(P.exportPoints)[0] == abi.O3R_ERR_UNSUPPORTED
            n = C.c_size_t(0)
            assert L.o3r_cloud_export_cells(P.handle, None, 0, C.byref(n)) == 0 and n.value == P.cloudSize() > 0
            buf = np.empty(n.value, dtype=abi.CELL)
            m = C.c_size_t(0)
            assert L.o3r_cloud_export_cells(P.handle, buf.ctypes.data, n.value - 1, C.byref(m)) == abi.O3R_ERR_CAPACITY
            assert m.value == n.value
            assert L.o3r_cloud_export_cells(P.handle, buf.ctypes.data, n.value, C.byref(m)) == 0 and m.value == n.value
            assert _bytes(buf) == _bytes(P.exportCells())
            P.importCells(np.zeros(0, dtype=abi.CELL))   # an empty import is a no-op
            assert P.cloudSize() == n.value


@pytest.mark.parametrize("mode", MODES)
def test_import_between_cycle_and_exchange_keeps_the_pending_batch(mode):
    keep = []
    cyc = _cycles(keep, 830, n=2)
    p = _params(mode, 2)
    with Pose(p) as F:
        F.createCycleClouds(_frames(840, 2, R, W, keep=keep, traj_start=2))
        imp = F.exportCells()
    with Pose(p) as S:
        for c in cyc:
            S.createCycleClouds(c)
        S.importCells(imp)
        plain, plain_ds = S.exportCells(), S.downsamplePtCloud()
    with Pose(p) as P:
        P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        P.createCycleClouds(cyc[0])
        P.exchangeCycle()
        P.createCycleClouds(cyc[1])
        last = P.lastCyclePoints() if mode == abi.MERGE_ACCUMULATE else None
        P.importCells(imp)
        if last is not None:
            _eq(P.lastCyclePoints(), last)
        P.exchangeCycle()
        got, got_ds = P.exportCells(), P.downsamplePtCloud()
    for f in ("key", "n", "sr", "sg", "sb"):
        assert np.array_equal(got[f], plain[f]), f
    _close(got_ds, plain_ds)
