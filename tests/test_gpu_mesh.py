"""o3r_cloud_mesh on the GPU against the numpy model (tests/mesh_model.py), with maps built through o3r_cloud_append and
o3r_cloud_import_cells in every accumulate mode: the vertices are the downsample's output bit for bit, the triangles and
normals equal the model built from the context's own export exactly, calls are reproducible, the host and device entry
points agree, and the context is left as it was."""
import ctypes as C

import numpy as np
import pytest

import mesh_model as mm
import register_model as reg
from online_3d_reconstruction_b200 import abi, lib
from online_3d_reconstruction_b200.pose import Pose

pytestmark = pytest.mark.gpu
MODES = [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE_FUSED]
V = 1.0


def _ctx(mode, min_points=1, **kw):
    return Pose(abi.make_params(voxel_size=V, min_points_per_voxel=min_points, merge_mode=mode, **kw))


def _code(fn, *a, **kw):
    with pytest.raises(lib.O3RError) as e:
        fn(*a, **kw)
    return e.value.code


def _holes_and_cliff(seed=3):
    """A plane with a 10 m high block on it (a cliff on four sides) and holes punched out of both."""
    rng = np.random.default_rng(seed)
    g = np.arange(-30.0, 30.0, 0.25) + 0.125
    x, y = np.meshgrid(g, g)
    x, y = x.ravel(), y.ravel()
    z = 0.02 * x + np.where((np.abs(x - 5) < 8) & (np.abs(y + 3) < 6), 10.0, 0.0)
    holes = rng.uniform(-30, 30, (25, 2))
    keep = np.ones(x.size, bool)
    for hx, hy in holes:
        keep &= np.hypot(x - hx, y - hy) > rng.uniform(0.5, 3.0)
    keep &= rng.random(x.size) > 0.3   # thins some cells below min_points = 3
    p = np.zeros(int(keep.sum()), dtype=abi.POINT)
    p["x"], p["y"], p["z"] = x[keep].astype(np.float32), y[keep].astype(np.float32), z[keep].astype(np.float32)
    p["rgb"] = 0x336699
    return p


SCENES = {
    "terrain": lambda: reg.terrain_scene()[0],
    "flat": lambda: reg.flat_scene(V)[0],
    "holes_cliff": _holes_and_cliff,
}


@pytest.fixture(scope="module")
def scenes():
    return {k: f() for k, f in SCENES.items()}


def _build(P, mp, how):
    if how == "append":
        P.appendPoints(mp)
    else:
        P.importCells(reg.cells_from_points(mp, V))


def _check(P, min_points, max_step=np.inf):
    """The mesh against the downsample and the model of the context's own export; returns it."""
    verts, nrm, tris = P.meshCloud(max_step)
    ds = P.downsamplePtCloud()
    assert verts.tobytes() == ds.tobytes()
    M, nrm_m, tris_m = mm.mesh(P.exportCells(), V, min_points, max_step)
    assert np.array_equal(tris, tris_m)
    assert nrm.tobytes() == nrm_m.tobytes(), np.argwhere(nrm != nrm_m)[:5]
    return verts, nrm, tris


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("how", ["append", "import"])
@pytest.mark.parametrize("scene", list(SCENES))
def test_matches_model(mode, how, scene, scenes):
    mp = scenes[scene]
    min_points = 3 if scene == "holes_cliff" else 1
    with _ctx(mode, min_points) as P:
        _build(P, mp, how)
        verts, nrm, tris = _check(P, min_points)
        assert len(tris) > len(verts)
        _check(P, min_points, max_step=1.0)
        if scene == "holes_cliff":   # the gate removes the walls of the block
            assert len(P.meshCloud(1.0)[2]) < len(tris)


@pytest.mark.parametrize("mode", MODES)
def test_boundary_cells(mode):
    lim = mm.LIM
    lo, hi = (-lim, -lim + 1, -lim + 2), (lim - 2, lim - 1, lim)
    ijk = [(a, b, k) for I in (lo, hi) for J in (lo, hi) for a in I for b in J for k in (-3, 0)]
    rng = np.random.default_rng(11)
    cells = mm.cells_at(ijk, rng.normal(0, 0.3, len(ijk)).astype(np.float32).astype(np.float64), n=2)
    with _ctx(mode) as P:
        P.importCells(cells)
        verts, nrm, tris = _check(P, 1)
        assert len(verts) == len(ijk) and len(tris) == 8 * 8
        assert np.count_nonzero(np.any(nrm != 0, axis=1)) == 8 * 4   # only |i|, |j| <= 2^20 - 2 fit


@pytest.mark.parametrize("mode", MODES)
def test_reproducible_and_dev_entry_agrees(mode, scenes):
    torch = pytest.importorskip("torch")

    def dev(ptr, n, dtype, width):
        if n == 0:
            return np.zeros(0, dtype=dtype)

        class DevArr:
            __cuda_array_interface__ = {"shape": (n * width,), "typestr": "|u1", "data": (ptr, False), "version": 2}
        return torch.as_tensor(DevArr(), device="cuda").cpu().numpy().view(dtype)

    with _ctx(mode) as P:
        _build(P, scenes["terrain"], "append")
        a = P.meshCloud(2.0)
        b = P.meshCloud(2.0)
        pv, pn, nv, pt, nt = P.meshCloudDevice(2.0)
        assert nv == len(a[0]) and nt == len(a[2])
        d = (dev(pv, nv, abi.POINT, 16), dev(pn, nv, np.float32, 12).reshape(-1, 3), dev(pt, nt, np.uint32, 12).reshape(-1, 3))
    for x in (b, d):
        for u, w in zip(a, x):
            assert u.tobytes() == w.tobytes()


@pytest.mark.parametrize("mode", MODES)
def test_no_side_effects(mode, scenes):
    mp = scenes["terrain"]
    with _ctx(mode) as P:
        P.appendPoints(mp[: len(mp) // 2])
        P.trackCloudChanges(True)
        P.cloudChanges()
        P.appendPoints(mp[len(mp) // 2:])
        last0 = P.lastCyclePoints().tobytes()
        cells0 = P.exportCells().tobytes()
        ds0 = P.downsamplePtCloud().tobytes()
        P.meshCloud()
        P.meshCloudDevice(0.5)
        assert P.exportCells().tobytes() == cells0
        assert P.downsamplePtCloud().tobytes() == ds0
        assert P.lastCyclePoints().tobytes() == last0
        ch, keys, _ = P.cloudChanges()
        with _ctx(mode) as Q:
            Q.appendPoints(mp[: len(mp) // 2])
            Q.trackCloudChanges(True)
            Q.cloudChanges()
            Q.appendPoints(mp[len(mp) // 2:])
            ch2, keys2, _ = Q.cloudChanges()
        assert len(ch) > 0 and keys.tobytes() == keys2.tobytes() and ch.tobytes() == ch2.tobytes()


@pytest.mark.parametrize("mode", MODES)
def test_empty_and_errors(mode, scenes):
    mp = scenes["flat"]
    with _ctx(mode, min_points=1000) as P:
        v, n, t = P.meshCloud()
        assert len(v) == len(n) == len(t) == 0                          # empty map
        assert P.meshCloudDevice()[2] == 0 and P.meshCloudDevice()[4] == 0
        P.appendPoints(mp)
        v, n, t = P.meshCloud()
        assert len(v) == len(t) == 0 and P.cloudSize() > 0              # every cell below min_points
    with _ctx(mode) as P:
        P.appendPoints(mp)
        for bad in (float("nan"), -1.0, -float("inf")):
            assert _code(P.meshCloud, bad) == abi.O3R_ERR_INVALID
        nv, nt = C.c_size_t(0), C.c_size_t(0)
        L = P._L
        assert L.o3r_cloud_mesh(P.handle, float("inf"), None, None, 0, C.byref(nv), None, 0, C.byref(nt)) == 0
        assert nv.value > 0 and nt.value > 0
        verts = np.empty(nv.value, dtype=abi.POINT)
        tris = np.empty((nt.value, 3), dtype=np.uint32)
        short_v, short_t = C.c_size_t(0), C.c_size_t(0)
        rc = L.o3r_cloud_mesh(P.handle, float("inf"), verts.ctypes.data, None, nv.value - 1, C.byref(short_v),
                              tris.ctypes.data, nt.value, C.byref(short_t))
        assert rc == abi.O3R_ERR_CAPACITY and (short_v.value, short_t.value) == (nv.value, nt.value)
        rc = L.o3r_cloud_mesh(P.handle, float("inf"), verts.ctypes.data, None, nv.value, C.byref(short_v),
                              tris.ctypes.data, nt.value - 1, C.byref(short_t))
        assert rc == abi.O3R_ERR_CAPACITY and (short_v.value, short_t.value) == (nv.value, nt.value)
        P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        assert _code(P.meshCloud) == abi.O3R_ERR_UNSUPPORTED
        assert _code(P.meshCloudDevice) == abi.O3R_ERR_UNSUPPORTED
        P.commDestroy()
        assert len(P.meshCloud()[2]) == nt.value
    with _ctx(mode, dont_downsample=True) as P:
        assert _code(P.meshCloud) == abi.O3R_ERR_UNSUPPORTED


def test_retain_is_unsupported():
    with _ctx(abi.MERGE_RETAIN) as P:
        assert _code(P.meshCloud) == abi.O3R_ERR_UNSUPPORTED
        assert _code(P.meshCloudDevice) == abi.O3R_ERR_UNSUPPORTED
