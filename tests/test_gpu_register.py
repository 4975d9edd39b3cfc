"""o3r_cloud_register on the GPU against the numpy model (tests/register_model.py), with maps built through o3r_cloud_append
and o3r_cloud_import_cells in every accumulate mode: one iteration agrees with the model's linearisation, a full run with
its result, flat ground leaves x, y and yaw alone, calls are reproducible bit for bit and leave the context as it was."""
import numpy as np
import pytest

import register_model as reg
from online_3d_reconstruction_b200 import abi, lib
from online_3d_reconstruction_b200.pose import Pose

pytestmark = pytest.mark.gpu
MODES = [abi.MERGE_ACCUMULATE, abi.MERGE_ACCUMULATE_TILED, abi.MERGE_ACCUMULATE_FUSED]
V = 1.0


def _ctx(mode, **kw):
    return Pose(abi.make_params(voxel_size=V, min_points_per_voxel=1, merge_mode=mode, **kw))


@pytest.fixture(scope="module")
def terrain():
    return reg.terrain_scene()


def _build(P, mp, how):
    if how == "append":
        P.appendPoints(mp)
    else:
        P.importCells(reg.cells_from_points(mp, V))
    return reg.MapModel(P.exportCells(), V, 1)


def _code(fn, *a, **kw):
    with pytest.raises(lib.O3RError) as e:
        fn(*a, **kw)
    return e.value.code


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("how", ["append", "import"])
def test_one_iteration_matches_model(mode, how, terrain):
    mp, src, _ = terrain
    with _ctx(mode) as P:
        M = _build(P, mp, how)
        T, st = P.registerCloud(src, max_iterations=1)
    Tm, sm = reg.register(M, src, max_iterations=1)
    assert st["n_inliers"] == sm["n_inliers"] > 0
    info, ref = st["info"], np.asarray(sm["info"])
    assert np.all(np.abs(info - ref) <= 1e-9 * np.abs(ref).max()), np.abs(info - ref).max()
    assert np.allclose(st["pivot"], sm["pivot"], rtol=0, atol=1e-9)
    assert np.abs(T.astype(np.float64) - Tm).max() <= 1e-6


@pytest.mark.parametrize("mode", MODES)
def test_full_run_matches_model_and_truth(mode, terrain):
    mp, src, E = terrain
    with _ctx(mode) as P:
        M = _build(P, mp, "append")
        T, st = P.registerCloud(src)
    Tm, sm = reg.register(M, src)
    assert np.abs(T.astype(np.float64) - Tm).max() <= 1e-5
    assert st["iterations"] == sm["iterations"] and st["rank"] == 6 and st["converged"] == 1
    t_err, r_err = reg.pose_error(Tm, E)
    g_err = reg.pose_error(T, E)
    print(f"model error {t_err:.4f} m {r_err:.5f} deg; GPU error {g_err[0]:.4f} m {g_err[1]:.5f} deg; "
          f"{st['iterations']} iterations, rms {st['rms_initial']:.4f} -> {st['rms_final']:.4f}")
    assert t_err < 0.2 * V and r_err < 0.05


@pytest.mark.parametrize("mode", MODES)
def test_flat_plane_keeps_x_y_yaw(mode):
    mp, src = reg.flat_scene(V, dz=0.25)
    with _ctx(mode) as P:
        P.appendPoints(mp)
        T0 = np.eye(4, dtype=np.float32)
        T, st = P.registerCloud(src, T0)
    assert st["rank"] == 3
    assert T[0, 3].tobytes() == T0[0, 3].tobytes() and T[1, 3].tobytes() == T0[1, 3].tobytes()
    assert T[:2, :2].tobytes() == T0[:2, :2].tobytes()
    assert abs(T[2, 3] + 0.25) < 1e-6


@pytest.mark.parametrize("mode", MODES)
def test_reproducible_and_dev_entry_agrees(mode, terrain):
    torch = pytest.importorskip("torch")
    mp, src, _ = terrain
    with _ctx(mode) as P:
        _build(P, mp, "append")
        a = P.registerCloud(src)
        b = P.registerCloud(src)
        d_src = torch.from_numpy(src.view(np.uint8).copy()).cuda()
        c = P.registerCloud(None, device_pointer=(d_src.data_ptr(), len(src)))
    for x in (b, c):
        assert x[0].tobytes() == a[0].tobytes()
        for k in a[1]:
            assert np.asarray(x[1][k]).tobytes() == np.asarray(a[1][k]).tobytes(), k


@pytest.mark.parametrize("mode", MODES)
def test_no_side_effects(mode, terrain):
    mp, src, _ = terrain
    with _ctx(mode) as P:
        P.appendPoints(mp[: len(mp) // 2])
        P.trackCloudChanges(True)
        P.cloudChanges()
        P.appendPoints(mp[len(mp) // 2:])
        last0 = P.lastCyclePoints().tobytes()
        cells0 = P.exportCells().tobytes()
        P.registerCloud(src)
        assert P.exportCells().tobytes() == cells0
        assert P.lastCyclePoints().tobytes() == last0
        ch, keys, cnt = P.cloudChanges()
        assert len(ch) > 0 and len(ch) == len(np.unique(keys))
        # the pending set is what the second half of the map grew, registration or not
        with _ctx(mode) as Q:
            Q.appendPoints(mp[: len(mp) // 2])
            Q.trackCloudChanges(True)
            Q.cloudChanges()
            Q.appendPoints(mp[len(mp) // 2:])
            ch2, keys2, _ = Q.cloudChanges()
        assert keys.tobytes() == keys2.tobytes() and ch.tobytes() == ch2.tobytes()


@pytest.mark.parametrize("mode", MODES)
def test_edge_cases(mode):
    mp, src = reg.flat_scene(V)
    with _ctx(mode) as P:
        T0 = reg.rigid(yaw_deg=10.0, t=(1.0, 2.0, 3.0)).astype(np.float32)
        T, st = P.registerCloud(src, T0)   # empty map
        assert st["n_inliers"] == 0 and T.tobytes() == T0.tobytes()
        P.appendPoints(mp)
        far = reg.rigid(t=(5000.0, 0.0, 0.0)).astype(np.float32)
        T, st = P.registerCloud(src, far)
        assert st["n_inliers"] == 0 and st["rank"] == 0 and T.tobytes() == far.tobytes()
        T, st = P.registerCloud(src[:0])
        assert st["n_inliers"] == 0 and T.tobytes() == np.eye(4, dtype=np.float32).tobytes()
        bad = src.copy()
        bad["z"][17] = np.nan
        assert _code(P.registerCloud, bad) == abi.O3R_ERR_INVALID
        Tb = np.eye(4, dtype=np.float32)
        Tb[3, 0] = 1.0
        assert _code(P.registerCloud, src, Tb) == abi.O3R_ERR_INVALID
        assert _code(P.registerCloud, src, 2 * np.eye(4, dtype=np.float32)) == abi.O3R_ERR_INVALID
        assert _code(P.registerCloud, src, max_iterations=0) == abi.O3R_ERR_INVALID
        assert _code(P.registerCloud, src, max_distance=-1.0) == abi.O3R_ERR_INVALID
        P.commInit(1, 0, Pose.commUniqueId(), 1 << 16)
        assert _code(P.registerCloud, src) == abi.O3R_ERR_UNSUPPORTED
        P.commDestroy()
    with _ctx(mode, dont_downsample=True) as P:
        assert _code(P.registerCloud, src) == abi.O3R_ERR_UNSUPPORTED


def test_retain_is_unsupported():
    _, src = reg.flat_scene(V)
    with _ctx(abi.MERGE_RETAIN) as P:
        assert _code(P.registerCloud, src) == abi.O3R_ERR_UNSUPPORTED
