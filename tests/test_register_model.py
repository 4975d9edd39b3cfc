"""The numpy model of o3r_cloud_register (tests/register_model.py) on its own: it recovers a known perturbation of a source
cloud against a terrain map with relief, and on a flat plane it updates only z, roll and pitch.  The GPU tests compare the
kernels with this model.  CPU only."""
import numpy as np

import register_model as reg

V = 1.0


def test_model_recovers_known_transform_on_terrain():
    mp, src, E = reg.terrain_scene()
    M = reg.MapModel(reg.cells_from_points(mp, V), V, 1)
    T0 = np.eye(4, dtype=np.float32)
    t_err0, r_err0 = reg.pose_error(T0, E)
    T, st = reg.register(M, src)
    t_err, r_err = reg.pose_error(T, E)
    assert t_err0 > 0.5 and r_err0 > 2.0
    assert t_err < 0.2 * V and r_err < 0.05, (t_err, r_err, st)
    assert st["rank"] == 6 and st["converged"] == 1 and st["rms_final"] < st["rms_initial"]
    assert st["n_inliers"] > 0.95 * len(src)


def test_model_flat_plane_updates_z_roll_pitch_only():
    mp, src = reg.flat_scene(V, dz=0.25)
    M = reg.MapModel(reg.cells_from_points(mp, V), V, 1)
    T, st = reg.register(M, src)
    assert st["rank"] == 3 and st["converged"] == 1
    expect = np.eye(4, dtype=np.float32)
    expect[2, 3] = -0.25
    assert np.array_equal(T, expect)
    # a jittered plane seen with a roll: x, y and yaw stay unobservable, the rest is corrected
    rng = np.random.default_rng(3)
    src2 = src.copy()
    src2["z"] = 0.0
    src2["x"] += rng.uniform(-0.2, 0.2, len(src)).astype(np.float32)
    src2["y"] += rng.uniform(-0.2, 0.2, len(src)).astype(np.float32)
    E = reg.rigid(roll_deg=1.0, t=(0.0, 0.0, 0.2))
    T2, st2 = reg.register(M, reg.transform_points(src2, E))
    assert st2["rank"] == 3
    D = T2.astype(np.float64) @ E
    assert abs(D[2, 3]) < 1e-3 and abs(D[2, 1]) < 1e-5 and abs(D[2, 0]) < 1e-5
    assert abs(np.arctan2(T2[1, 0], T2[0, 0])) < 1e-6


def test_model_too_few_correspondences_keeps_T_init():
    mp, src = reg.flat_scene(V)
    M = reg.MapModel(reg.cells_from_points(mp, V), V, 1)
    T0 = reg.rigid(t=(1000.0, 0.0, 0.0)).astype(np.float32)
    T, st = reg.register(M, src, T0)
    assert np.array_equal(T, T0) and st["n_inliers"] == 0 and st["rank"] == 0 and st["iterations"] == 0
