"""The host driver's --register_map: a second cycle whose GPS altitude is 0.3 m off is corrected against the map built by
the first, and without the flag nothing changes."""
import os
import subprocess

import numpy as np
import pytest

from online_3d_reconstruction_b200 import abi, synth
from test_host_driver import pose_bin, write_png  # noqa: F401 (pose_bin is a fixture)

pytestmark = pytest.mark.gpu


def _write_same_frames(root, n, rows, cols, lifted, seed=91):
    """n frames of one image pair at one pose; the frames in `lifted` carry +0.3 m altitude in pose.txt."""
    for d in ("data_files", "images", "disparities"):
        os.makedirs(os.path.join(root, d))
    Q = abi.Q_CAM13
    with open(os.path.join(root, "data_files", "cam13calib.yml"), "w") as f:
        f.write("%YAML:1.0\nM1: !!opencv-matrix\n   rows: 1\n   cols: 1\n   dt: d\n   data: [ 1. ]\n"
                "Q: !!opencv-matrix\n   rows: 4\n   cols: 4\n   dt: d\n   data: [ " +
                ",\n       ".join(", ".join(repr(float(v)) for v in Q[i:i + 3]) for i in range(0, 16, 3)) + " ]\n")
    rng = np.random.default_rng(seed)
    img = synth.make_frame_images(rng, rows, cols)[1]
    yy, xx = np.mgrid[0:rows, 0:cols]
    # relief along both image axes, gentle enough at 720 x 1280 (slopes below 1) to be a height field at 5 cm cells, within
    # the variance gate of pose.cpp:187-196
    d = np.clip(np.rint(105 + 1.6 * np.sin(xx / 95.0) + 1.6 * np.sin(yy / 80.0 + 0.5) + rng.normal(0, 0.5, (rows, cols))),
                0, 127).astype(np.uint8)
    q = np.array([0.01, -0.02, 0.05, -0.9985]); q /= np.linalg.norm(q)
    times, poses = [], []
    for i in range(n):
        num = 100 + i
        write_png(os.path.join(root, "disparities", f"{num}.png"), d)
        write_png(os.path.join(root, "images", f"{num}.png"), img[:, :, ::-1])
        t_ns = 1532043429586341888 + i * 227000000
        times.append((num, t_ns))
        poses.append((t_ns, 0.0, 0.0, 22.0 + (0.3 if i in lifted else 0.0), *q))
    with open(os.path.join(root, "data_files", "images.txt"), "w") as f:
        for num, t in times:
            f.write(f"{num}.000000,{t / 1e9:.6f},{t}.000000\n")
    with open(os.path.join(root, "data_files", "pose.txt"), "w") as f:
        t0 = poses[0][0]
        rows_out = [(t0 - (25 - k) * 227000000, 99.0, 99.0, 99.0, 0.0, 0.0, 0.0, 1.0) for k in range(25)] + poses + \
                   [(poses[-1][0] + (k + 1) * 227000000, 99.0, 99.0, 99.0, 0.0, 0.0, 0.0, 1.0) for k in range(25)]
        for k, (t, *p) in enumerate(rows_out):
            f.write(f"{900 + k},{t / 1e9:.6f},{t}," + ",".join(f"{v:.9f}" for v in p) + "\n")


def _run(pose_bin, root, out, *extra):
    r = subprocess.run([pose_bin, "100", "105", "--seq_len", "3", "--jump_pixels", "1", "--voxel_size", "0.05",
                        "--only_MAVLink", "--data_root", root, "--output", out, *extra], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return r, os.path.join(out, sorted(os.listdir(out))[0])


def test_register_map_corrects_altitude(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_same_frames(root, 6, 720, 1280, lifted={3, 4, 5})
    r, run_dir = _run(pose_bin, root, str(tmp_path / "reg"), "--register_map")
    lines = [l for l in r.stdout.splitlines() if l.startswith("Map registration: ")]
    assert len(lines) == 1, r.stdout
    log = open(os.path.join(run_dir, "log.txt")).read()
    assert lines[0] in log
    t = [float(v) for v in lines[0].split("t = (")[1].rstrip(")").split(",")]
    print(lines[0])
    assert abs(t[2] + 0.3) < 0.005 and abs(t[0]) < 0.005 and abs(t[1]) < 0.005, lines[0]


def test_without_flag_nothing_changes(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_same_frames(root, 6, 128, 256, lifted={3, 4, 5})
    r, run_dir = _run(pose_bin, root, str(tmp_path / "a"))
    assert "Map registration" not in r.stdout
    assert "Map registration" not in open(os.path.join(run_dir, "log.txt")).read()
