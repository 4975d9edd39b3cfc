"""The host driver's --preview: a per-cycle preview.ply kept up to date from the cells each cycle changed."""
import os
import subprocess

import pytest

from test_host_driver import _write_dataset, pose_bin, read_ply  # noqa: F401 (pose_bin is a fixture)

pytestmark = pytest.mark.gpu


def _run(pose_bin, root, out, *extra):
    r = subprocess.run([pose_bin, "100", "105", "--seq_len", "2", "--voxel_size", "0.05", "--jump_pixels", "1",
                        "--min_points_per_voxel", "2", "--only_MAVLink", "--data_root", root, "--output", out, *extra],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return r, os.path.join(out, sorted(os.listdir(out))[0])


def test_preview_ply_equals_cloud_ply_and_logs_every_cycle(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_dataset(root, 6, 128, 256)
    r, run_dir = _run(pose_bin, root, str(tmp_path / "out"), "--preview")
    preview = open(os.path.join(run_dir, "preview.ply"), "rb").read()
    cloud = open(os.path.join(run_dir, "cloud.ply"), "rb").read()
    assert len(read_ply(os.path.join(run_dir, "cloud.ply"))[0]) > 100
    assert preview == cloud
    log = open(os.path.join(run_dir, "log.txt")).read()
    cycles = len([l for l in log.splitlines() if l.startswith("Cycle ") and l.split()[1].isdigit()])
    lines = [l for l in log.splitlines() if l.startswith("Preview cells changed/total: ")]
    assert cycles == 3 and len(lines) == cycles, log
    totals = [int(l.split("/")[-1]) for l in lines]
    assert totals == sorted(totals) and totals[-1] == len(read_ply(os.path.join(run_dir, "cloud.ply"))[0])
    assert int(lines[0].split(": ")[1].split("/")[0]) == totals[0]   # the first cycle changes every cell it shows
    assert "Preview cells changed/total" in r.stdout


def test_preview_with_dont_downsample_writes_no_preview(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_dataset(root, 6, 128, 256)
    r, run_dir = _run(pose_bin, root, str(tmp_path / "a"), "--dont_downsample", "--preview")
    assert "--preview needs the combined grid" in r.stdout
    assert not os.path.exists(os.path.join(run_dir, "preview.ply"))
    _, plain_dir = _run(pose_bin, root, str(tmp_path / "b"), "--dont_downsample")
    assert open(os.path.join(run_dir, "cloud.ply"), "rb").read() == open(os.path.join(plain_dir, "cloud.ply"), "rb").read()
