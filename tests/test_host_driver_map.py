"""The host driver's --save_map / --resume_map: a run split across two processes writes the same cloud.ply as one run."""
import os
import subprocess

import numpy as np
import pytest

from online_3d_reconstruction_b200 import abi, mapfile
from online_3d_reconstruction_b200.pose import Pose
from test_host_driver import _write_dataset, pose_bin  # noqa: F401 (pose_bin is a fixture)

pytestmark = pytest.mark.gpu


def _run(pose_bin, root, out, first, last, *extra, ok=True):
    r = subprocess.run([pose_bin, str(first), str(last), "--seq_len", "2", "--jump_pixels", "1", "--min_points_per_voxel", "2",
                        "--only_MAVLink", "--data_root", root, "--output", out, *extra], capture_output=True, text=True)
    if ok:
        assert r.returncode == 0, r.stdout + r.stderr
    return r, (os.path.join(out, sorted(os.listdir(out))[0]) if os.path.isdir(out) and os.listdir(out) else None)


@pytest.mark.parametrize("dont_downsample", [False, True])
def test_save_then_resume_equals_one_run(pose_bin, tmp_path, dont_downsample):
    root = str(tmp_path / "data")
    _write_dataset(root, 6, 128, 256)
    ex = ["--voxel_size", "0.05"] + (["--dont_downsample"] if dont_downsample else [])
    _, one = _run(pose_bin, root, str(tmp_path / "one"), 100, 105, *ex)
    _, first = _run(pose_bin, root, str(tmp_path / "a"), 100, 103, "--save_map", *ex)
    saved = os.path.join(first, "map.o3rmap")
    r, second = _run(pose_bin, root, str(tmp_path / "b"), 104, 105, "--resume_map", saved, *ex)
    assert "Resumed map" in r.stdout
    whole = open(os.path.join(one, "cloud.ply"), "rb").read()
    assert open(os.path.join(second, "cloud.ply"), "rb").read() == whole
    assert len(whole) > 2000
    # the driver's file is what mapfile.py reads, and it holds the first run's resident map
    h, recs = mapfile.read(saved)
    assert int(h["kind"]) == (mapfile.KIND_POINTS if dont_downsample else mapfile.KIND_CELLS)
    assert float(h["voxel_size"]) == 0.05 and (int(h["world"]), int(h["rank"])) == (1, 0)
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=0.05, min_points_per_voxel=2,
                        dont_downsample=dont_downsample)
    with Pose(p) as P:
        assert mapfile.load(saved, P) == len(recs) > 100
        again = P.exportPoints() if dont_downsample else P.exportCells()
    assert again.tobytes() == recs.tobytes()


def test_resume_refuses_another_grid_and_a_corrupt_file(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_dataset(root, 6, 128, 256)
    _, first = _run(pose_bin, root, str(tmp_path / "a"), 100, 101, "--save_map", "--voxel_size", "0.05")
    saved = os.path.join(first, "map.o3rmap")
    r, _ = _run(pose_bin, root, str(tmp_path / "b"), 102, 103, "--resume_map", saved, "--voxel_size", "0.1", ok=False)
    assert r.returncode != 0 and "voxel_size" in r.stderr, r.stdout + r.stderr
    r, _ = _run(pose_bin, root, str(tmp_path / "c"), 102, 103, "--resume_map", saved, "--voxel_size", "0.05",
                "--dont_downsample", ok=False)
    assert r.returncode != 0 and "holds cells" in r.stderr, r.stdout + r.stderr
    bad = tmp_path / "bad.o3rmap"
    bad.write_bytes(open(saved, "rb").read()[:-5])
    r, _ = _run(pose_bin, root, str(tmp_path / "d"), 102, 103, "--resume_map", str(bad), "--voxel_size", "0.05", ok=False)
    assert r.returncode != 0 and "header announces" in r.stderr, r.stdout + r.stderr
    # a well-formed file whose records the library refuses: the import's message, nothing written
    h, recs = mapfile.read(saved)
    broken = recs.copy()
    broken["n"][3] = 0
    mapfile.write(str(bad), mapfile.KIND_CELLS, broken, 0.05)
    r, _ = _run(pose_bin, root, str(tmp_path / "e"), 102, 103, "--resume_map", str(bad), "--voxel_size", "0.05", ok=False)
    assert r.returncode != 0 and "cell record 3 refused" in r.stderr, r.stdout + r.stderr


def test_preview_shows_the_resumed_map(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_dataset(root, 6, 128, 256)
    _, first = _run(pose_bin, root, str(tmp_path / "a"), 100, 103, "--save_map", "--voxel_size", "0.05")
    _, run_dir = _run(pose_bin, root, str(tmp_path / "b"), 104, 105, "--resume_map", os.path.join(first, "map.o3rmap"),
                      "--voxel_size", "0.05", "--preview")
    preview = open(os.path.join(run_dir, "preview.ply"), "rb").read()
    assert preview == open(os.path.join(run_dir, "cloud.ply"), "rb").read()
    log = open(os.path.join(run_dir, "log.txt")).read()
    first_total = int([l for l in log.splitlines() if l.startswith("Preview cells changed/total: ")][0].split("/")[-1])
    cells = mapfile.read(os.path.join(first, "map.o3rmap"))[1]
    assert first_total >= np.count_nonzero(cells["n"] >= 2) > 0   # the first preview already holds the resumed map
