"""CPU checks of bench.py's bookkeeping: the algorithmic-byte formulas against SURVEY.md 8(d)'s per-frame figures, one config
object for both arms (the driver compares them), every workload's parameters buildable, and the reference arm end to end on a
tiny sample (it runs on the host cores only)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from online_3d_reconstruction_b200 import abi  # noqa: E402


def test_stage_a_bytes_match_the_survey_figure():
    """SURVEY 8(d): 720p u8, J = 1, all valid: W*H*b_d + 3*Npix + 16*Nvalid = 921 600 + 2 244 000 + 11 968 000 = 15.13 MB per frame."""
    F = bench.WORKLOADS["config3_dont_downsample_720p"][7]
    npix = 748000
    alg = bench.algorithmic_bytes("config3_dont_downsample_720p", n_valid=npix * F, n_vox=0, n_cells_cycle=1, bd=1)
    # the two-pass stage A reads the ROI disparity twice (k_pre + k_emit) and the colours once, and writes 16 B per point
    assert alg["k_emit"] == F * (npix * 1 + npix * 3 + npix * 16)
    assert alg["k_pre"] == F * npix
    # the fused tile kernel's figure is SURVEY's "fused A+B": every input plane once + 20 B per per-frame voxel
    n_vox = 26_000_000
    alg2 = bench.algorithmic_bytes("config2_semidense_720p", n_valid=npix * F, n_vox=n_vox, n_cells_cycle=1, bd=1, np1=0, np2=3,
                                   n_part=840_000)
    assert alg2["k_tv"] == F * (720 * 1280 * 1 + 3 * npix) + 20 * n_vox
    assert alg2["k_rs_onesweep_u32"] == 3 * 840_000 * 16   # no per-frame index sort in the tile engine: only the 3 merge passes
    assert all(v >= 0 for v in alg2.values())


def test_both_arms_print_one_config_object_and_every_workload_builds():
    for wl in bench.WORKLOADS:
        c1, c2 = bench.static_config(wl, 1), bench.static_config(wl, 1)
        assert c1 == c2 and c1["workload"] == wl and "model" not in c1
        p = bench.params_for(wl, 0)
        ny, nx = abi.scan_dims(p)
        assert ny > 0 and nx > 0
    assert bench.static_config("config2_semidense_720p", 8)["frames_per_step"] == 50   # per GPU: weak scaling


def _cloud(rng, n):
    pts = np.zeros(n, abi.POINT)
    pts["x"], pts["y"], pts["z"] = rng.normal(size=(3, n)).astype(np.float32)
    pts["rgb"] = rng.integers(0, 1 << 32, n, dtype=np.uint32)   # every bit of the colour word, the top byte too
    return pts


def test_dump_outputs_writes_float_arrays_and_a_fixed_sample(tmp_path, monkeypatch):
    """--dump-outputs: counts as float64, a cloud as xyz float32 and the whole colour word as float64; a cloud larger than the
    cap becomes the same ascending sample on every run, with its indices."""
    monkeypatch.setattr(bench, "DUMP_MAX_POINTS", 1000)
    pts = _cloud(np.random.default_rng(3), 5000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"frame_counts": np.array([3, 0, 7], np.uint32), "cloud": pts})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["cloud_index.npy", "cloud_rgb.npy", "cloud_xyz.npy", "frame_counts.npy"]
    out = {}
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
        out[f[:-4]] = a
    idx = out["cloud_index"].astype(np.int64)
    assert len(idx) == 1000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(out["cloud_xyz"], np.stack([pts["x"][idx], pts["y"][idx], pts["z"][idx]], 1))
    assert np.array_equal(out["cloud_rgb"].astype(np.uint32), pts["rgb"][idx])
    assert out["frame_counts"].tolist() == [3, 0, 7]


@pytest.mark.parametrize("world", [1, 3])
def test_dump_outputs_of_all_ranks_stay_under_64_mb(tmp_path, world):
    """Every rank writes its shard into the same directory: with each shard larger than its share of the cap, the files of all
    ranks together stay under 64 MB."""
    rng = np.random.default_rng(4)
    n = bench.DUMP_MAX_POINTS // world + 100_000
    for r in range(world):
        bench.dump_outputs(str(tmp_path), {"frame_counts": np.arange(50, dtype=np.uint32), "cloud": _cloud(rng, n)}, r, world)
    files = os.listdir(tmp_path)
    assert len(files) == 4 * world
    assert sum(os.path.getsize(tmp_path / f) for f in files) < 64e6
    xyz = [np.load(tmp_path / f, mmap_mode="r") for f in files if "cloud_xyz" in f]
    assert len(xyz) == world and all(len(a) == bench.DUMP_MAX_POINTS // world for a in xyz)


@pytest.mark.timeout(600)
def test_reference_arm_prints_the_contract_line_on_a_tiny_sample():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-frames", "2"], capture_output=True, text=True, timeout=590)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "frames_per_sec" and line["higher_is_better"] is True
    assert line["config"] == bench.static_config("config2_semidense_720p", 1)
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
