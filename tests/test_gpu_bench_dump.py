"""bench.py --dump-outputs on the GPU: the combined cloud of the last timed step is read back from the context's device result
buffer (or, with --dont_downsample, the cycle's points from the context), and two runs with the same arguments write identical
files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, workload):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--workload", workload,
           "--no-cpu-baseline", "--parity-steps", "0", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.timeout(1300)
@pytest.mark.parametrize("workload", ["config2_semidense_720p", "config3_dont_downsample_720p"])
def test_dump_outputs_read_back_and_reproducible(tmp_path, workload):
    line, a = _bench(tmp_path / "a", workload)
    _, b = _bench(tmp_path / "b", workload)
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert line["steps"] == 2 and line["warmup"] == 1
    counts = a["frame_counts"]
    F = line["config"]["frames_per_step"]
    # the per-frame counts of a cycle do not depend on the leg: the last profiled step ran the same cycle
    assert counts.shape == (F,) and counts.sum() == line["run"]["per_frame_voxels_per_step_per_gpu"]
    if line["config"]["dont_downsample"]:
        xyz, rgb, idx = a["cycle_points_xyz"], a["cycle_points_rgb"], a["cycle_points_index"]
        assert counts.sum() > len(xyz) == len(idx) == len(rgb)            # sampled: the cycle has ~37 M points
        assert np.all(np.diff(idx) > 0) and idx[-1] < counts.sum()
    else:
        xyz, rgb = a["cloud_xyz"], a["cloud_rgb"]
        assert "cloud_index" not in a
        # as many cells as the host entry point returned for the same cycles in the end-to-end leg (16 B a cell + 4 B a frame)
        assert len(xyz) == (line["e2e"]["d2h_bytes_per_step"] - 4 * F) // 16 > 10000
    assert xyz.dtype == np.float32 and xyz.shape[1] == 3 and np.all(np.isfinite(xyz))
    assert rgb.dtype == np.float64 and np.all(rgb < (1 << 24)) and np.all(rgb == np.floor(rgb))
