"""State a fused cycle leaves behind on the device: counters, tickets, cursors, look-back words and the uploaded pass-through
guesses are reused from one call to the next (most are reset by the fills of the next batch, the guesses only re-uploaded
when they change).  A context that has gone through a record-list rerun (TV_FLAG_SPACE), a window widening
(TV_FLAG_RANGE), a pass-through misguess (TV_FLAG_PASS), a refused call or clearCloud must afterwards give the same cloud,
bit for bit, as a fresh context on the same frames.  Also: the launches of a steady-state fused cycle, and that every
kernel of the library waits for its predecessor before it touches memory (the library launches with programmatic
dependent launch).

The rerun cases run in a process of their own (this file is also the worker) with O3R_TRACE=1, so that the test can see
from stderr that the flag it is about was raised."""
import glob
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import test_gpu_fused_edges as fe  # noqa: E402
from online_3d_reconstruction_b200 import abi, synth  # noqa: E402
from online_3d_reconstruction_b200.lib import O3RError  # noqa: E402
from online_3d_reconstruction_b200.pose import Pose  # noqa: E402

FUSED = abi.MERGE_ACCUMULATE_FUSED
CSRC = os.path.join(ROOT, "online_3d_reconstruction_b200", "csrc")
# launch_count() of one steady-state cycle of _steady_cycles: frames call (frame descriptors, one fill, k_tv, tile-count
# scan, compaction, partial-count update), merge (one fill, layout, key, plan, radix passes, heads, scan, reduce, update, scan,
# place new / old, finish) and the combined downsample (count, scan, emit)
STEADY_LAUNCH_BOUND = 24


def _run(p, cycles, disturb=None):
    """createCycleClouds over `cycles` (lists of frames) -> (per-cycle counts, exportCells(), downsamplePtCloud()).
    `disturb(P)` runs first on the same context."""
    with Pose(p) as P:
        if disturb:
            disturb(P)
        counts = [P.createCycleClouds(c).copy() for c in cycles]
        engines = P.lastCycleEngine()
        return counts, P.exportCells(), P.downsamplePtCloud(), engines


def _same_as_fresh(p, cycles, disturb):
    a = _run(p, cycles, disturb)
    b = _run(p, cycles)
    for ca, cb in zip(a[0], b[0]):
        assert np.array_equal(ca, cb)
    assert a[1].tobytes() == b[1].tobytes(), "resident cells differ from a fresh context's"
    assert a[2].tobytes() == b[2].tobytes(), "combined cloud differs from a fresh context's"
    assert a[3] == b[3] == fe.TILE, (a[3], b[3])


def _synth(seed, n, rows=128, cols=256, keep=None, start=0):
    return [abi.make_frame(d, img, T, keep=keep) for d, img, T in synth.sequence(seed, n, rows, cols, traj_start=start)]


# ------------------------------------------------------------------------------------------------------------ worker cases
def _space_frames(keep):
    rows, cols = 128, 256
    p = abi.make_params(rows=rows, cols=cols, jump_pixels=1, voxel_size=0.013, merge_mode=FUSED)
    rng = np.random.default_rng(5)
    small = np.zeros((rows, cols), np.uint8)
    small[40:50, 100:110] = 100
    wall = np.zeros((rows, cols), np.uint8)
    wall[p.bounding_box:rows - p.bounding_box, p.cols_start_aft_cutout:cols - p.bounding_box] = 100
    first = [abi.make_frame(small, fe._bgr(rng, rows, cols), fe._eye(0.0, 0.0, 1.0), keep=keep)]
    dense = [abi.make_frame(wall, fe._bgr(rng, rows, cols), fe._eye(0.003 * q, 0.002 * q, 1.0), keep=keep) for q in range(2)]
    more = [abi.make_frame(wall, fe._bgr(rng, rows, cols), fe._eye(0.001, 0.004, 1.0), keep=keep)]
    return p, first, dense, more


def case_space():
    """A small batch sizes the record lists; the dense one overflows them (rerun); then the map is cleared and the dense
    batches run again on the grown lists."""
    keep = []
    p, first, dense, more = _space_frames(keep)

    def disturb(P):
        P.createCycleClouds(first)
        P.createCycleClouds(dense)
        P.clearCloud()
    _same_as_fresh(p, [dense, more], disturb)


def case_range():
    """R = 2 serves a batch; the next one raises TV_FLAG_RANGE and reruns with R = 3; cleared, the same batch again."""
    keep = []
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=fe.R_VOXEL[2], merge_mode=FUSED)
    seq = synth.sequence(320, 3, 128, 256)
    near = seq[1][0].copy()
    near[30:70, 60:200] = 195
    near[40:50, 90:110] = 196
    f0 = abi.make_frame(seq[0][0], seq[0][1], seq[0][2], keep=keep)
    rest = [abi.make_frame(near, seq[1][1], seq[1][2], keep=keep), abi.make_frame(seq[2][0], seq[2][1], seq[2][2], keep=keep)]

    def disturb(P):
        P.createCycleClouds([f0])
        P.createCycleClouds(rest)
        P.clearCloud()
    _same_as_fresh(p, [rest, [f0]], disturb)


def case_pass():
    """A batch whose pass-through guess is wrong (TV_FLAG_PASS, rerun with the exact verdicts); cleared, a batch whose
    guesses differ again, then the first one."""
    keep = []
    p, first, dense, more = _space_frames(keep)

    def disturb(P):
        P.createCycleClouds(first)
        P.clearCloud()
    _same_as_fresh(p, [first, more, first], disturb)


def _traced(case):
    env = dict(os.environ, O3R_TRACE="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), case], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "CASE OK" in r.stdout, (r.stdout[-3000:], r.stderr[-6000:])
    return [int(m) for m in re.findall(r"tile engine flags (\d+) \(R \d+\)", r.stderr)]


@pytest.mark.gpu
@pytest.mark.parametrize("case,flag", [("case_space", fe.FLAG_SPACE), ("case_range", fe.FLAG_RANGE), ("case_pass", fe.FLAG_PASS)])
def test_rerun_leaves_no_state(case, flag):
    flags = _traced(case)
    assert any(f & flag for f in flags), flags


# ------------------------------------------------------------------------------------------------------------ in process
@pytest.mark.gpu
def test_refused_call_leaves_no_state():
    """A batch refused for cells beyond +-2^20 between two good ones: the context goes on as if it had never seen it.  The
    refused batch is built like the good one (four patch frames on the x / y cell limits, one step further out), so that the
    engine policy its verdict teaches the context is the one the good batch teaches."""
    keep = []
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED, min_disparity=4.0)
    ok, over = [], []
    for axis in (0, 1):
        for sign in (1, -1):
            ok.append(fe._place(p, keep, 6, axis, sign * fe.LIM))
            over.append(fe._place(p, keep, 6, axis, sign * (fe.LIM + 1)))
    with Pose(p) as P:
        P.createCycleClouds(ok)
        with pytest.raises(O3RError):
            P.createCycleClouds(over)
        P.createCycleClouds(ok)
        got = P.exportCells(), P.downsamplePtCloud(), P.lastCycleEngine()
    with Pose(p) as P:
        P.createCycleClouds(ok)
        P.createCycleClouds(ok)
        ref = P.exportCells(), P.downsamplePtCloud(), P.lastCycleEngine()
    assert got[2] == ref[2], (got[2], ref[2])
    assert got[0].tobytes() == ref[0].tobytes() and got[1].tobytes() == ref[1].tobytes()


@pytest.mark.gpu
def test_clear_cloud_leaves_no_state():
    keep = []
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED)
    a, b = _synth(21, 4, keep=keep), _synth(22, 4, keep=keep, start=4)

    def disturb(P):
        P.createCycleClouds(a)
        P.downsamplePtCloud()
        P.clearCloud()
    _same_as_fresh(p, [b, a], disturb)


@pytest.mark.gpu
def test_steady_state_fused_cycle_launches():
    """Steady state of a fused cycle (inputs on the device, as bench.py times it): at most STEADY_LAUNCH_BOUND launches, the
    same number every cycle."""
    import torch
    keep = []
    p = abi.make_params(rows=128, cols=256, jump_pixels=1, voxel_size=0.05, merge_mode=FUSED)
    seq = synth.sequence(31, 8, 128, 256)
    d_disp = [torch.from_numpy(d).cuda() for d, _, _ in seq]
    d_bgr = [torch.from_numpy(img).cuda() for _, img, _ in seq]
    torch.cuda.synchronize()
    host = [abi.make_frame(d, img, T, keep=keep) for d, img, T in seq]
    for f, dd, db in zip(host, d_disp, d_bgr):
        f.disp, f.bgr = dd.data_ptr(), db.data_ptr()
    per = []
    with Pose(p) as P:
        for c in range(8):
            l0 = P.launch_count()
            P.createCycleClouds(host[c:c + 1] * 4, device_pointers=True)
            P.downsamplePtCloudDevice()
            per.append(P.launch_count() - l0)
        assert P.lastCycleEngine() == fe.TILE
    steady = per[3:]
    print("launches per cycle", per)
    assert len(set(steady)) == 1 and steady[0] <= STEADY_LAUNCH_BOUND, per


# ------------------------------------------------------------------------------------------------------------ CPU
KERNEL = re.compile(r"__global__\b")


def test_every_kernel_waits_for_its_predecessor_first():
    """Every __global__ of csrc begins its body with wait_prior(): with programmatic dependent launch, a kernel that touched
    memory before it could read what its predecessor has not written yet, and one kernel without it would break the
    chain for every later one."""
    n = 0
    for path in sorted(glob.glob(os.path.join(CSRC, "*.cu*"))):
        src = open(path).read()
        for m in KERNEL.finditer(src):
            if "//" in src[src.rfind("\n", 0, m.start()) + 1:m.start()]:
                continue   # (a comment)
            i, depth = m.end(), 0
            while not (depth == 0 and src[i] in "{;"):
                depth += {"(": 1, ")": -1}.get(src[i], 0)
                i += 1
            if src[i] == ";":
                continue   # a declaration
            line = src.count("\n", 0, m.start()) + 1
            assert src[i + 1:].lstrip().startswith("wait_prior();"), f"{os.path.basename(path)}:{line}: kernel does not start with wait_prior()"
            n += 1
    assert n >= 60, n
    launch = open(os.path.join(CSRC, "host_ctx.cuh")).read()
    assert "cudaLaunchAttributeProgrammaticStreamSerialization" in launch


if __name__ == "__main__":
    globals()[sys.argv[1]](*sys.argv[2:])
    print("CASE OK", flush=True)
