"""Sharded RETAIN (ICP-on) mode on REAL ranks: N processes, N GPUs, o3r_cloud_transform on every rank and the collective
o3r_cloud_downsample.  The union of the shards is the single-rank RETAIN cloud and the oracle's cloud bit for bit.  Needs
>= 2 devices; tests/test_gpu_retain_sharded.py drives the same path at world size 1."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 4])
def test_n_ranks_retain_equal_one_rank_bit_for_bit(world):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multirank_retain_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MULTIRANK RETAIN OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
