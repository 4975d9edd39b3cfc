"""Map checkpoints of a sharded map on real ranks (tests/multirank_map_worker.py): N-GPU shards reload on one GPU, a rank
refuses cells it does not own, and a resumed multi-rank run equals the uninterrupted one.  Needs >= 2 devices."""
import os
import subprocess
import sys

import pytest

from test_gpu_multirank import _free_port

pytestmark = pytest.mark.gpu
# imported at collection, before any test of the session attaches a communicator: the library loads libnccl.so.2 only when no
# NCCL is in the process yet, and torch must bring its own first
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_map_checkpoints(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multirank_map_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MULTIRANK MAP OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
