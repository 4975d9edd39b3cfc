"""Worker of tests/test_gpu_fused_edges.py: runs one of its cases in a process of its own, so that the test can switch on
O3R_TRACE (read once per process) and read from stderr which window radius, rerun flags and engine served each batch.

    python tests/fused_edges_worker.py <case function> [args...]

The case does all its own comparisons against the oracle; a failed one exits non-zero."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import test_gpu_fused_edges as cases  # noqa: E402

if __name__ == "__main__":
    getattr(cases, sys.argv[1])(*sys.argv[2:])
    print("CASE OK", flush=True)
