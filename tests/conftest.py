import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def real(golden_dir):
    """The reference's three real frames (disparity + labels) and what it logged for them, plus a seeded synthetic colour
    plane: colours only travel with the points, nothing compares them with the reference."""
    import numpy as np

    from online_3d_reconstruction_b200 import synth
    g = dict(np.load(os.path.join(golden_dir, "real_frames.npz")))
    g["bgr"] = synth.make_frame_images(np.random.default_rng(1248), 720, 1280)[1]
    return g
