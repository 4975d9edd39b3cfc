"""Host mirrors of the multi-GPU split on CPU: frame sharding and the owner hash the device uses to assign cells to
ranks."""
import numpy as np

from online_3d_reconstruction_b200 import abi, exchange


def _make_cells(rank, n, seed=0):
    rng = np.random.default_rng(seed + rank)
    c = np.zeros(n, dtype=abi.CELL)
    i = rng.integers(-300, 300, n) + (1 << 20)
    j = rng.integers(-200, 500, n) + (1 << 20)
    c["key"] = (np.uint64(1 << 20) << np.uint64(42)) | (j.astype(np.uint64) << np.uint64(21)) | i.astype(np.uint64)
    c["sx"], c["sy"], c["sz"] = rng.normal(size=(3, n)).astype(np.float32)
    c["n"] = rng.integers(1, 50, n)
    c["sr"], c["sg"], c["sb"] = rng.integers(0, 255 * 50, (3, n))
    return c


def test_frame_sharding_covers_the_cycle_once():
    for world in (1, 2, 4, 8):
        seen = sorted(f for r in range(world) for f in exchange.shard_frames(50, r, world))
        assert seen == list(range(50))
        assert max(len(exchange.shard_frames(50, r, world)) for r in range(world)) - \
            min(len(exchange.shard_frames(50, r, world)) for r in range(world)) <= 1


def test_owner_hash_is_uniform_and_stable():
    keys = _make_cells(0, 100000)["key"]
    for world in (2, 4, 8):
        cnt = np.bincount(exchange.owner_of(keys, world), minlength=world)
        assert cnt.min() > 0.9 * len(keys) / world
    # known answers of the splitmix64 finaliser (the device uses the same constants)
    assert int(exchange.hash64(np.uint64(1))) == 0x5692161D100B05E5
    assert int(exchange.hash64(np.uint64(0))) == 0
