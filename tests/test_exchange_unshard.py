"""Host mirror of the sharded RETAIN frame order on CPU: the ranks' own points (pass-through grid, dont_downsample),
interleaved back cycle by cycle and frame by frame, are the single-GPU cloud_big."""
import numpy as np

from online_3d_reconstruction_b200 import abi, exchange


def test_unshard_points_restores_frame_order_with_ranks_without_frames():
    rng = np.random.default_rng(5)
    per_cycle = [5, 3, 1, 0, 2]
    for world in (1, 2, 4):
        big, shards, counts = [], [[] for _ in range(world)], [[] for _ in range(world)]
        for n in per_cycle:
            cyc = [[] for _ in range(world)]
            for f in range(n):
                pts = np.zeros(int(rng.integers(0, 6)), dtype=abi.POINT)
                pts["x"] = rng.normal(size=pts.size)
                pts["rgb"] = rng.integers(0, 1 << 24, pts.size)
                big.append(pts)
                shards[f % world].append(pts)
                cyc[f % world].append(pts.size)
            for r in range(world):
                counts[r].append(np.array(cyc[r], dtype=np.uint32))
        got = exchange.unshard_points([np.concatenate(s) if s else np.zeros(0, abi.POINT) for s in shards], counts, world)
        assert np.array_equal(got, np.concatenate(big))
