"""Host mirrors of the multi-GPU split (SURVEY §8e): one process per GPU, frames sharded f mod P, and each
combined-grid cell owned by the rank hash64(key) mod P names.  The exchange itself runs inside libo3r.so
(o3r_comm_init / o3r_exchange_cycle); this module lets a caller or a test compute the same split on the host.
"""
import numpy as np


def hash64(x):
    """splitmix64 finaliser — host mirror of the device hash that assigns a cell key to its owner rank."""
    x = np.asarray(x, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xbf58476d1ce4e5b9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94d049bb133111eb)
        x ^= x >> np.uint64(31)
    return x


def owner_of(keys, world):
    return (hash64(keys) % np.uint64(world)).astype(np.int64)


def shard_frames(n_frames, rank, world):
    """Indices of the cycle's frames this rank reconstructs (frame f -> rank f mod P)."""
    return list(range(rank, n_frames, world))


def unshard_points(shards, counts, world):
    """Sharded RETAIN: the ranks' own points (pass-through grid, dont_downsample) -> the single-GPU cloud_big order.

    shards[r] = rank r's points in its local order; counts[r] = its per-cycle arrays of per-frame point counts (what
    createCycleClouds returned, an empty array for a cycle without frames).  Cycle by cycle, global frame f = i*world + r
    is rank r's i-th frame of that cycle, so the frames are taken in order f = 0, 1, ... from rank f mod world."""
    at = [0] * world
    parts = []
    for s in range(len(counts[0])):
        n_frames = sum(len(counts[r][s]) for r in range(world))
        for f in range(n_frames):
            r, i = f % world, f // world
            c = int(counts[r][s][i])
            parts.append(shards[r][at[r]:at[r] + c])
            at[r] += c
    assert all(at[r] == len(shards[r]) for r in range(world)), "counts do not cover the shards"
    return np.concatenate(parts) if parts else np.zeros(0, dtype=shards[0].dtype)
