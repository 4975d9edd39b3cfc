"""Map checkpoint files (online_3d_reconstruction_b200/mapfile.py) on the CPU: layout, refusals and re-sharding."""
import struct

import numpy as np
import pytest

from online_3d_reconstruction_b200 import abi, exchange, mapfile


def _cells(n, seed):
    rng = np.random.default_rng(seed)
    c = np.zeros(n, dtype=abi.CELL)
    B = 1 << 20
    i, j, k = (rng.integers(-5000, 5000, n) + B for _ in range(3))
    c["key"] = (k.astype(np.uint64) << np.uint64(42)) | (j.astype(np.uint64) << np.uint64(21)) | i.astype(np.uint64)
    c["n"] = rng.integers(1, 300, n)
    c["sx"], c["sy"], c["sz"] = (rng.normal(0, 50, n).astype(np.float32) for _ in range(3))
    for ch in ("sr", "sg", "sb"):
        c[ch] = rng.integers(0, 256, n) * c["n"] // 2
    return c


def test_round_trip_and_header_offsets(tmp_path):
    cells = _cells(1000, 1)
    path = str(tmp_path / "a.o3rmap")
    mapfile.write(path, mapfile.KIND_CELLS, cells, 0.05, world=4, rank=3)
    raw = open(path, "rb").read()
    assert len(raw) == 64 + 40 * len(cells)
    assert raw[0:8] == b"O3RMAP01"
    assert struct.unpack_from("<IId", raw, 8) == (1, 1, 0.05)
    assert struct.unpack_from("<IIQ", raw, 24) == (4, 3, len(cells))
    assert raw[40:64] == bytes(24)
    assert raw[64:] == cells.tobytes()
    h, back = mapfile.read(path)
    assert (int(h["world"]), int(h["rank"]), float(h["voxel_size"])) == (4, 3, 0.05)
    assert back.tobytes() == cells.tobytes()
    pts = np.zeros(7, dtype=abi.POINT)
    pts["x"] = np.arange(7, dtype=np.float32)
    pts["rgb"] = 0x00112233
    pp = str(tmp_path / "p.o3rmap")
    mapfile.write(pp, mapfile.KIND_POINTS, pts, 0.1)
    raw = open(pp, "rb").read()
    assert len(raw) == 64 + 16 * 7 and struct.unpack_from("<I", raw, 12) == (2,)
    assert mapfile.read_for(pp, mapfile.KIND_POINTS, 0.1).tobytes() == pts.tobytes()
    assert mapfile.kind_for(abi.make_params(merge_mode=abi.MERGE_RETAIN)) == mapfile.KIND_POINTS
    assert mapfile.kind_for(abi.make_params(dont_downsample=True)) == mapfile.KIND_POINTS
    assert mapfile.kind_for(abi.make_params(merge_mode=abi.MERGE_ACCUMULATE_FUSED)) == mapfile.KIND_CELLS


def test_refusals(tmp_path):
    cells = _cells(10, 2)
    good = str(tmp_path / "g.o3rmap")
    mapfile.write(good, mapfile.KIND_CELLS, cells, 0.05)
    raw = open(good, "rb").read()
    cases = {"truncated": raw[:-1], "magic": b"O3RMAP02" + raw[8:], "version": raw[:8] + struct.pack("<I", 2) + raw[12:],
             "header": raw[:40], "kind": raw[:12] + struct.pack("<I", 3) + raw[16:]}
    for name, data in cases.items():
        p = tmp_path / f"{name}.o3rmap"
        p.write_bytes(data)
        with pytest.raises(mapfile.MapFileError):
            mapfile.read_for(str(p), mapfile.KIND_CELLS, 0.05)
    with pytest.raises(mapfile.MapFileError, match="voxel_size"):
        mapfile.read_for(good, mapfile.KIND_CELLS, 0.1)
    with pytest.raises(mapfile.MapFileError, match="voxel_size"):   # bit for bit: one ulp off is another grid
        mapfile.read_for(good, mapfile.KIND_CELLS, float(np.nextafter(0.05, 1.0)))
    with pytest.raises(mapfile.MapFileError, match="points"):
        mapfile.read_for(good, mapfile.KIND_POINTS, 0.05)


def test_resplit_two_shards_for_world_1_and_3(tmp_path):
    cells = _cells(5000, 3)
    owner2 = exchange.owner_of(cells["key"], 2)
    paths = []
    for r in range(2):
        paths.append(str(tmp_path / f"s{r}.o3rmap"))
        mapfile.write(paths[-1], mapfile.KIND_CELLS, cells[owner2 == r], 0.05, world=2, rank=r)
    both = np.concatenate([cells[owner2 == 0], cells[owner2 == 1]])
    assert mapfile.read_for(paths, mapfile.KIND_CELLS, 0.05).tobytes() == both.tobytes()   # world 1 keeps everything
    got = [mapfile.read_for(paths, mapfile.KIND_CELLS, 0.05, world=3, rank=r) for r in range(3)]
    for r in range(3):
        assert np.all(exchange.owner_of(got[r]["key"], 3) == r)
        assert got[r].tobytes() == both[exchange.owner_of(both["key"], 3) == r].tobytes()
    assert sum(len(g) for g in got) == len(cells)
    assert np.array_equal(np.sort(np.concatenate(got)["key"]), np.sort(cells["key"]))
