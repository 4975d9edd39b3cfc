"""Map checkpoint files (.o3rmap): the resident map of a context written to disk and loaded into another, the same bytes as
host/mapfile.hpp writes and reads.

Layout, little-endian: a 64-byte header, then n_records records.

    offset  field       type
    0       magic       8 bytes "O3RMAP01"
    8       version     u32, 1
    12      kind        u32: 1 = cells (abi.CELL, 40 B: o3r_cloud_export_cells), 2 = points (abi.POINT, 16 B: cloud_big)
    16      voxel_size  f64, the o3r_params value the map was built with
    24      world       u32 \\ the shard the file came from
    28      rank        u32 /
    32      n_records   u64
    40      reserved    zero up to byte 64

A loader refuses a bad magic or version, a file whose size is not 64 + n_records * record size, a kind the context's merge
mode cannot take, and a voxel_size that differs bit for bit from the context's (cell keys mean nothing on another grid).
"""
import os

import numpy as np

from . import abi, exchange

MAGIC = b"O3RMAP01"
VERSION = 1
KIND_CELLS, KIND_POINTS = 1, 2
HEADER_BYTES = 64
HEADER = np.dtype([("magic", "S8"), ("version", "<u4"), ("kind", "<u4"), ("voxel_size", "<f8"), ("world", "<u4"),
                   ("rank", "<u4"), ("n_records", "<u8"), ("reserved", "V24")])
RECORD = {KIND_CELLS: abi.CELL, KIND_POINTS: abi.POINT}
assert HEADER.itemsize == HEADER_BYTES


class MapFileError(ValueError):
    pass


def kind_for(params):
    """The record kind a context keeps: points in MERGE_RETAIN and with dont_downsample, cells otherwise."""
    return KIND_POINTS if params.dont_downsample or params.merge_mode == abi.MERGE_RETAIN else KIND_CELLS


def write(path, kind, records, voxel_size, world=1, rank=0):
    records = np.ascontiguousarray(records, dtype=RECORD[kind])
    h = np.zeros(1, dtype=HEADER)
    h["magic"], h["version"], h["kind"] = MAGIC, VERSION, kind
    h["voxel_size"], h["world"], h["rank"], h["n_records"] = voxel_size, world, rank, records.size
    with open(path, "wb") as f:
        f.write(h.tobytes())
        f.write(records.tobytes())


def read(path):
    """-> (header record, records).  Raises MapFileError for a malformed file."""
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        raw = f.read(HEADER_BYTES)
        if len(raw) < HEADER_BYTES:
            raise MapFileError(f"{path}: {size} bytes, shorter than the 64-byte header")
        h = np.frombuffer(raw, dtype=HEADER)[0]
        if h["magic"] != MAGIC:
            raise MapFileError(f"{path}: not a map file (magic {bytes(h['magic'])!r})")
        if h["version"] != VERSION:
            raise MapFileError(f"{path}: map file version {int(h['version'])}, this build reads {VERSION}")
        kind = int(h["kind"])
        if kind not in RECORD:
            raise MapFileError(f"{path}: unknown record kind {kind}")
        rec = RECORD[kind]
        n = int(h["n_records"])
        if size != HEADER_BYTES + n * rec.itemsize:
            raise MapFileError(f"{path}: {size} bytes, the header announces {n} records = {HEADER_BYTES + n * rec.itemsize}")
        data = np.frombuffer(f.read(n * rec.itemsize), dtype=rec)
    return h, data


def read_for(paths, kind, voxel_size, world=1, rank=0):
    """The records of one or several map files that a context of `kind` and `voxel_size` takes, as rank `rank` of `world`:
    cell files are concatenated in the given order and re-split by owner (exchange.owner_of(key, world) == rank), so a map
    saved on N GPUs reloads on M.  Point files are concatenated (a point cloud is not sharded)."""
    if isinstance(paths, (str, os.PathLike)):
        paths = [paths]
    parts = []
    for p in paths:
        h, data = read(p)
        if int(h["kind"]) != kind:
            raise MapFileError(f"{p}: holds {'cells' if int(h['kind']) == KIND_CELLS else 'points'}, the context keeps "
                               f"{'cells' if kind == KIND_CELLS else 'points'} (merge mode / dont_downsample differ)")
        if np.float64(h["voxel_size"]).tobytes() != np.float64(voxel_size).tobytes():
            raise MapFileError(f"{p}: saved at voxel_size {float(h['voxel_size'])!r}, the context uses {float(voxel_size)!r}")
        parts.append(data)
    recs = np.concatenate(parts) if parts else np.zeros(0, dtype=RECORD[kind])
    if kind == KIND_CELLS and world > 1:
        recs = recs[exchange.owner_of(recs["key"], world) == rank]
    return recs


def save(path, pose):
    """Writes pose's resident map: cells (exportCells) in the accumulate modes, cloud_big (exportPoints) otherwise."""
    kind = kind_for(pose.params)
    recs = pose.exportCells() if kind == KIND_CELLS else pose.exportPoints()
    write(path, kind, recs, pose.params.voxel_size, pose.world, pose.rank)
    return len(recs)


def load(paths, pose):
    """Loads one or several map files into pose (importCells / appendPoints); returns the records merged."""
    kind = kind_for(pose.params)
    recs = read_for(paths, kind, pose.params.voxel_size, pose.world, pose.rank)
    if kind == KIND_CELLS:
        pose.importCells(recs)
    else:
        pose.appendPoints(recs)
    return len(recs)
