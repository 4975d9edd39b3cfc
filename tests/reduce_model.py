"""Plain numpy model of the accumulate modes' combined-grid downsample (engine 2 + k_acc_emit), for clouds where the
oracle's semantics do not apply (channel sums past 2^24, cell extents past PCL's int32 guard).

  * absolute cell (i, j, k) = floor(x * (1/v)), floor(y * (1/v)), floor((z + 500) * (1/1000)), all in float32;
    records ordered by (k, j, i)
  * x, y and z + 500 folded in float32, sequentially, in arrival order
  * colour channels summed exactly as uint32
  * record = (sx / n, sy / n, sz / n - 500, uint32(f32(sum) / f32(n)) per channel); cells with n < min_points dropped
"""
import numpy as np

from online_3d_reconstruction_b200 import abi

F32 = np.float32
B = 1 << 20


def cells(pts, v):
    """-> (i, j, k) int64 absolute combined-grid cells, float32 arithmetic as on the device."""
    ix = F32(1.0) / F32(v)
    iz = F32(1.0) / F32(1000.0)
    zs = pts["z"].astype(F32) + F32(500.0)
    i = np.floor(pts["x"].astype(F32) * ix).astype(np.int64)
    j = np.floor(pts["y"].astype(F32) * ix).astype(np.int64)
    k = np.floor(zs * iz).astype(np.int64)
    return i, j, k


def cell_keys(i, j, k):
    """The library's 64-bit cell key: (k + 2^20) << 42 | (j + 2^20) << 21 | (i + 2^20)."""
    return ((k + B).astype(np.uint64) << np.uint64(42)) | ((j + B).astype(np.uint64) << np.uint64(21)) | \
        (i + B).astype(np.uint64)


def _seq_fold(vals, starts, lens):
    """Sequential float32 left fold of vals[starts[g] : starts[g] + lens[g]] for every group g."""
    out = np.zeros(len(starts), dtype=F32)
    short = lens <= 64
    idx = np.nonzero(short)[0]
    for r in range(int(lens[idx].max()) if len(idx) else 0):
        live = idx[lens[idx] > r]
        out[live] = out[live] + vals[starts[live] + r]   # float32 + float32 -> float32, one rounding per step
    for g in np.nonzero(~short)[0]:
        out[g] = np.add.accumulate(vals[starts[g]:starts[g] + lens[g]], dtype=F32)[-1]
    return out


def accumulate_downsample(pts, v, min_points=1):
    """-> (records abi.POINT in (k, j, i) order, keys u64, counts u32) of the cloud appended in array order."""
    pts = np.ascontiguousarray(pts, dtype=abi.POINT)
    i, j, k = cells(pts, v)
    order = np.lexsort((i, j, k))   # stable: arrival order inside a cell
    key = cell_keys(i, j, k)[order]
    head = np.ones(len(order), dtype=bool)
    head[1:] = key[1:] != key[:-1]
    starts = np.nonzero(head)[0]
    lens = np.diff(np.append(starts, len(order)))
    p = pts[order]
    sx = _seq_fold(p["x"].astype(F32), starts, lens)
    sy = _seq_fold(p["y"].astype(F32), starts, lens)
    sz = _seq_fold(p["z"].astype(F32) + F32(500.0), starts, lens)
    c = p["rgb"].astype(np.uint64)
    csum = [np.add.reduceat((c >> np.uint64(s)) & np.uint64(255), starts).astype(np.uint32) for s in (16, 8, 0)]
    fn = lens.astype(F32)
    keep = lens >= min_points
    out = np.zeros(int(keep.sum()), dtype=abi.POINT)
    out["x"] = (sx / fn)[keep]
    out["y"] = (sy / fn)[keep]
    out["z"] = (sz / fn - F32(500.0))[keep]
    ch = [(s.astype(F32) / fn).astype(np.uint32)[keep] for s in csum]
    out["rgb"] = (ch[0] << np.uint32(16)) | (ch[1] << np.uint32(8)) | ch[2]
    return out, key[starts][keep], lens[keep].astype(np.uint32)


def float_fold_channel(vals):
    """CentroidPoint's colour: a float32 left fold of the channel values, uint32(sum / n)."""
    s = np.add.accumulate(np.asarray(vals, dtype=F32), dtype=F32)[-1]
    return int(np.uint32(s / F32(len(vals))))


def uint_sum_channel(vals):
    """The accumulate modes' colour: an exact integer sum, uint32(f32(sum) / n)."""
    return int(np.uint32(F32(int(np.sum(np.asarray(vals, dtype=np.uint64)))) / F32(len(vals))))
