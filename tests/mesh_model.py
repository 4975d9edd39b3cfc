"""Plain numpy model of o3r_cloud_mesh (csrc/mesh.cuh), from a map's exported cells.

  * vertices: the cells with n >= min_points in key order, each at its float32 centroid (register_model.MapModel), which is
    o3r_cloud_downsample's output
  * quads A = (i, j), B = (i+1, j), C = (i, j+1), D = (i+1, j+1) at one k, of vertices only; neighbours beyond +-(2^20 - 1)
    do not exist.  Four vertices: split along A-D when |zA - zD| <= |zB - zC| (float32) -> (A, B, D), (A, D, C), else
    (A, B, C), (B, D, C).  Three: A missing (B, D, C), B missing (A, D, C), C missing (A, B, D), D missing (A, B, C)
  * gate: a triangle is kept iff max |dz| over its pairs (float32), as a float64, is <= max_step
  * order: by the key of the quad's A corner, then the order above; a vertex emits the quad to its left (when (i-1, j) is
    not a vertex) and then its own
  * normals: register_model's plane fit at the vertex, n = (-a, -b, 1) / |.| in float64, rounded to float32; (0, 0, 0)
    without a fit

Every step is the kernel's operation sequence (float32 compares, float64 fit without contraction), so the GPU must agree
bit for bit.
"""
import numpy as np

import reduce_model as rm
import register_model as reg

F32 = np.float32
LIM = (1 << 20) - 1
B20 = 1 << 20


def decode(keys):
    """-> (i, j, k) int64 of 64-bit cell keys."""
    keys = np.asarray(keys, dtype=np.uint64)
    m = np.uint64((1 << 21) - 1)
    i = (keys & m).astype(np.int64) - B20
    j = ((keys >> np.uint64(21)) & m).astype(np.int64) - B20
    k = (keys >> np.uint64(42)).astype(np.int64) - B20
    return i, j, k


def _vertex_at(M, i, j, k):
    """Vertex index of cells (i, j, k), -1 where there is none or the cell is outside +-(2^20 - 1)."""
    ok = (i >= -LIM) & (i <= LIM) & (j >= -LIM) & (j <= LIM)
    pr, at = M.lookup(np.where(ok, i, 0), np.where(ok, j, 0), k)
    return np.where(pr & ok, at, -1)


def _quad(z, A, Bv, Cv, D):
    """Triangles of quads with corners A, B, C, D (-1 = absent) -> (t0, t1: (n, 3) int64, ok0, ok1 masks)."""
    pres = (A >= 0).astype(int) + (Bv >= 0) + (Cv >= 0) + (D >= 0)
    za, zb, zc, zd = (z[np.maximum(x, 0)] for x in (A, Bv, Cv, D))
    full = pres == 4
    ad = np.abs(za - zd) <= np.abs(zb - zc)
    t0 = np.where(ad[:, None], np.stack([A, Bv, D], 1), np.stack([A, Bv, Cv], 1))
    t1 = np.where(ad[:, None], np.stack([A, D, Cv], 1), np.stack([Bv, D, Cv], 1))
    three = np.where((A < 0)[:, None], np.stack([Bv, D, Cv], 1),
                     np.where((Bv < 0)[:, None], np.stack([A, D, Cv], 1),
                              np.where((Cv < 0)[:, None], np.stack([A, Bv, D], 1), np.stack([A, Bv, Cv], 1))))
    t0 = np.where(full[:, None], t0, three)
    return t0, t1, pres >= 3, full


def _gate(z, t, max_step):
    a, b, c = z[t[:, 0]], z[t[:, 1]], z[t[:, 2]]
    m = np.maximum(np.maximum(np.abs(a - b), np.abs(b - c)), np.abs(a - c))
    return m.astype(np.float64) <= max_step


def triangles(M, max_step=np.inf):
    """-> (m, 3) uint32 vertex indices of o3r_cloud_mesh's triangles, in its order."""
    n = len(M.keys)
    if n == 0:
        return np.zeros((0, 3), np.uint32)
    z = M.cz.astype(F32)
    i, j, k = decode(M.keys)
    a = np.arange(n, dtype=np.int64)
    left = _vertex_at(M, i - 1, j, k)
    right = _vertex_at(M, i + 1, j, k)
    ul, up, ur = (_vertex_at(M, i + d, j + 1, k) for d in (-1, 0, 1))
    none = np.full(n, -1, np.int64)
    # slots per vertex: the left quad's triangle (A missing: at most one), then the own quad's two
    l0, _, lok0, _ = _quad(z, none, a, ul, up)
    o0, o1, ook0, ook1 = _quad(z, a, right, up, ur)
    lok0 &= left < 0
    T = np.stack([l0, o0, o1], 1)                      # (n, 3 slots, 3)
    ok = np.stack([lok0, ook0, ook1], 1)
    flat, okf = T.reshape(-1, 3), ok.reshape(-1)
    t = flat[okf]
    t = t[_gate(z, t, max_step)]
    return t.astype(np.uint32)


def normals(M):
    """-> (n, 3) float32 vertex normals: the registration's plane fit at each vertex's cell, (0, 0, 0) without one."""
    n = len(M.keys)
    out = np.zeros((n, 3), F32)
    if n == 0:
        return out
    i, j, k = decode(M.keys)
    x0, y0, z0 = M.cx.astype(np.float64), M.cy.astype(np.float64), M.cz.astype(np.float64)
    S = {q: np.zeros(n) for q in ("uu", "uw", "u", "ww", "w", "1", "uh", "wh", "h")}
    for dj in (0, -1, 1):
        for di in (-1, 0, 1):
            at = _vertex_at(M, i + di, j + dj, k)
            pr = at >= 0
            at = np.maximum(at, 0)
            u = M.cx[at].astype(np.float64) - x0
            w = M.cy[at].astype(np.float64) - y0
            h = M.cz[at].astype(np.float64) - z0
            for q, val in (("uu", u * u), ("uw", u * w), ("u", u), ("ww", w * w), ("w", w), ("1", np.ones_like(u)),
                           ("uh", u * h), ("wh", w * h), ("h", h)):
                S[q] = S[q] + np.where(pr, val, 0.0)
    Suu, Suw, Su, Sww, Sw, S1, Suh, Swh, Sh = (S[q] for q in ("uu", "uw", "u", "ww", "w", "1", "uh", "wh", "h"))
    with np.errstate(divide="ignore", invalid="ignore"):
        c00 = Sww * S1 - Sw * Sw
        c01 = Sw * Su - Suw * S1
        c02 = Suw * Sw - Sww * Su
        c11 = Suu * S1 - Su * Su
        c12 = Su * Suw - Suu * Sw
        det = Suu * c00 + Suw * c01 + Su * c02
        inside = (np.abs(i) <= LIM - 1) & (np.abs(j) <= LIM - 1)
        fit = inside & (S1 >= 3.0) & (det > reg.FIT_COND * Suu * Sww * S1)
        a = (c00 * Suh + c01 * Swh + c02 * Sh) / det
        b = (c01 * Suh + c11 * Swh + c12 * Sh) / det
        nn = np.sqrt(a * a + b * b + 1.0)
        nrm = np.stack([-a / nn, -b / nn, 1.0 / nn], 1).astype(F32)
    out[fit] = nrm[fit]
    return out


def mesh(cells, v, min_points=1, max_step=np.inf):
    """-> (vertices as (x, y, z) float32 columns via MapModel, normals, triangles) of the map given by abi.CELL records."""
    M = reg.MapModel(cells, v, min_points)
    return M, normals(M), triangles(M, max_step)


def cells_at(ijk, z=None, n=1, v=1.0):
    """abi.CELL records of hand-placed cells: (i, j, k) triples, centroid at the cell's (i + 0.5, j + 0.5) v and height z
    (default 0.25 + the cell's k band), n points each (sums n * centroid, exact for these values)."""
    from online_3d_reconstruction_b200 import abi
    ijk = np.asarray(ijk, dtype=np.int64).reshape(-1, 3)
    zz = np.zeros(len(ijk)) + 0.25 if z is None else np.asarray(z, dtype=np.float64)
    zz = zz + ijk[:, 2] * 1000.0
    c = np.zeros(len(ijk), dtype=abi.CELL)
    c["key"] = rm.cell_keys(ijk[:, 0], ijk[:, 1], ijk[:, 2])
    c["n"] = n
    c["sx"] = ((ijk[:, 0] + 0.5) * v * n).astype(F32)
    c["sy"] = ((ijk[:, 1] + 0.5) * v * n).astype(F32)
    c["sz"] = ((zz + 500.0) * n).astype(F32)
    return np.sort(c, order="key")
