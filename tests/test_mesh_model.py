"""The numpy model of o3r_cloud_mesh (tests/mesh_model.py) on hand-built grids, and against a per-quad loop written straight
from the contract in include/o3r.h.  CPU only."""
import numpy as np

import mesh_model as mm
import register_model as reg

LIM = mm.LIM


def _tris(ijk, z=None, n=1, min_points=1, max_step=np.inf):
    M, nrm, t = mm.mesh(mm.cells_at(ijk, z, n), 1.0, min_points, max_step)
    return M, nrm, [tuple(int(v) for v in row) for row in t]


def _loop(cells, min_points=1, max_step=np.inf):
    """The contract as a loop over quads: every (i, j, k) with a vertex among its corners' A or B."""
    M = reg.MapModel(cells, 1.0, min_points)
    i, j, k = mm.decode(M.keys)
    at = {(int(a), int(b), int(c)): q for q, (a, b, c) in enumerate(zip(i, j, k))}
    z = M.cz
    quads = sorted({(a, b, c) for a, b, c in at} | {(a - 1, b, c) for a, b, c in at if a - 1 >= -LIM},
                   key=lambda q: (q[2], q[1], q[0]))   # key order
    out = []
    for a, b, c in quads:
        A, B, C, D = (at.get(x) for x in ((a, b, c), (a + 1, b, c), (a, b + 1, c), (a + 1, b + 1, c)))
        have = [x is not None for x in (A, B, C, D)]
        if sum(have) == 4:
            if abs(z[A] - z[D]) <= abs(z[B] - z[C]):
                ts = [(A, B, D), (A, D, C)]
            else:
                ts = [(A, B, C), (B, D, C)]
        elif sum(have) == 3:
            ts = [[(B, D, C), (A, D, C), (A, B, D), (A, B, C)][have.index(False)]]
        else:
            ts = []
        for t in ts:
            dz = max(abs(z[t[0]] - z[t[1]]), abs(z[t[1]] - z[t[2]]), abs(z[t[0]] - z[t[2]]))
            if float(dz) <= max_step:
                out.append(t)
    return out


def test_diagonal_rule_and_tie():
    sq = [(0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 0)]     # key order: A, B, C, D
    # |zA - zD| = 0.1 < |zB - zC| = 0.5: A-D
    assert _tris(sq, [0.0, 0.5, 0.0, 0.1])[2] == [(0, 1, 3), (0, 3, 2)]
    # |zA - zD| = 0.5 > |zB - zC| = 0.1: B-C
    assert _tris(sq, [0.0, 0.1, 0.0, 0.5])[2] == [(0, 1, 2), (1, 3, 2)]
    # tie: A-D
    assert _tris(sq, [0.0, 0.25, 0.0, 0.25])[2] == [(0, 1, 3), (0, 3, 2)]


def test_each_missing_corner():
    A, B, C, D = (0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 0)
    assert _tris([B, C, D])[2] == [(0, 2, 1)]          # vertices B=0, C=1, D=2: (B, D, C)
    assert _tris([A, C, D])[2] == [(0, 2, 1)]          # A=0, C=1, D=2: (A, D, C)
    assert _tris([A, B, D])[2] == [(0, 1, 2)]          # A=0, B=1, D=2: (A, B, D)
    assert _tris([A, B, C])[2] == [(0, 1, 2)]          # (A, B, C)
    assert _tris([A, D])[2] == [] and _tris([A, B])[2] == []


def _signed_area(M, t):
    x, y = M.cx.astype(np.float64), M.cy.astype(np.float64)
    a, b, c = t[:, 0], t[:, 1], t[:, 2]
    return (x[b] - x[a]) * (y[c] - y[a]) - (x[c] - x[a]) * (y[b] - y[a])


def test_counter_clockwise_on_terrain():
    mp, _, _ = reg.terrain_scene()
    cells = reg.cells_from_points(mp, 1.0)
    M, nrm, t = mm.mesh(cells, 1.0)
    assert len(t) > 1.9 * len(M.keys)
    assert np.all(_signed_area(M, t.astype(np.int64)) > 0)
    # upward normals where a plane fits, and the same orientation as the faces
    fit = np.any(nrm != 0, axis=1)
    assert fit.mean() > 0.95 and np.all(nrm[fit, 2] > 0)
    assert np.allclose(np.linalg.norm(nrm[fit].astype(np.float64), axis=1), 1.0, atol=1e-6)


def test_gate_cuts_a_cliff():
    ijk = [(a, b, 0) for b in range(3) for a in range(4)]
    z = [0.0 if a < 2 else 5.0 for b in range(3) for a in range(4)]
    M, _, all_t = _tris(ijk, z)
    _, _, gated = _tris(ijk, z, max_step=1.0)
    assert len(all_t) == 12
    assert len(gated) == 8          # the two quads of the column i = 1 .. 2 hang over the cliff
    for t in gated:
        zs = [M.cz[v] for v in t]
        assert max(zs) - min(zs) == 0.0
    _, _, edge = _tris(ijk, z, max_step=5.0)
    assert edge == all_t            # <= is inclusive


def test_order_and_left_quads():
    # a hole at (0, 0) and one at (2, 1): the quad of A = (0, 0) is emitted by B = (1, 0), before (1, 0)'s own quad
    ijk = [(a, b, 0) for b in range(3) for a in range(4) if (a, b) not in ((0, 0), (2, 1))]
    cells = mm.cells_at(ijk)
    M, _, t = mm.mesh(cells, 1.0)
    got = [tuple(int(v) for v in r) for r in t]
    assert got == _loop(cells)
    idx = {tuple(int(v) for v in c): q for q, c in enumerate(zip(*mm.decode(M.keys)))}
    assert got[0] == (idx[(1, 0, 0)], idx[(1, 1, 0)], idx[(0, 1, 0)])   # (B, D, C) of the quad at (0, 0)


def test_sub_threshold_cells_are_not_vertices():
    ijk = [(0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 0)]
    cells = mm.cells_at(ijk)
    cells["n"][3] = 1
    cells["sx"][3], cells["sy"][3], cells["sz"][3] = cells["sx"][3] / 2, cells["sy"][3] / 2, cells["sz"][3] / 2
    for c in range(3):
        cells["n"][c] = 2
        cells["sx"][c], cells["sy"][c], cells["sz"][c] = 2 * cells["sx"][c], 2 * cells["sy"][c], 2 * cells["sz"][c]
    M, nrm, t = mm.mesh(cells, 1.0, min_points=2)
    assert len(M.keys) == 3 and [tuple(r) for r in t] == [(0, 1, 2)]
    assert np.array_equal(t, np.asarray(_loop(cells, 2), np.uint32).reshape(-1, 3))
    assert np.all(nrm[:, 2] > 0)   # three cells fit a plane


def test_different_k_are_separate():
    # the same columns at k = 0 and k = 1: 5 vertices at k = 0 give a full quad and a three-vertex one (3 triangles), the 3
    # at k = 1 one triangle; no triangle joins the two
    ijk = [(0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 0), (2, 0, 0), (0, 0, 1), (1, 0, 1), (0, 1, 1)]
    cells = mm.cells_at(ijk)
    M, _, t = mm.mesh(cells, 1.0)
    _, _, k = mm.decode(M.keys)
    assert len(t) == 4 and all(len(set(k[list(r)])) == 1 for r in t)
    assert [tuple(int(v) for v in r) for r in t] == _loop(cells)


def test_boundary_cells():
    # corners of the key range: 2 x 2 blocks at (+-LIM, +-LIM); no neighbour is formed beyond them
    lo, hi = (-LIM, -LIM + 1), (LIM - 1, LIM)
    ijk = [(a, b, 0) for I in (lo, hi) for J in (lo, hi) for a in I for b in J]
    cells = mm.cells_at(ijk)
    M, nrm, t = mm.mesh(cells, 1.0)
    assert len(M.keys) == 16 and len(t) == 8
    assert [tuple(int(v) for v in r) for r in t] == _loop(cells)
    i, j, _ = mm.decode(M.keys)
    edge = (np.abs(i) == LIM) | (np.abs(j) == LIM)
    assert np.all(nrm[edge] == 0)   # no fit at |i| or |j| = 2^20 - 1
    # each block's inner cell fits its flat 2 x 2 block
    assert edge.sum() == 12 and np.array_equal(nrm[~edge], np.tile(np.float32([0, 0, 1]), (4, 1)))


def test_random_grids_match_the_loop():
    rng = np.random.default_rng(5)
    for trial in range(20):
        keep = rng.random((9, 7, 2)) < rng.uniform(0.3, 0.95)
        ijk = [(a - 4, b - 3, c) for a in range(9) for b in range(7) for c in range(2) if keep[a, b, c]]
        if not ijk:
            continue
        z = rng.normal(0, 1, len(ijk)).astype(np.float32).astype(np.float64)
        if trial % 3 == 0:
            z = np.round(z * 2) / 2   # ties
        cells = mm.cells_at(ijk, z)
        for step in (np.inf, 0.7):
            _, _, t = mm.mesh(cells, 1.0, 1, step)
            assert [tuple(int(v) for v in r) for r in t] == _loop(cells, 1, step), trial
