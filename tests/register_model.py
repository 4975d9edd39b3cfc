"""Plain numpy / float64 model of o3r_cloud_register (csrc/register.cuh), from a map's exported cells.

  * the map: cells with n >= min_points; centroid (sx / n, sy / n, sz / n - 500) in float32, as acc_centroid divides
  * a point p' = T p (double, left to right) falls into the combined-grid cell of float32(p') (reduce_model.cells)
  * the plane z - z0 = a (x - x0) + b (y - y0) + d is fitted over the hit cell's centroid (x0, y0, z0) and the centroids
    of its 8 same-k neighbours that are in the map, summed in the order row j, j-1, j+1, each i-1, i, i+1; at least 3
    cells and det > 1e-3 * Suu * Sww * S1, else no normal
  * n = (-a, -b, 1) / |.|, r = n . (p' - c0), inlier when |r| <= max_distance
  * J = ((p' - pivot) x n, n); the 6 x 6 system J^T J x = -J^T r, its rotations scaled to arc lengths at
    L = sqrt(tr(rotation block) / tr(translation block)), is solved by cyclic Jacobi, directions below
    degenerate_ratio * lambda_max dropped; x = (axis-angle about the pivot, translation), composed in double

Per-point arithmetic follows the kernel operation for operation; sums over points are taken in numpy's order, so results
agree with the GPU to rounding of those sums.
"""
import math

import numpy as np

import reduce_model as rm

F32 = np.float32
FIT_COND = 1e-3


def defaults(v):
    return dict(max_iterations=20, max_distance=3.0 * v, min_rotation=1e-5, min_translation=1e-4, degenerate_ratio=1e-3)


class MapModel:
    """The registration target built from abi.CELL records (an o3r_cloud_export_cells result)."""

    def __init__(self, cells, v, min_points):
        cells = np.asarray(cells)
        keep = cells["n"] >= np.uint32(min_points)
        c = cells[keep]
        fn = c["n"].astype(F32)
        self.keys = c["key"].astype(np.uint64)
        self.cx = (c["sx"].astype(F32) / fn).astype(F32)
        self.cy = (c["sy"].astype(F32) / fn).astype(F32)
        self.cz = ((c["sz"].astype(F32) / fn).astype(F32) - F32(500.0)).astype(F32)
        self.v = v

    def lookup(self, i, j, k):
        """-> (present mask, index) of cells (i, j, k) (int64 arrays)."""
        key = rm.cell_keys(i, j, k)
        if len(self.keys) == 0:
            return np.zeros(key.shape, bool), np.zeros(key.shape, np.int64)
        at = np.minimum(np.searchsorted(self.keys, key), len(self.keys) - 1)
        return self.keys[at] == key, at


def _apply(T, P):
    px, py, pz = P[:, 0], P[:, 1], P[:, 2]
    x = T[0] * px + T[1] * py + T[2] * pz + T[3]
    y = T[4] * px + T[5] * py + T[6] * pz + T[7]
    z = T[8] * px + T[9] * py + T[10] * pz + T[11]
    return x, y, z


def linearise(M, P, T, pivot, max_distance):
    """One linearisation at T (3 x 4 row-major, 12 doubles) -> (J^T J 6x6, J^T r 6, inliers, sum r^2)."""
    x, y, z = _apply(T, P)
    pts = np.zeros(len(x), dtype=[("x", "<f4"), ("y", "<f4"), ("z", "<f4")])
    pts["x"], pts["y"], pts["z"] = x.astype(F32), y.astype(F32), z.astype(F32)
    ci, cj, ck = rm.cells(pts, M.v)
    lim = (1 << 20) - 1
    ok = (ci >= -lim + 1) & (ci <= lim - 1) & (cj >= -lim + 1) & (cj <= lim - 1) & (ck >= -lim) & (ck <= lim)
    ci, cj, ck = np.where(ok, ci, 0), np.where(ok, cj, 0), np.where(ok, ck, 0)
    hit, h_at = M.lookup(ci, cj, ck)
    hit &= ok
    x0, y0, z0 = M.cx[h_at].astype(np.float64), M.cy[h_at].astype(np.float64), M.cz[h_at].astype(np.float64)
    S = {k: np.zeros(len(x)) for k in ("uu", "uw", "u", "ww", "w", "1", "uh", "wh", "h")}
    for dj in (0, -1, 1):
        for di in (-1, 0, 1):
            pr, at = M.lookup(ci + di, cj + dj, ck)
            pr &= hit
            u = M.cx[at].astype(np.float64) - x0
            w = M.cy[at].astype(np.float64) - y0
            h = M.cz[at].astype(np.float64) - z0
            for k, val in (("uu", u * u), ("uw", u * w), ("u", u), ("ww", w * w), ("w", w), ("1", np.ones_like(u)),
                           ("uh", u * h), ("wh", w * h), ("h", h)):
                S[k] = S[k] + np.where(pr, val, 0.0)
    Suu, Suw, Su, Sww, Sw, S1, Suh, Swh, Sh = (S[k] for k in ("uu", "uw", "u", "ww", "w", "1", "uh", "wh", "h"))
    with np.errstate(divide="ignore", invalid="ignore"):
        c00 = Sww * S1 - Sw * Sw
        c01 = Sw * Su - Suw * S1
        c02 = Suw * Sw - Sww * Su
        c11 = Suu * S1 - Su * Su
        c12 = Su * Suw - Suu * Sw
        det = Suu * c00 + Suw * c01 + Su * c02
        fit = hit & (S1 >= 3.0) & (det > FIT_COND * Suu * Sww * S1)
        a = (c00 * Suh + c01 * Swh + c02 * Sh) / det
        b = (c01 * Suh + c11 * Swh + c12 * Sh) / det
        nn = np.sqrt(a * a + b * b + 1.0)
        nx, ny, nz = -a / nn, -b / nn, 1.0 / nn
        r = nx * (x - x0) + ny * (y - y0) + nz * (z - z0)
    inl = fit & (np.abs(r) <= max_distance)
    qx, qy, qz = x - pivot[0], y - pivot[1], z - pivot[2]
    J = np.stack([qy * nz - qz * ny, qz * nx - qx * nz, qx * ny - qy * nx, nx, ny, nz], axis=1)[inl]
    r = r[inl]
    return J.T @ J, J.T @ r, int(inl.sum()), float(np.sum(r * r))


def eigen6(A):
    """Cyclic Jacobi as reg_eigen6 -> (eigenvalues, V with eigenvectors in columns)."""
    A = [list(map(float, row)) for row in A]
    V = [[1.0 if i == j else 0.0 for j in range(6)] for i in range(6)]
    for _ in range(50):
        rotated = False
        for p in range(5):
            for q in range(p + 1, 6):
                apq = A[p][q]
                if apq == 0.0:
                    continue
                if abs(apq) <= 1e-300 or abs(apq) <= 1e-18 * (abs(A[p][p]) + abs(A[q][q])):
                    A[p][q] = A[q][p] = 0.0
                    continue
                rotated = True
                theta = (A[q][q] - A[p][p]) / (2.0 * apq)
                t = (1.0 if theta >= 0 else -1.0) / (abs(theta) + math.sqrt(theta * theta + 1.0))
                c = 1.0 / math.sqrt(t * t + 1.0)
                sn = t * c
                for k in range(6):
                    akp, akq = A[k][p], A[k][q]
                    A[k][p], A[k][q] = c * akp - sn * akq, sn * akp + c * akq
                for k in range(6):
                    apk, aqk = A[p][k], A[q][k]
                    A[p][k], A[q][k] = c * apk - sn * aqk, sn * apk + c * aqk
                for k in range(6):
                    vkp, vkq = V[k][p], V[k][q]
                    V[k][p], V[k][q] = c * vkp - sn * vkq, sn * vkp + c * vkq
        if not rotated:
            break
    return [A[i][i] for i in range(6)], V


def solve(H, g, degenerate_ratio):
    """-> (update x (wx, wy, wz, tx, ty, tz), rank).  Rotations are scaled to arc lengths at L = sqrt(tr(H_rot) / tr(H_t))."""
    H = [[float(H[i][j]) for j in range(6)] for i in range(6)]
    tr_r, tr_t = H[0][0] + H[1][1] + H[2][2], H[3][3] + H[4][4] + H[5][5]
    L = math.sqrt(tr_r / tr_t) if tr_r > 0.0 and tr_t > 0.0 else 1.0
    sc = [1.0 / L] * 3 + [1.0] * 3
    g = [float(g[i]) * sc[i] for i in range(6)]
    H = [[H[i][j] * (sc[i] * sc[j]) for j in range(6)] for i in range(6)]
    w, V = eigen6(H)
    thr = degenerate_ratio * max(0.0, max(w))
    x = [0.0] * 6
    rank = 0
    for e in range(6):
        if not (w[e] > 0.0) or w[e] < thr:
            continue
        d = sum(V[i][e] * g[i] for i in range(6))
        f = -d / w[e]
        for i in range(6):
            x[i] += f * V[i][e]
        rank += 1
    return [x[i] * sc[i] for i in range(6)], rank


def compose(T, x, pivot):
    """T <- [R(x[:3]) | pivot + x[3:] - R pivot] T"""
    th = math.sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2])
    R = [1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0]
    if th > 0.0:
        kx, ky, kz = x[0] / th, x[1] / th, x[2] / th
        c, s = math.cos(th), math.sin(th)
        v = 1.0 - c
        R = [c + kx * kx * v, kx * ky * v - kz * s, kx * kz * v + ky * s,
             ky * kx * v + kz * s, c + ky * ky * v, ky * kz * v - kx * s,
             kz * kx * v - ky * s, kz * ky * v + kx * s, c + kz * kz * v]
    D = []
    for i in range(3):
        D += [R[3 * i], R[3 * i + 1], R[3 * i + 2],
              pivot[i] + x[3 + i] - (R[3 * i] * pivot[0] + R[3 * i + 1] * pivot[1] + R[3 * i + 2] * pivot[2])]
    Tn = []
    for i in range(3):
        for j in range(4):
            s = D[4 * i] * T[j] + D[4 * i + 1] * T[4 + j] + D[4 * i + 2] * T[8 + j]
            if j == 3:
                s += D[4 * i + 3]
            Tn.append(s)
    return Tn, th, math.sqrt(x[3] ** 2 + x[4] ** 2 + x[5] ** 2)


def register(M, pts, T_init=None, **params):
    """-> (T_out float32 4x4, stats dict) as o3r_cloud_register returns them.  pts: abi.POINT records or (n, 3) float32."""
    prm = defaults(M.v)
    prm.update(params)
    if getattr(pts, "dtype", None) is not None and pts.dtype.names:
        P = np.stack([pts["x"], pts["y"], pts["z"]], axis=1).astype(np.float64)
    else:
        P = np.asarray(pts, dtype=F32).reshape(-1, 3).astype(np.float64)
    T0 = np.eye(4, dtype=F32) if T_init is None else np.asarray(T_init, dtype=F32).reshape(4, 4)
    T0d = [float(t) for t in T0.reshape(16)[:12]]
    T = list(T0d)
    st = dict(iterations=0, converged=0, rank=0, n_inliers=0, rms_initial=0.0, rms_final=0.0,
              pivot=np.zeros(3), info=np.zeros((6, 6)))
    if len(P):
        x, y, z = _apply(T0d, P)
        pivot = [float(np.sum(x)) / len(P), float(np.sum(y)) / len(P), float(np.sum(z)) / len(P)]
        st["pivot"] = np.array(pivot)
        for it in range(prm["max_iterations"]):
            H, g, n_in, ss = linearise(M, P, T, pivot, prm["max_distance"])
            rms = math.sqrt(ss / n_in) if n_in else 0.0
            st["info"], st["n_inliers"], st["rms_final"] = H, n_in, rms
            if it == 0:
                st["rms_initial"] = rms
            if n_in < 6:
                T, st["rank"], st["converged"] = list(T0d), 0, 0
                break
            st["iterations"] += 1
            upd, st["rank"] = solve(H, g, prm["degenerate_ratio"])
            T, th, tn = compose(T, upd, pivot)
            if th < prm["min_rotation"] and tn < prm["min_translation"]:
                st["converged"] = 1
                break
    out = np.eye(4, dtype=F32)
    out[:3, :] = np.array(T, dtype=np.float64).reshape(3, 4).astype(F32)
    return out, st


# ---- scenes shared by the model test and the GPU tests --------------------------------------------------------------------
def cells_from_points(pts, v):
    """abi.CELL records of a cloud appended in one go (sums rounded once to float32: a map, not the device's bits)."""
    from online_3d_reconstruction_b200 import abi
    s = rm.cell_sums(pts, v)
    c = np.zeros(len(s), dtype=abi.CELL)
    c["key"], c["n"] = s["key"], s["n"]
    c["sx"], c["sy"], c["sz"] = s["sx"].astype(F32), s["sy"].astype(F32), s["sz"].astype(F32)
    c["sr"], c["sg"], c["sb"] = s["sr"], s["sg"], s["sb"]
    return c


def _terrain(seed):
    rng = np.random.default_rng(seed)
    waves = [(rng.uniform(1.0, 3.0), *(rng.uniform(-1, 1, 2) * 2 * math.pi / rng.uniform(25.0, 70.0)), rng.uniform(0, 2 * math.pi))
             for _ in range(4)]
    boxes = [(*rng.uniform(-80, 80, 2), *rng.uniform(6.0, 18.0, 2), rng.uniform(3.0, 8.0)) for _ in range(8)]

    def h(x, y):
        z = np.zeros_like(x, dtype=np.float64)
        for a, kx, ky, ph in waves:
            z += a * np.sin(kx * x + ky * y + ph)
        for bx, by, sx, sy, bh in boxes:
            z += np.where((np.abs(x - bx) < sx / 2) & (np.abs(y - by) < sy / 2), bh, 0.0)
        return z
    return h


def _samples(h, rng, half, step, cx=0.0, cy=0.0):
    g = np.arange(-half, half, step)
    x, y = np.meshgrid(g + cx, g + cy)
    x = x.ravel() + rng.uniform(-step / 2, step / 2, x.size)
    y = y.ravel() + rng.uniform(-step / 2, step / 2, y.size)
    from online_3d_reconstruction_b200 import abi
    p = np.zeros(x.size, dtype=abi.POINT)
    p["x"], p["y"], p["z"] = x.astype(F32), y.astype(F32), h(x, y).astype(F32)
    p["rgb"] = 0x808080
    return p


def rigid(yaw_deg=0.0, pitch_deg=0.0, roll_deg=0.0, t=(0.0, 0.0, 0.0)):
    """4 x 4 float64: Rz(yaw) Ry(pitch) Rx(roll), then t."""
    a, b, c = (math.radians(d) for d in (yaw_deg, pitch_deg, roll_deg))
    Rz = np.array([[math.cos(a), -math.sin(a), 0], [math.sin(a), math.cos(a), 0], [0, 0, 1]])
    Ry = np.array([[math.cos(b), 0, math.sin(b)], [0, 1, 0], [-math.sin(b), 0, math.cos(b)]])
    Rx = np.array([[1, 0, 0], [0, math.cos(c), -math.sin(c)], [0, math.sin(c), math.cos(c)]])
    T = np.eye(4)
    T[:3, :3] = Rz @ Ry @ Rx
    T[:3, 3] = t
    return T


def transform_points(pts, T):
    out = pts.copy()
    P = np.stack([pts["x"], pts["y"], pts["z"]], axis=1).astype(np.float64) @ T[:3, :3].T + T[:3, 3]
    out["x"], out["y"], out["z"] = (P[:, i].astype(F32) for i in range(3))
    return out


def terrain_scene(seed=7, map_half=100.0, map_step=0.25, src_half=45.0, src_step=0.5):
    """-> (map points, source points, E): dense jittered samples of a height field with relief (sinusoids plus boxes) as the
    map; other jittered samples of a sub-window, moved by E (2 deg yaw, 1 deg roll, 0.3 m on each axis), as the source.
    Registration should return about E^-1."""
    h = _terrain(seed)
    rng = np.random.default_rng(seed + 1000)
    mp = _samples(h, rng, map_half, map_step)
    src = _samples(h, rng, src_half, src_step, cx=7.3, cy=-4.1)
    E = rigid(yaw_deg=2.0, roll_deg=1.0, t=(0.3, 0.3, 0.3))
    return mp, transform_points(src, E), E


def flat_scene(v=1.0, dz=0.25):
    """-> (map points, source points): a plane z = 0 sampled on a regular dyadic grid (every sum exact), and a source on
    z = dz over a regular grid symmetric about the origin."""
    from online_3d_reconstruction_b200 import abi
    g = np.arange(-40.0, 40.0, v / 4) + v / 8
    x, y = np.meshgrid(g, g)
    mp = np.zeros(x.size, dtype=abi.POINT)
    mp["x"], mp["y"] = x.ravel(), y.ravel()
    s = np.arange(-20.0, 20.0, v / 2) + v / 4
    x, y = np.meshgrid(s, s)
    src = np.zeros(x.size, dtype=abi.POINT)
    src["x"], src["y"], src["z"] = x.ravel(), y.ravel(), dz
    return mp, src


def pose_error(T_out, E):
    """-> (translation error m, rotation error deg) of T_out against the inverse of the perturbation E."""
    D = np.asarray(T_out, dtype=np.float64) @ E
    ang = math.degrees(math.acos(max(-1.0, min(1.0, (np.trace(D[:3, :3]) - 1.0) / 2.0))))
    return float(np.linalg.norm(D[:3, 3])), ang
