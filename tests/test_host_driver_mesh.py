"""The host driver's --save_mesh: mesh.ply holds cloud.ply's points as its vertices and the triangles and normals of the
numpy model (tests/mesh_model.py) of the saved map; without the flag there is no mesh.ply and cloud.ply is unchanged."""
import os

import numpy as np
import pytest

import mesh_model as mm
from online_3d_reconstruction_b200 import mapfile
from test_host_driver import pose_bin  # noqa: F401 (a fixture)
from test_host_driver_register import _run, _write_same_frames

pytestmark = pytest.mark.gpu
VOX = 0.05


def _read_ply(path):
    """-> (header lines, payload bytes) of a binary PLY."""
    raw = open(path, "rb").read()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    return raw[:end].decode().splitlines(), raw[end:]


def _read_mesh(path):
    head, body = _read_ply(path)
    nv = int(next(l for l in head if l.startswith("element vertex")).split()[-1])
    nf = int(next(l for l in head if l.startswith("element face")).split()[-1])
    assert head[1] == "format binary_little_endian 1.0"
    assert [l.split()[-1] for l in head if l.startswith("property")] == \
        ["x", "y", "z", "nx", "ny", "nz", "red", "green", "blue", "vertex_indices"]
    vt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("n", "<f4", 3), ("r", "u1"), ("g", "u1"), ("b", "u1")])
    ft = np.dtype([("k", "u1"), ("v", "<i4", 3)])
    assert len(body) == nv * vt.itemsize + nf * ft.itemsize
    v = np.frombuffer(body[:nv * vt.itemsize], dtype=vt)
    f = np.frombuffer(body[nv * vt.itemsize:], dtype=ft)
    assert np.all(f["k"] == 3)
    return v, f["v"]


def _read_cloud(path):
    head, body = _read_ply(path)
    n = int(next(l for l in head if l.startswith("element vertex")).split()[-1])
    return np.frombuffer(body[:n * 15], dtype=np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("r", "u1"), ("g", "u1"),
                                                         ("b", "u1")]))


def test_save_mesh(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_same_frames(root, 6, 128, 256, lifted=set())
    _, plain = _run(pose_bin, root, str(tmp_path / "plain"))
    assert not os.path.exists(os.path.join(plain, "mesh.ply"))
    _, meshed = _run(pose_bin, root, str(tmp_path / "mesh"), "--save_mesh")
    for name in ("cloud.ply", "cloud_uavpos.ply"):
        assert open(os.path.join(plain, name), "rb").read() == open(os.path.join(meshed, name), "rb").read(), name
    step = 0.05
    _, gated = _run(pose_bin, root, str(tmp_path / "gated"), "--save_mesh", "--mesh_max_step", str(step), "--save_map")
    _, cells = mapfile.read(os.path.join(gated, "map.o3rmap"))
    cloud = _read_cloud(os.path.join(gated, "cloud.ply"))
    for run_dir, max_step in ((meshed, np.inf), (gated, step)):
        v, f = _read_mesh(os.path.join(run_dir, "mesh.ply"))
        assert len(v) == len(cloud) > 0
        for a, b in (("x", "x"), ("y", "y"), ("z", "z"), ("r", "r"), ("g", "g"), ("b", "b")):
            assert v[a].tobytes() == cloud[b].tobytes(), a
        _, nrm, tris = mm.mesh(cells, VOX, 1, max_step)
        assert (len(tris) > 0 or max_step < np.inf) and np.array_equal(f.astype(np.uint32).reshape(-1, 3), tris)
        assert v["n"].tobytes() == nrm.tobytes()
    assert len(_read_mesh(os.path.join(gated, "mesh.ply"))[1]) <= len(_read_mesh(os.path.join(meshed, "mesh.ply"))[1])


def test_dont_downsample_writes_no_mesh(pose_bin, tmp_path):
    root = str(tmp_path / "data")
    _write_same_frames(root, 6, 128, 256, lifted=set())
    r, run_dir = _run(pose_bin, root, str(tmp_path / "dd"), "--save_mesh", "--dont_downsample")
    assert "no mesh.ply is written" in r.stdout
    assert not os.path.exists(os.path.join(run_dir, "mesh.ply"))
