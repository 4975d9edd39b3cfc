"""CPU-side checks: the C-ABI library loads and exports every symbol include/o3r.h declares, the ctypes
mirror matches the C layout, host pose composition matches the oracle, the generator is deterministic."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle_binding as ob
from online_3d_reconstruction_b200 import abi, lib, synth, tmat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(lib.SO_PATH):
        import __graft_entry__ as g
        g.build()
    return lib.load()


def test_library_exports_every_declared_symbol(L):
    hdr = open(os.path.join(ROOT, "include", "o3r.h")).read()
    declared = set(re.findall(r"\b(o3r_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(lib.SYMBOLS), declared ^ set(lib.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), s
    assert L.o3r_version() == 1


def test_ctypes_layout_matches_c():
    o = ob.lib()
    o.orc_sizeof.restype = C.c_size_t
    assert o.orc_sizeof(0) == C.sizeof(abi.Params)
    assert o.orc_sizeof(1) == C.sizeof(abi.Frame)
    assert o.orc_sizeof(2) == abi.POINT.itemsize
    assert o.orc_sizeof(3) == abi.CELL.itemsize


def test_no_cpu_fallback_without_device(L):
    """Without a GPU the product must fail loudly, not compute on the CPU.  The check runs in a child process that sees
    no device, so it also runs on a machine that has one."""
    code = ("import ctypes as C, sys; sys.path.insert(0, sys.argv[1])\n"
            "from online_3d_reconstruction_b200 import abi, lib\n"
            "L = lib.load(); p = abi.make_params(); h = C.c_void_p()\n"
            "rc = L.o3r_create(C.byref(p), C.byref(h))\n"
            "assert rc == abi.O3R_ERR_CUDA and not h.value, rc\n"
            "assert b'no CPU fallback' in L.o3r_last_error(None), L.o3r_last_error(None)\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


def test_invalid_params_rejected(L):
    p = abi.make_params()
    p.voxel_size = 0.0
    h = C.c_void_p()
    assert L.o3r_create(C.byref(p), C.byref(h)) == abi.O3R_ERR_INVALID


def test_product_does_not_touch_the_oracle():
    pkg = os.path.join(ROOT, "online_3d_reconstruction_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", "Makefile")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle_binding" not in txt and "o3r_oracle" not in txt and "oracle/" not in txt, f


def test_generate_tmat_matches_oracle_bitwise():
    rng = np.random.default_rng(0)
    for _ in range(50):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        t = rng.uniform(-50, 50, 3)
        a = tmat.generate_tmat(*t, *q)
        b = ob.generate_tmat(*t, *q)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    with pytest.raises(ValueError):
        tmat.generate_tmat(0, 0, 0, 1, 1, 0, 0)
    m1, m2 = rng.normal(size=(4, 4)).astype(np.float32), rng.normal(size=(4, 4)).astype(np.float32)
    assert np.array_equal(tmat.mat4_mul(m1, m2), ob.mat4_mul(m1, m2))


def test_synthetic_sequence_is_deterministic_and_fixture_like():
    a = synth.uav720(1002, 2)
    b = synth.uav720(1002, 2)
    for (d1, i1, t1), (d2, i2, t2) in zip(a, b):
        assert np.array_equal(d1, d2) and np.array_equal(i1, i2) and np.array_equal(t1, t2)
    d = a[0][0]
    assert d.shape == (720, 1280) and d.dtype == np.uint8 and d[:, :160].max() == 0
    roi = d[20:700, 160:1260]
    valid = roi > 64
    assert 0.97 < valid.mean() < 0.995
    assert 100 < roi[valid].mean() < 116 and roi.max() <= 127
    p = abi.make_params(jump_pixels=1)
    assert 1.0 < ob.get_variance(p, d, False) < 80.0
    # consecutive frames are ~0.45 m apart
    step = np.linalg.norm(a[1][2][:3, 3] - a[0][2][:3, 3])
    assert 0.1 < step < 1.2
