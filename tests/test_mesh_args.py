"""Mesh extraction without a GPU: the generated case table, the NumPy restatement of ctx_marching_cubes on analytic
fields (closed, consistently oriented meshes of the right topology, volume and accuracy) and the C-ABI's argument
errors."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import marching_cubes as mc
from oracle import mc_tables


def test_generator_reproduces_the_committed_header():
    out = subprocess.run([sys.executable, "-m", "oracle.mc_tables"], cwd=ROOT, capture_output=True, check=True).stdout
    with open(os.path.join(ROOT, "contexture-nerf_b200", "csrc", "mc_tables.cuh"), "rb") as fh:
        assert out == fh.read()


def test_every_case_loops_through_exactly_its_crossing_edges():
    tab, cnt = mc_tables.table()
    for case in range(256):
        loops = mc_tables.loops(case)
        assert sorted(e for lp in loops for e in lp) == mc_tables.crossing_edges(case), case
        assert all(len(lp) >= 3 for lp in loops) and all(lp[0] == min(lp) for lp in loops)
        assert cnt[case] == sum(len(lp) - 2 for lp in loops) <= mc_tables.MAX_TRIS
        # the complement swaps inside and outside: the same edges, the opposite orientation
        assert sorted(mc_tables.crossing_edges(case)) == sorted(mc_tables.crossing_edges(255 - case))


def _field(n, fn, lo=-1.0, hi=1.0):
    o, h = mc.spacing((lo,) * 3, (hi,) * 3, (n,) * 3)
    x = [mc.lattice_axis(n + 1, o[a], h[a]).astype(np.float64) for a in range(3)]
    X, Y, Z = np.meshgrid(*x, indexing="ij")
    return fn(X, Y, Z).astype(np.float32), o, h


def _check_closed(verts, faces):
    _, cnt, bal = mc.edge_use(faces)
    assert (cnt == 2).all() and (bal == 0).all()     # every edge twice, once in each direction


def test_sphere_is_closed_accurate_and_encloses_its_volume():
    r, n = 0.7, 64
    s, o, h = _field(n, lambda X, Y, Z: r - np.sqrt(X * X + Y * Y + Z * Z))
    v, f, nrm = mc.marching_cubes(s, 0.0, o, h)
    _check_closed(v, f)
    assert mc.euler_characteristic(len(v), f) == 2
    rad = np.linalg.norm(v.astype(np.float64), axis=1)
    assert np.abs(rad - r).max() < float(h[0]) ** 2         # O(h^2): the field is linear along the radius
    vol = mc.signed_volume(v, f)
    assert vol > 0 and abs(vol / (4.0 / 3.0 * np.pi * r ** 3) - 1.0) < 0.01
    # normals: unit, pointing away from the denser inside
    assert np.allclose(np.linalg.norm(nrm, axis=1), 1.0, atol=1e-5)
    assert ((nrm * v).sum(1) > 0).all()


def test_torus_and_two_spheres_have_the_right_euler_characteristic():
    R, r = 0.55, 0.2
    s, o, h = _field(64, lambda X, Y, Z: r - np.sqrt((np.sqrt(X * X + Y * Y) - R) ** 2 + Z * Z))
    v, f, _ = mc.marching_cubes(s, 0.0, o, h)
    _check_closed(v, f)
    assert mc.euler_characteristic(len(v), f) == 0
    assert mc.signed_volume(v, f) > 0
    s, o, h = _field(48, lambda X, Y, Z: np.maximum(0.3 - np.sqrt((X - 0.45) ** 2 + Y * Y + Z * Z),
                                                    0.3 - np.sqrt((X + 0.45) ** 2 + Y * Y + Z * Z)))
    v, f, _ = mc.marching_cubes(s, 0.0, o, h)
    _check_closed(v, f)
    assert mc.euler_characteristic(len(v), f) == 4


def _closed_away_from_border(s, iso):
    """The mesh has no boundary away from the lattice border: every edge off the border is used as often in one
    direction as in the other.  (On a noisy field a few edges are used four times: a fan diagonal between two vertices
    of a shared ambiguous face can be drawn by both cells.  Its uses still cancel.)"""
    v, f, _ = mc.marching_cubes(s, iso)
    assert len(f) > 0
    e, cnt, bal = mc.edge_use(f)
    lim = np.asarray(s.shape, np.float32) - 1
    on_border = ((v == 0) | (v == lim)).any(1)
    inner = ~(on_border[e[:, 0]] & on_border[e[:, 1]])
    assert (bal[inner] == 0).all() and (cnt[inner] % 2 == 0).all()
    assert (bal != 0).any() or len(f) < 8            # the border does cut the surface open
    return v, f


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_fields_are_closed_away_from_the_border(seed):
    s = np.random.default_rng(seed).random((13, 11, 9), dtype=np.float32)
    _closed_away_from_border(s, 0.5)


def test_plateau_fields_are_closed_away_from_the_border():
    """values exactly at iso count as inside; the vertices of such edges sit on lattice points (t = 0 or 1)"""
    rng = np.random.default_rng(3)
    s = rng.choice(np.array([0.0, 0.5, 1.0], np.float32), size=(12, 10, 14))
    v, _ = _closed_away_from_border(s, 0.5)
    assert (v == np.rint(v)).any()
    _closed_away_from_border(np.where(rng.random((9, 9, 9)) < 0.5, 0.5, 0.25).astype(np.float32), 0.5)


def test_single_cells_follow_the_table():
    tab, cnt = mc_tables.table()
    for case in range(256):
        s = np.array([1.0 if case >> c & 1 else 0.0 for c in range(8)], np.float32).reshape(2, 2, 2, order="F")
        v, f, _ = mc.marching_cubes(s, 0.5)
        assert len(v) == len(mc_tables.crossing_edges(case)) and len(f) == cnt[case]


def test_lattice_spacing_is_formed_in_float64():
    o, h = mc.spacing((-1.2,) * 3, (1.2,) * 3, (256, 256, 256))
    assert h.dtype == np.float32 and h[0] == np.float32(2.4 / 256)
    x = mc.lattice_axis(257, o[0], h[0])
    assert x[0] == np.float32(-1.2) and x[128] == np.float32(np.float32(-1.2) + np.float32(h[0]) * np.float32(128))


def test_abi_argument_errors_do_not_need_a_gpu(libpath):
    from ctxnerf import _lib
    lib = _lib.lib()
    assert lib.ctx_density_grid_workspace(0, 4, 4) == -1 and lib.ctx_density_grid_workspace(1025, 4, 4) == -1
    assert lib.ctx_density_grid_workspace(1024, 1024, 1024) > 0
    assert lib.ctx_density_grid_workspace(1, 1, 1) > 0
    assert lib.ctx_marching_cubes_workspace(0, 1, 1) == -1
    assert lib.ctx_marching_cubes_workspace(2048, 1024, 1024) == -1          # 2^31 points or more
    assert lib.ctx_marching_cubes_workspace(512, 512, 512) > 0
    assert lib.ctx_vertex_colors_workspace(0) == -1 and lib.ctx_vertex_colors_workspace(1) > 0
    fake = ctypes.c_void_p(256)
    args = (0.0, 0.0, 0.0, 1.0, 1.0, 1.0)
    # density grid: bad sizes, no net, no workspace
    assert lib.ctx_density_grid(None, 10, 4, 4, 4, 4, *args, fake, 1 << 20, fake, None) == -1
    assert lib.ctx_density_grid(None, 10, 4, 1025, 4, 4, *args, fake, 1 << 20, fake, None) == -1
    # marching cubes: sizes, nulls, pass, a short or misaligned workspace
    need = lib.ctx_marching_cubes_workspace(4, 4, 4)
    assert lib.ctx_marching_cubes(fake, 0, 4, 4, *args, 0.5, fake, need, fake, None, None, None, 0, None) == -1
    assert lib.ctx_marching_cubes(None, 4, 4, 4, *args, 0.5, fake, need, fake, None, None, None, 0, None) == -1
    assert lib.ctx_marching_cubes(fake, 4, 4, 4, *args, 0.5, fake, need - 1, fake, None, None, None, 0, None) == -1
    assert lib.ctx_marching_cubes(fake, 4, 4, 4, *args, 0.5, ctypes.c_void_p(8), need, fake, None, None, None, 0,
                                  None) == -1
    assert lib.ctx_marching_cubes(fake, 4, 4, 4, *args, 0.5, fake, need, fake, None, None, None, 2, None) == -1
    assert lib.ctx_marching_cubes(fake, 4, 4, 4, *args, 0.5, fake, need, fake, None, None, None, 1, None) == -1
    # vertex colours: no net
    assert lib.ctx_vertex_colors(None, 10, 4, fake, None, 4, fake, 1 << 20, fake, None) == -1
    assert lib.ctx_vertex_colors(None, 10, 4, fake, None, -1, fake, 1 << 20, fake, None) == -1


def test_python_refusals_do_not_need_a_gpu(libpath):
    from ctxnerf import mesh
    from ctxnerf._lib import CtxNerfError
    for bad in (((0, 0, 0), (0, 1, 1)), ((1, 1, 1), (-1, 2, 2)), ((0, 0, float("nan")), (1, 1, 1)), ((0, 0), (1, 1))):
        with pytest.raises(CtxNerfError):
            mesh.lattice(bad, (4, 4, 4))
    with pytest.raises(CtxNerfError):
        mesh._cells((4, 4))
    o, h = mesh.lattice(((-1.2,) * 3, (1.2,) * 3), (256, 128, 64))
    assert h == [float(np.float32(2.4 / 256)), float(np.float32(2.4 / 128)), float(np.float32(2.4 / 64))]
    with pytest.raises(CtxNerfError):
        mesh.marching_cubes(np.zeros((4, 4, 4), np.float32), 0.5)
