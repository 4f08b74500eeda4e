"""Vectorised NumPy restatement of ctx_marching_cubes (csrc/mcubes.cu) and of the lattice of ctx_density_grid
(csrc/field.cu), with the case table of oracle/mc_tables.py.  No GPU.

Contract restated here bit for bit:

* lattice point ``(i, j, k)`` of a ``sigma [X, Y, Z]`` field sits at ``o + h * idx`` per axis, in fp32, one rounding
  per operation;
* one vertex per lattice edge whose ends straddle ``iso`` (``sigma >= iso`` is inside), numbered in the order (linear
  index of the lower endpoint, then axis x < y < z); its position along the edge is ``t = (iso - s0) / (s1 - s0)`` and
  ``o + h * (idx + t)`` (fp32, one rounding per operation);
* the normal is the normalised negative density gradient: central differences (one-sided on the lattice border)
  divided by ``2 h`` (``h``), linearly interpolated along the edge; a zero gradient gives ``(0, 0, 0)``;
* faces in cell order (C order over the cells), then in table order within a cell.
"""
from __future__ import annotations

import numpy as np

from . import mc_tables

F32 = np.float32


def lattice_axis(n_points, o, h):
    """fp32 coordinates o + h * i, i < n_points, as the kernels form them"""
    return (F32(o) + F32(h) * np.arange(n_points, dtype=F32)).astype(F32)


def spacing(lo, hi, cells):
    """per-axis (origin, spacing) in fp32: spacing (hi - lo) / n formed in float64, as NerfTrainer passes them"""
    lo, hi = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
    return lo.astype(F32), ((hi - lo) / np.asarray(cells, np.float64)).astype(F32)


def _gradient(s, h):
    """fp32 density gradient per axis, [X, Y, Z, 3]"""
    g = np.empty(s.shape + (3,), F32)
    for a in range(3):
        n = s.shape[a]
        sl = lambda x: tuple(x if b == a else slice(None) for b in range(3))   # noqa: E731
        ga = np.empty_like(s)
        if n > 2:
            ga[sl(slice(1, -1))] = (s[sl(slice(2, None))] - s[sl(slice(None, -2))]) / (F32(2) * F32(h[a]))
        ga[sl(slice(0, 1))] = (s[sl(slice(1, 2))] - s[sl(slice(0, 1))]) / F32(h[a])
        ga[sl(slice(n - 1, n))] = (s[sl(slice(n - 1, n))] - s[sl(slice(n - 2, n - 1))]) / F32(h[a])
        g[..., a] = ga
    return g


def edge_mask(sigma, iso):
    """bool [X, Y, Z, 3]: the edge from point (i, j, k) along each axis straddles iso"""
    inside = sigma >= F32(iso)
    m = np.zeros(sigma.shape + (3,), bool)
    m[:-1, :, :, 0] = inside[:-1] != inside[1:]
    m[:, :-1, :, 1] = inside[:, :-1] != inside[:, 1:]
    m[:, :, :-1, 2] = inside[:, :, :-1] != inside[:, :, 1:]
    return m


def cases(sigma, iso):
    """uint8 [X-1, Y-1, Z-1]: the bit set of the inside corners of each cell"""
    inside = (sigma >= F32(iso)).astype(np.uint8)
    c = np.zeros(tuple(n - 1 for n in sigma.shape), np.uint8)
    for k, (dx, dy, dz) in enumerate(mc_tables.CORNERS):
        c |= inside[dx:dx + c.shape[0], dy:dy + c.shape[1], dz:dz + c.shape[2]] << k
    return c


def marching_cubes(sigma, iso, origin=(0.0, 0.0, 0.0), h=(1.0, 1.0, 1.0), with_normals=True,
                   index_offset=(0, 0, 0)):
    """(vertices [V,3] fp32, faces [F,3] int32, normals [V,3] fp32 or None) of ctx_marching_cubes.  ``index_offset``:
    the lattice index of sigma[0, 0, 0] when sigma is a block of a larger lattice (the vertices are then those of the
    whole lattice; the normals are not, since the gradient turns one-sided on the block's border)."""
    s = np.ascontiguousarray(sigma, dtype=F32)
    assert s.ndim == 3 and min(s.shape) >= 2
    iso, o, h = F32(iso), np.asarray(origin, F32), np.asarray(h, F32)
    m = edge_mask(s, iso)
    ids = np.cumsum(m.reshape(-1)).reshape(m.shape).astype(np.int64) - 1      # vertex id of each crossing edge
    p, axis = np.nonzero(m.reshape(-1, 3))
    idx = np.stack(np.unravel_index(p, s.shape), -1)                          # lower endpoint [V,3]
    step = np.eye(3, dtype=np.int64)[axis]
    s0 = s.reshape(-1)[p]
    s1 = s[tuple((idx + step).T)]
    t = ((iso - s0) / (s1 - s0)).astype(F32)
    frac = (idx + np.asarray(index_offset, np.int64)).astype(F32)
    frac[np.arange(len(p)), axis] += t
    verts = (o + h * frac).astype(F32)
    normals = None
    if with_normals:
        g = _gradient(s, h)
        g0, g1 = g.reshape(-1, 3)[p], g[tuple((idx + step).T)]
        gi = (g0 + t[:, None] * (g1 - g0)).astype(F32)
        nrm = np.sqrt((gi * gi).sum(-1, dtype=F32)).astype(F32)
        safe = np.where(nrm > 0, nrm, F32(1))[:, None]
        normals = np.where(nrm[:, None] > 0, -gi / safe, F32(0)).astype(F32)
    c = cases(s, iso)
    tab, cnt = mc_tables.table()
    cell = np.nonzero(cnt[c.reshape(-1)] > 0)[0]
    ci = np.stack(np.unravel_index(cell, c.shape), -1)                        # [C,3]
    tri = tab[c.reshape(-1)[cell]].astype(np.int64)                          # [C, MAX, 3] edge ids
    valid = tri[..., 0] >= 0
    e = np.where(tri >= 0, tri, 0)
    ax, o4 = e // 4, e % 4
    u, v = o4 & 1, o4 >> 1
    q = np.broadcast_to(ci[:, None, None, :], e.shape + (3,)).copy()
    # the other two axes of each edge take the offsets (u, v) in increasing axis order
    oth0 = np.where(ax == 0, 1, 0)
    oth1 = np.where(ax == 2, 1, 2)
    for a in range(3):
        q[..., a] += np.where(oth0 == a, u, 0) + np.where(oth1 == a, v, 0)
    faces = ids[q[..., 0], q[..., 1], q[..., 2], ax][valid].astype(np.int32)
    return verts, faces.reshape(-1, 3), normals


# ---------------------------------------------------------------- whole-mesh properties (used by the tests)
def directed_edges(faces):
    f = np.asarray(faces, np.int64)
    return np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])


def edge_use(faces):
    """(unique undirected edges [E,2], times used, directed-use balance): a closed, consistently oriented mesh uses
    each edge twice, once in each direction (balance 0)"""
    d = directed_edges(faces)
    und = np.sort(d, 1)
    sign = np.where(d[:, 0] < d[:, 1], 1, -1)
    key = und[:, 0] * (int(und.max()) + 1 if len(und) else 1) + und[:, 1]
    uk, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    bal = np.zeros(len(uk), np.int64)
    np.add.at(bal, inv.reshape(-1), sign)
    first = np.zeros(len(uk), np.int64)
    first[inv.reshape(-1)] = np.arange(len(d))
    return und[first], cnt, bal


def euler_characteristic(n_vertices, faces):
    e, _, _ = edge_use(faces)
    return int(n_vertices) - len(e) + len(faces)


def signed_volume(verts, faces):
    v = np.asarray(verts, np.float64)[np.asarray(faces, np.int64)]
    return float(np.einsum("ij,ij->i", v[:, 0], np.cross(v[:, 1], v[:, 2])).sum() / 6.0)
