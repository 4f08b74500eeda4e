"""Mesh extraction from a trained field, as the original NeRF release's ``extract_mesh.ipynb`` does it: the density of
the (fine) network on a regular lattice with zero view directions, ``relu``, marching cubes at a threshold, and the
index-space vertices placed in world coordinates -- here with a colour per vertex and a binary PLY writer.

Every numeric stage is a libctxnerf.so kernel (include/ctxnerf.h: ``ctx_density_grid``, ``ctx_marching_cubes``,
``ctx_vertex_colors``); ``oracle/marching_cubes.py`` restates the lattice and the marching cubes in NumPy.  A lattice
of ``n = (nx, ny, nz)`` cells over ``bounds = (lo, hi)`` has ``(nx+1) x (ny+1) x (nz+1)`` points; point ``(i, j, k)``
is at ``lo + h * (i, j, k)`` in fp32 with ``h = (hi - lo) / n`` formed in float64 and rounded to fp32.
"""
from __future__ import annotations

import ctypes
import math

import numpy as np
import torch

from . import _lib
from ._lib import CtxNerfError, call, ptr, stream_ptr

DEFAULT_BOUNDS = ((-1.2, -1.2, -1.2), (1.2, 1.2, 1.2))   # extract_mesh.ipynb's [-1.2, 1.2]^3
_SLAB_BYTES = 1 << 30      # default workspace of the lattice query: slabs of x-planes up to 1 GiB


def _cells(resolution):
    n = (resolution,) * 3 if isinstance(resolution, (int, np.integer)) else tuple(resolution)
    if len(n) != 3 or not all(isinstance(c, (int, np.integer)) and c >= 1 for c in n):
        raise CtxNerfError(f"mesh: resolution must be an int or (nx, ny, nz) cells (each >= 1), got {resolution!r}")
    return tuple(int(c) for c in n)


def lattice(bounds, cells):
    """(origin, spacing) of the lattice, fp32 values as Python floats: origin = lo, spacing = (hi - lo) / n formed in
    float64.  Refuses empty, inverted or non-finite bounds."""
    try:
        lo, hi = (np.asarray(b, dtype=np.float64).reshape(3) for b in bounds)
    except (TypeError, ValueError):
        raise CtxNerfError(f"mesh: bounds must be (lo, hi) with three coordinates each, got {bounds!r}") from None
    if not (np.isfinite(lo).all() and np.isfinite(hi).all() and (hi > lo).all()):
        raise CtxNerfError(f"mesh: bounds must be finite with hi > lo on every axis, got lo={lo}, hi={hi}")
    h = (hi - lo) / np.asarray(cells, dtype=np.float64)
    return [float(v) for v in lo.astype(np.float32)], [float(v) for v in h.astype(np.float32)]


def _ctxnet(net, packed):
    w, _, f = packed
    return _lib.CtxNet(ctypes.addressof(net._desc.blob), w.data_ptr(), f.data_ptr())


def density_grid(net, packed, resolution, bounds=DEFAULT_BOUNDS, workspace_bytes=None):
    """``relu(raw[..., 3])`` of ``net`` (a view-direction NeRF module) with the packed weights ``packed`` = (w, wt,
    fparams) on the lattice, zero view directions: fp32 ``[nx+1, ny+1, nz+1]`` on the weights' device.
    ``workspace_bytes`` sizes the slabs (default up to 1 GiB); the result does not depend on it."""
    cells = _cells(resolution)
    need = int(_lib.lib().ctx_density_grid_workspace(*cells))
    if need < 0:
        raise CtxNerfError(f"density_grid: {cells} cells: every axis needs 1..1024 cells and the lattice < 2^31 points")
    o, h = lattice(bounds, cells)
    dev = packed[0].device
    X, Y, Z = (c + 1 for c in cells)
    if workspace_bytes is None:
        workspace_bytes = max(need, min(_SLAB_BYTES, need * X))
    if workspace_bytes < need:
        raise CtxNerfError(f"density_grid: the workspace needs at least {need} bytes (one x-plane)")
    ws = torch.empty(int(workspace_bytes), dtype=torch.uint8, device=dev)
    sigma = torch.empty(X, Y, Z, dtype=torch.float32, device=dev)
    cn = _ctxnet(net, packed)
    with torch.cuda.device(dev):
        call("ctx_density_grid", ctypes.byref(cn), net.L_pts, net.L_dirs, *cells, *o, *h, ptr(ws), ws.numel(),
             ptr(sigma), stream_ptr(dev))
    return sigma


def marching_cubes(sigma, threshold, bounds=DEFAULT_BOUNDS, normals=True):
    """The surface ``sigma == threshold`` of a lattice ``sigma [nx+1, ny+1, nz+1]`` (fp32, CUDA) over ``bounds``:
    ``dict(vertices [V,3] fp32, faces [F,3] int32, normals [V,3] fp32 or None)`` on sigma's device, in the order of
    ``ctx_marching_cubes`` (one vertex per crossing lattice edge, faces in cell order).  ``sigma >= threshold`` is
    inside; triangle and vertex normals point towards decreasing density.  One host synchronisation (the counts)."""
    if not (torch.is_tensor(sigma) and sigma.is_cuda and sigma.dtype == torch.float32 and sigma.dim() == 3):
        raise CtxNerfError("marching_cubes: sigma must be a 3-D fp32 CUDA tensor [nx+1, ny+1, nz+1]")
    if not math.isfinite(float(threshold)):
        raise CtxNerfError(f"marching_cubes: threshold must be finite, got {threshold}")
    cells = tuple(int(n) - 1 for n in sigma.shape)
    need = int(_lib.lib().ctx_marching_cubes_workspace(*cells))
    if need < 0:
        raise CtxNerfError(f"marching_cubes: sigma {tuple(sigma.shape)} needs >= 2 points per axis and < 2^31 points")
    o, h = lattice(bounds, cells)
    dev = sigma.device
    sigma = sigma.contiguous()
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    counts = torch.zeros(2, dtype=torch.int64, device=dev)
    args = (ptr(sigma), *cells, *o, *h, float(threshold), ptr(ws), need, ptr(counts))
    with torch.cuda.device(dev):
        call("ctx_marching_cubes", *args, None, None, None, 0, stream_ptr(dev))
        V, F = (int(v) for v in counts.cpu())
        if V >= 2 ** 31:
            raise CtxNerfError(f"marching_cubes: {V} vertices do not fit the int32 faces")
        verts = torch.empty(V, 3, dtype=torch.float32, device=dev)
        nrm = torch.empty(V, 3, dtype=torch.float32, device=dev) if normals else None
        faces = torch.empty(F, 3, dtype=torch.int32, device=dev)
        if V > 0:
            call("ctx_marching_cubes", *args, ptr(verts), ptr(nrm), ptr(faces), 1, stream_ptr(dev))
    return dict(vertices=verts, faces=faces, normals=nrm)


def vertex_colors(net, packed, vertices, normals=None, workspace_bytes=None):
    """``sigmoid(raw[:, :3])`` of ``net`` at each vertex ``[V,3]``, seen along ``-normal`` (``normals`` None: a zero
    view direction): fp32 ``[V,3]`` in [0, 1].  ``workspace_bytes`` sizes the chunks; the result does not depend on
    it."""
    for t in (vertices, normals):
        if t is not None and not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32 and t.dim() == 2
                                  and t.shape[1] == 3):
            raise CtxNerfError("vertex_colors: vertices / normals must be fp32 CUDA tensors [V, 3]")
    if normals is not None and normals.shape != vertices.shape:
        raise CtxNerfError("vertex_colors: normals must match vertices")
    V, dev = vertices.shape[0], vertices.device
    rgb = torch.empty(V, 3, dtype=torch.float32, device=dev)
    if V == 0:
        return rgb
    need = int(_lib.lib().ctx_vertex_colors_workspace(1))
    if workspace_bytes is None:
        workspace_bytes = int(_lib.lib().ctx_vertex_colors_workspace(min(V, 1 << 22)))
    if workspace_bytes < need:
        raise CtxNerfError(f"vertex_colors: the workspace needs at least {need} bytes")
    ws = torch.empty(int(workspace_bytes), dtype=torch.uint8, device=dev)
    vertices = vertices.contiguous()
    normals = normals.contiguous() if normals is not None else None
    cn = _ctxnet(net, packed)
    with torch.cuda.device(dev):
        call("ctx_vertex_colors", ctypes.byref(cn), net.L_pts, net.L_dirs, ptr(vertices), ptr(normals), V, ptr(ws),
             ws.numel(), ptr(rgb), stream_ptr(dev))
    return rgb


def write_ply(path, mesh):
    """Binary little-endian PLY of ``mesh`` (a dict as ``NerfTrainer.extract_mesh`` returns): float x y z, optional
    float nx ny nz (``normals``), optional uchar red green blue (``colors`` in [0, 1], rounded to 0..255), and int32
    triangles (``list uchar int vertex_indices``)."""
    v = np.ascontiguousarray(_host(mesh["vertices"]), dtype="<f4").reshape(-1, 3)
    f = np.ascontiguousarray(_host(mesh["faces"]), dtype="<i4").reshape(-1, 3)
    n, c = mesh.get("normals"), mesh.get("colors")
    fields = [("x", "<f4"), ("y", "<f4"), ("z", "<f4")]
    cols = [v]
    props = ["property float x", "property float y", "property float z"]
    if n is not None:
        fields += [("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4")]
        cols.append(np.asarray(_host(n), dtype="<f4").reshape(-1, 3))
        props += ["property float nx", "property float ny", "property float nz"]
    if c is not None:
        fields += [("red", "u1"), ("green", "u1"), ("blue", "u1")]
        cols.append(np.rint(np.clip(np.asarray(_host(c), dtype=np.float64), 0.0, 1.0) * 255.0).astype(np.uint8)
                    .reshape(-1, 3))
        props += ["property uchar red", "property uchar green", "property uchar blue"]
    vert = np.empty(len(v), dtype=fields)
    names = [name for name, _ in fields]
    for k, col in enumerate(cols):
        for j in range(3):
            vert[names[3 * k + j]] = col[:, j]
    face = np.empty(len(f), dtype=[("n", "u1"), ("idx", "<i4", (3,))])
    face["n"], face["idx"] = 3, f
    head = "\n".join(["ply", "format binary_little_endian 1.0", f"element vertex {len(v)}", *props,
                      f"element face {len(f)}", "property list uchar int vertex_indices", "end_header"]) + "\n"
    with open(path, "wb") as fh:
        fh.write(head.encode("ascii"))
        fh.write(vert.tobytes())
        fh.write(face.tobytes())


def _host(t):
    return t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
