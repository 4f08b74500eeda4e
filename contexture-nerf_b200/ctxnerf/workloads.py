"""Synthetic workloads named by BASELINE.json (shapes only; weights are
random-init, data is synthetic -- there is no network for datasets)."""
from __future__ import annotations

import math

import torch


def orbit_camera(H=800, W=800, focal=1111.1, radius=4.0311, elev_deg=30.0, azim_deg=0.0, target=(0.0, 0.0, 0.0)):
    """Intrinsics K and camera-to-world [3,4] of a camera on a sphere around
    ``target`` looking at it (OpenGL axes: x right, y up, camera looks along -z).
    Defaults: BASELINE config 2 (Blender-lego-like 800x800 view)."""
    K = [[focal, 0.0, 0.5 * W], [0.0, focal, 0.5 * H], [0.0, 0.0, 1.0]]
    e, a = math.radians(elev_deg), math.radians(azim_deg)
    tgt = torch.tensor(target, dtype=torch.float64)
    eye = tgt + radius * torch.tensor([math.cos(e) * math.sin(a), math.sin(e), math.cos(e) * math.cos(a)],
                                      dtype=torch.float64)
    fwd = (tgt - eye) / (tgt - eye).norm()
    right = torch.linalg.cross(fwd, torch.tensor([0.0, 1.0, 0.0], dtype=torch.float64))
    right = right / right.norm()
    up = torch.linalg.cross(right, fwd)
    c2w = torch.stack([right, up, -fwd, eye], dim=1).to(torch.float32)
    return K, c2w


def multiview_cameras(n_views=8, res=1024, radius=1.5, theta_deg=60.0, fovy=math.pi / 3, look_at=(0.0, 0.25, 0.0)):
    """BASELINE config 4: the reference's MultiviewDataset poses
    (/root/reference/src/training/views_dataset.py:158-168: theta 60 deg, phi in
    {0,45,315,90,270,135,225,180}), camera model of src/models/render.py:35-46,
    fovy = pi/3 (trainer.py:253).  Returns [(K, c2w)], bounding sphere (cx,cy,cz,r)
    of the normalised mesh (src/models/mesh.py:53-64: radius shape_scale=0.6, dy=0.25)."""
    phis = [0, 45, 315, 90, 270, 135, 225, 180][:n_views]
    f = 0.5 * res / math.tan(0.5 * fovy)
    out = []
    for phi in phis:
        out.append(orbit_camera(res, res, f, radius, 90.0 - theta_deg, float(phi), look_at))
    return out, (look_at[0], look_at[1], look_at[2], 0.6)


def forward_facing_camera(H=756, W=1008, focal=815.0, yaw=0.08, pitch=-0.05, eye=(0.05, -0.03, 0.1)):
    """K and camera-to-world [3,4] of one view of a recentred forward-facing (LLFF) capture: near the origin, looking
    down -z, slightly turned, so that every ray crosses the NDC near plane z = -1.  Defaults: the size of upstream's
    LLFF images at factor 4."""
    K = [[focal, 0.0, 0.5 * W], [0.0, focal, 0.5 * H], [0.0, 0.0, 1.0]]
    cy, sy, cp, sp = math.cos(yaw), math.sin(yaw), math.cos(pitch), math.sin(pitch)
    ry = torch.tensor([[cy, 0.0, sy], [0.0, 1.0, 0.0], [-sy, 0.0, cy]], dtype=torch.float64)
    rx = torch.tensor([[1.0, 0.0, 0.0], [0.0, cp, -sp], [0.0, sp, cp]], dtype=torch.float64)
    c2w = torch.cat([ry @ rx, torch.tensor(eye, dtype=torch.float64)[:, None]], 1).to(torch.float32)
    return K, c2w
