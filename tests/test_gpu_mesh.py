"""Mesh extraction on the GPU: ctx_marching_cubes against the NumPy restatement bit for bit, ctx_density_grid against
the fused forward and the fp32 oracle network, NerfTrainer.extract_mesh end to end (colours, training left undisturbed,
refusals, PLY), and a fit that shows in the extracted geometry."""
import numpy as np
import pytest
import torch

from ctxnerf.workloads import orbit_camera
from oracle import marching_cubes as mc
from oracle import mc_tables
from oracle import nerf_oracle as orc

pytestmark = pytest.mark.gpu

UNIT = ((0.0, 0.0, 0.0), (1.0, 1.0, 1.0))


def _diag(msg):
    print(msg)        # measured figures: shown with pytest -s


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _against_oracle(cuda, s, iso, bounds):
    from ctxnerf import mesh
    out = mesh.marching_cubes(torch.from_numpy(s).to(cuda), iso, bounds)
    o, h = mesh.lattice(bounds, [n - 1 for n in s.shape])
    v, f, n = mc.marching_cubes(s, iso, o, h)
    gv, gf, gn = (out[k].cpu().numpy() for k in ("vertices", "faces", "normals"))
    assert gf.dtype == np.int32 and np.array_equal(gf, f)
    assert np.array_equal(_bits(gv), _bits(v))
    assert np.abs(gn - n).max(initial=0.0) <= 1e-6
    return out


# ---------------------------------------------------------------- 1. marching cubes against the oracle
def test_every_single_cell_case(cuda):
    rng = np.random.default_rng(0)
    for case in range(256):
        inside = np.array([case >> c & 1 for c in range(8)], bool).reshape(2, 2, 2, order="F")
        s = np.where(inside, 0.5 + 0.5 * rng.random((2, 2, 2)), 0.49 * rng.random((2, 2, 2))).astype(np.float32)
        out = _against_oracle(cuda, s, 0.5, UNIT)
        assert out["faces"].shape[0] == mc_tables.table()[1][case]


def _field(n, fn, lo, hi):
    o, h = mc.spacing(lo, hi, n)
    x = [mc.lattice_axis(n[a] + 1, o[a], h[a]).astype(np.float64) for a in range(3)]
    return fn(*np.meshgrid(*x, indexing="ij")).astype(np.float32)


@pytest.mark.parametrize("kind", ["random17", "sphere64", "torus64", "aniso"])
def test_lattices_against_the_oracle(cuda, kind):
    B = ((-1.0,) * 3, (1.0,) * 3)
    if kind == "random17":
        s, iso = np.random.default_rng(1).random((17, 17, 17), dtype=np.float32), 0.5
    elif kind == "sphere64":
        s, iso = _field((64,) * 3, lambda X, Y, Z: 0.7 - np.sqrt(X * X + Y * Y + Z * Z), *B), 0.0
    elif kind == "torus64":
        s, iso = _field((64,) * 3, lambda X, Y, Z: 0.2 - np.sqrt((np.sqrt(X * X + Y * Y) - 0.55) ** 2 + Z * Z), *B), 0.0
    else:       # 129 x 65 x 33 points, anisotropic spacing, a wavy ellipsoid of density
        B = ((-1.2, -0.6, -0.3), (1.2, 0.6, 0.3))
        s = _field((128, 64, 32), lambda X, Y, Z: 60.0 * (1.0 - (X / 1.0) ** 2 - (Y / 0.5) ** 2 - (Z / 0.25) ** 2)
                   + 8.0 * np.sin(9 * X) * np.cos(7 * Y), *B)
        s, iso = np.maximum(s, 0.0), 50.0
    out = _against_oracle(cuda, s, iso, B)
    _diag(f"marching cubes {kind}: {out['vertices'].shape[0]} vertices, {out['faces'].shape[0]} faces")


def _edge_use_gpu(faces):
    """(times used, directed balance) per undirected edge, on the device"""
    f = faces.long()
    d = torch.cat([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    lo, hi = d.min(1).values, d.max(1).values
    key = lo * (int(hi.max()) + 1) + hi
    uk, inv, cnt = torch.unique(key, return_inverse=True, return_counts=True)
    bal = torch.zeros(len(uk), dtype=torch.int64, device=f.device)
    bal.scatter_add_(0, inv, torch.where(d[:, 0] < d[:, 1], 1, -1))
    return cnt, bal


def test_512_cube_lattice(cuda):
    """A sphere of radius 1 over [-1.2, 1.2]^3 at 512^3 cells (135 M points, 0.5 GB of sigma: more than L2): a closed,
    consistently oriented mesh of genus 0 enclosing 4/3 pi, vertices within h^2 of the sphere, repeat runs
    bit-identical, and a block of 33^3 points bit-equal to the oracle's mesh of that block."""
    from ctxnerf import mesh
    n, B = 512, ((-1.2,) * 3, (1.2,) * 3)
    o, h = mesh.lattice(B, (n, n, n))
    ax = torch.from_numpy(mc.lattice_axis(n + 1, o[0], h[0])).to(cuda).double()
    s = (1.0 - torch.sqrt(ax[:, None, None] ** 2 + ax[None, :, None] ** 2 + ax[None, None, :] ** 2)).float()
    a = mesh.marching_cubes(s, 0.0, B)
    b = mesh.marching_cubes(s, 0.0, B)
    for k in ("vertices", "faces", "normals"):
        assert torch.equal(a[k], b[k]), k
    v, f = a["vertices"], a["faces"]
    cnt, bal = _edge_use_gpu(f)
    assert bool((cnt == 2).all()) and bool((bal == 0).all())
    assert v.shape[0] - cnt.numel() + f.shape[0] == 2
    t = v.double()[f.long()]
    vol = float((t[:, 0] * torch.linalg.cross(t[:, 1], t[:, 2])).sum() / 6.0)
    err = float((v.double().norm(dim=1) - 1.0).abs().max())
    _diag(f"512^3 sphere: {v.shape[0]} vertices, {f.shape[0]} faces, volume {vol:.6f} vs {4 / 3 * np.pi:.6f}, "
          f"max radius error {err:.2e} (h^2 = {h[0] ** 2:.2e})")
    assert abs(vol / (4.0 / 3.0 * np.pi) - 1.0) < 1e-3 and err < h[0] ** 2
    # a block of the lattice where the surface passes, against the oracle, in whole-lattice ids
    i0, j0, k0, m = 460, 240, 240, 33
    blk = s[i0:i0 + m, j0:j0 + m, k0:k0 + m].cpu().numpy()
    bv, bf, _ = mc.marching_cubes(blk, 0.0, o, h, with_normals=False, index_offset=(i0, j0, k0))
    assert len(bf) > 100
    inside = s >= 0
    M = torch.zeros(s.shape + (3,), dtype=torch.bool, device=cuda)
    M[:-1, :, :, 0] = inside[:-1] != inside[1:]
    M[:, :-1, :, 1] = inside[:, :-1] != inside[:, 1:]
    M[:, :, :-1, 2] = inside[:, :, :-1] != inside[:, :, 1:]
    ids = (torch.cumsum(M.reshape(-1), 0) - 1).reshape(M.shape)
    del M
    bm = torch.from_numpy(mc.edge_mask(blk, 0.0)).to(cuda)
    gid = ids[i0:i0 + m, j0:j0 + m, k0:k0 + m][bm]                        # block vertex -> whole-lattice id
    del ids
    assert np.array_equal(_bits(v[gid].cpu().numpy()), _bits(bv))
    # the faces of the block's cells: offsets from the per-cell triangle counts
    tab, ntri = mc_tables.table()
    cs = torch.zeros((n, n, n), dtype=torch.int64, device=cuda)
    for c, (dx, dy, dz) in enumerate(mc_tables.CORNERS):
        cs |= inside[dx:dx + n, dy:dy + n, dz:dz + n].long() << c
    nt = torch.from_numpy(ntri).to(cuda)[cs]
    first = (torch.cumsum(nt.reshape(-1), 0) - nt.reshape(-1)).reshape(nt.shape)
    cells = (slice(i0, i0 + m - 1), slice(j0, j0 + m - 1), slice(k0, k0 + m - 1))
    rows = torch.repeat_interleave(first[cells].reshape(-1), nt[cells].reshape(-1))
    rows = rows + torch.arange(len(rows), device=cuda) - torch.repeat_interleave(
        torch.cumsum(nt[cells].reshape(-1), 0) - nt[cells].reshape(-1), nt[cells].reshape(-1))
    assert torch.equal(f[rows].long(), gid[torch.from_numpy(bf).to(cuda).long()])


# ---------------------------------------------------------------- 2. the density lattice
def _trainer(cuda, **kw):
    from ctxnerf.train import NerfTrainer
    K, c2w = orbit_camera(32, 32, focal=40.0)
    torch.manual_seed(3)
    return NerfTrainer(32, 32, K, c2w, N_samples=16, N_importance=16, device=cuda, seed=2, **kw)


def _params(net):
    return {k: v.detach().cpu() for k, v in net.state_dict().items()}


def test_density_grid_is_the_fused_forward_on_the_lattice(cuda):
    from ctxnerf import mesh
    from ctxnerf.mlp import launch_fwd
    tr = _trainer(cuda)
    cells, B = (20, 17, 33), ((-1.2, -0.9, -1.5), (1.1, 1.3, 0.7))
    o, h = mesh.lattice(B, cells)
    X, Y, Z = (c + 1 for c in cells)
    for net in (tr.fine, tr.coarse):
        sigma = tr.density_grid(cells, B, network="fine" if net is tr.fine else "coarse")
        assert sigma.shape == (X, Y, Z) and sigma.dtype == torch.float32
        xs = [torch.from_numpy(mc.lattice_axis(n, o[a], h[a])) for a, n in enumerate((X, Y, Z))]
        ro = torch.stack([xs[0][:, None].expand(X, Y), xs[1][None, :].expand(X, Y), torch.zeros(X, Y)], -1)
        ro = ro.reshape(-1, 3).contiguous().to(cuda)
        rd = torch.tensor([0.0, 0.0, 1.0]).expand(X * Y, 3).contiguous().to(cuda)
        vd = torch.zeros(X * Y, 3, device=cuda)
        z = xs[2][None, :].expand(X * Y, Z).contiguous().to(cuda)
        raw = torch.empty(X * Y * Z, 4, device=cuda)
        launch_fwd(net, tr._pk[net], raw, rays=(ro, rd, vd, z))
        assert torch.equal(sigma.reshape(-1), raw[:, 3].clamp_min(0.0))
        # the fp32 oracle network at the lattice points, zero view directions
        pts = torch.stack(torch.meshgrid(*xs, indexing="ij"), -1).reshape(X * Y, Z, 3)
        ref = orc.run_network(pts, torch.zeros(X * Y, 3), _params(net))[..., 3].clamp_min(0.0)
        err = float((sigma.cpu().reshape(X * Y, Z) - ref).abs().max())
        _diag(f"density_grid vs the fp32 oracle: max |err| {err:.2e} (sigma up to {float(ref.max()):.3f})")
        assert err <= 2e-2
    # the slab size does not change a bit
    from ctxnerf import _lib
    need = int(_lib.lib().ctx_density_grid_workspace(*cells))
    small = mesh.density_grid(tr.fine, tr._pk[tr.fine], cells, B, workspace_bytes=need)
    mid = mesh.density_grid(tr.fine, tr._pk[tr.fine], cells, B, workspace_bytes=7 * need + 1000)
    assert torch.equal(small, tr.density_grid(cells, B)) and torch.equal(mid, small)


# ---------------------------------------------------------------- 3. extract_mesh
def _threshold(sigma):
    pos = sigma[sigma > 0]
    return float(pos.median()) if pos.numel() else 1.0


def test_extract_mesh_end_to_end(cuda, tmp_path):
    from ctxnerf import mesh
    tr = _trainer(cuda)
    B = ((-1.0, -1.0, -1.0), (1.0, 1.0, 1.0))
    sigma = tr.density_grid(40, B)
    thr = _threshold(sigma)
    m = tr.extract_mesh(40, B, threshold=thr)
    ref = mesh.marching_cubes(sigma, thr, B)
    for k in ("vertices", "faces", "normals"):
        assert torch.equal(m[k], ref[k]), k
    V = m["vertices"].shape[0]
    assert V > 100 and m["colors"].shape == (V, 3)
    # colours: sigmoid of the oracle network at the vertices, seen along -normal
    want = torch.sigmoid(orc.run_network(m["vertices"].cpu()[:, None], -m["normals"].cpu(), _params(tr.fine))[:, 0, :3])
    err = float((m["colors"].cpu() - want).abs().max())
    _diag(f"extract_mesh: {V} vertices at threshold {thr:.3f}; colours vs the oracle max |err| {err:.2e}")
    assert err <= 2e-2
    # chunked colouring gives the same bits
    small = mesh.vertex_colors(tr.fine, tr._pk[tr.fine], m["vertices"], m["normals"], workspace_bytes=200_000)
    assert torch.equal(small, m["colors"])
    assert tr.extract_mesh(40, B, threshold=thr, colors=False)["colors"] is None
    # PLY round trip
    path = tmp_path / "mesh.ply"
    mesh.write_ply(str(path), m)
    got = _read_ply(str(path))
    assert np.array_equal(got["vertices"], m["vertices"].cpu().numpy())
    assert np.array_equal(got["normals"], m["normals"].cpu().numpy())
    assert np.array_equal(got["faces"], m["faces"].cpu().numpy())
    assert np.array_equal(got["colors"], np.rint(m["colors"].cpu().numpy().astype(np.float64) * 255).astype(np.uint8))


def _read_ply(path):
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    head = data[:end].decode().splitlines()
    assert head[1] == "format binary_little_endian 1.0"
    nv = int(next(ln for ln in head if ln.startswith("element vertex")).split()[-1])
    nf = int(next(ln for ln in head if ln.startswith("element face")).split()[-1])
    props = [ln.split() for ln in head if ln.startswith("property ") and "list" not in ln]
    dt = np.dtype([(p[2], "<f4" if p[1] == "float" else "u1") for p in props])
    vert = np.frombuffer(data, dt, nv, end)
    face = np.frombuffer(data, np.dtype([("n", "u1"), ("idx", "<i4", (3,))]), nf, end + nv * dt.itemsize)
    assert (face["n"] == 3).all() and end + nv * dt.itemsize + nf * 13 == len(data)
    cols = lambda *ks: np.stack([vert[k] for k in ks], 1)   # noqa: E731
    return dict(vertices=cols("x", "y", "z"), normals=cols("nx", "ny", "nz"), colors=cols("red", "green", "blue"),
                faces=face["idx"].copy())


def test_extract_mesh_does_not_disturb_training(cuda):
    from ctxnerf.train import NerfTrainer
    H = W = 32
    cams = [orbit_camera(H, W, focal=40.0, azim_deg=a) for a in (0.0, 120.0, 240.0)]
    poses = torch.stack([c for _, c in cams])
    images = torch.rand(3, H, W, 3, generator=torch.Generator().manual_seed(1))
    runs = []
    for with_mesh in (True, False):
        torch.manual_seed(6)
        tr = NerfTrainer(H, W, cams[0][0], poses, images=images, N_samples=32, N_importance=32, device=cuda, seed=5)
        losses = [tr.step_random(256).item() for _ in range(3)]
        if with_mesh:
            pl = tr._plans[(256, "draw")]
            assert pl.graph is not None
            torch.cuda.synchronize()
            before = dict(ctr=tr._ctr.clone(), loss=tr._loss.clone(), m=tr.exp_avg.clone(), v=tr.exp_avg_sq.clone(),
                          flat=tr.bucket.flat.clone(), rng=torch.random.get_rng_state(),
                          cuda_rng=torch.cuda.get_rng_state(cuda), graph=pl.graph, plans=dict(tr._plans),
                          pk={n: [t.clone() for t in tr._pk[n]] for n in (tr.coarse, tr.fine)})
            sigma = tr.density_grid(32)
            m = tr.extract_mesh(32, threshold=_threshold(sigma))
            torch.cuda.synchronize()
            assert m["vertices"].shape[0] > 0
            assert torch.equal(tr._ctr, before["ctr"]) and torch.equal(tr._loss, before["loss"])
            assert torch.equal(tr.exp_avg, before["m"]) and torch.equal(tr.exp_avg_sq, before["v"])
            assert torch.equal(tr.bucket.flat, before["flat"])
            assert torch.equal(torch.random.get_rng_state(), before["rng"])
            assert torch.equal(torch.cuda.get_rng_state(cuda), before["cuda_rng"])
            assert tr._plans == before["plans"] and pl.graph is before["graph"]
            for n in (tr.coarse, tr.fine):
                assert all(torch.equal(a, b) for a, b in zip(tr._pk[n], before["pk"][n]))
        losses += [tr.step_random(256).item() for _ in range(3)]
        torch.cuda.synchronize()
        runs.append((losses, tr.bucket.flat.clone()))
    (l1, p1), (l2, p2) = runs
    assert l1 == l2, (l1, l2)
    assert torch.equal(p1, p2)


def test_refusals(cuda):
    from ctxnerf._lib import CtxNerfError
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import forward_facing_camera
    K, c2w = forward_facing_camera(24, 32, focal=30.0)
    ff = NerfTrainer(24, 32, K, c2w, near=0.0, far=1.0, N_samples=8, N_importance=8, ndc=True, device=cuda)
    for call in (lambda: ff.extract_mesh(8), lambda: ff.density_grid(8)):
        with pytest.raises(CtxNerfError, match="ndc"):
            call()
    tr = _trainer(cuda)
    for kw in (dict(threshold=0.0), dict(threshold=-1.0), dict(network="medium"),
               dict(bounds=((0, 0, 0), (0, 1, 1))), dict(bounds=((1, 1, 1), (-1, -1, -1))), dict(resolution=0),
               dict(resolution=1025)):
        with pytest.raises(CtxNerfError):
            tr.extract_mesh(**{"resolution": 8, **kw})


# ---------------------------------------------------------------- 4. a fit shows in the geometry
def _sphere_image(H, W, K, c2w, radius=1.0):
    """a coloured sphere at the origin (colour 0.5 + 0.5 * normal) on white, rendered analytically"""
    ro, rd = orc.get_rays(H, W, K, c2w)
    ro, rd = ro.double(), rd.double()
    a, b = (rd * rd).sum(-1), (ro * rd).sum(-1)
    disc = b * b - a * ((ro * ro).sum(-1) - radius ** 2)
    t = (-b - disc.clamp_min(0).sqrt()) / a
    nrm = (ro + t[..., None] * rd) / radius
    return torch.where((disc > 0)[..., None], 0.5 + 0.5 * nrm, torch.ones_like(nrm)).clamp(0, 1).float()


def test_a_fit_shows_in_the_geometry(cuda):
    """The coloured unit sphere at 32 x 32 from 24 orbit poses (8 azimuths at elevations -30, 15 and 60 degrees), 800
    step_random steps of 512 rays, then extract_mesh at 64^3 over [-1.2, 1.2]^3 with a threshold of a quarter of the
    density's 0.999 quantile on the lattice (a small fit's densities need not reach upstream's 50).  The box corners
    lie outside most views, and the fit leaves stray density there, so the radius is measured inside the ball the
    lattice inscribes.

    Measured on a B200: 36 593 vertices, 18 523 of them inside radius 1.2 with a median radius of 0.904 (the fit also
    puts surfaces inside the sphere, which no view sees); no open edge off the lattice border.  The bar (0.2) leaves
    a wide margin."""
    from ctxnerf.train import NerfTrainer
    H = W = 32
    cams = [orbit_camera(H, W, focal=40.0, azim_deg=a, elev_deg=e) for e in (-30.0, 15.0, 60.0)
            for a in range(0, 360, 45)]
    K = cams[0][0]
    poses = torch.stack([c for _, c in cams])
    images = torch.stack([_sphere_image(H, W, K, c) for _, c in cams])
    torch.manual_seed(1)
    tr = NerfTrainer(H, W, K, poses, images=images, N_samples=64, N_importance=64, precrop_iters=50,
                     precrop_frac=0.75, device=cuda, seed=1)
    for _ in range(800):
        tr.step_random(512)
    sigma = tr.density_grid(64)
    thr = 0.25 * float(torch.quantile(sigma.reshape(-1), 0.999))
    m = tr.extract_mesh(64, threshold=thr)
    v, f = m["vertices"], m["faces"]
    _, bal = _edge_use_gpu(f)
    fl = f.long()
    d = torch.cat([fl[:, [0, 1]], fl[:, [1, 2]], fl[:, [2, 0]]])
    base = int(d.max()) + 1
    uk = torch.unique(d.min(1).values * base + d.max(1).values)
    border = (v.abs() >= 1.2 - 1e-6).any(1)
    inner = ~(border[uk // base] & border[uk % base])
    rad = v.norm(dim=1)
    ball = rad < 1.2          # the ball inscribed in the lattice: unobserved corners of the box hold stray density
    med = float(rad[ball].median())
    _diag(f"fit geometry: threshold {thr:.2f}, {v.shape[0]} vertices ({int(ball.sum())} inside radius 1.2), "
          f"{f.shape[0]} faces, median radius inside the ball {med:.4f}, {int((bal != 0).sum())} open edge(s) with "
          f"{int(border.sum())} vertices on the border")
    assert bool((bal[inner] == 0).all())
    assert int(ball.sum()) > 1000 and abs(med - 1.0) < 0.2
