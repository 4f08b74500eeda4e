"""Multi-view training in NerfTrainer: ray generation over a pose stack (ctx_raygen_views), ray batches drawn and their
targets gathered on the device (ctx_draw_rays), step_random inside the captured step, and render(c2w=...)."""
import os

import numpy as np
import pytest
import torch

from ctxnerf.workloads import forward_facing_camera, orbit_camera
from oracle import nerf_oracle as orc

pytestmark = pytest.mark.gpu


def _diag(msg):
    print(msg)        # measured figures: shown with pytest -s


# ---------------------------------------------------------------- restatement of csrc/raybatch.cu
_M32 = np.uint64(0xFFFFFFFF)


def _philox_x(key, c0, c1, c2, c3):
    """word x of Philox4x32-10 (ctx::Philox) for counter words (c0, c1, c2, c3), vectorised over numpy uint64 arrays"""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _M32 for c in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0, k1 = np.uint64(key & 0xFFFFFFFF), np.uint64((key >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
    return c0


def _perm(key, tweak, x, n):
    """pi(x) over [0, n): 4-round Feistel on the smallest even bit width b >= 2 covering n, round function word x of
    Philox(key) at counter (v, tweak, i + 1, 4), cycle-walking back into [0, n)"""
    b = 2
    while b < 32 and (1 << b) < n:
        b += 2
    h, m = np.uint64(b // 2), np.uint64((1 << (b // 2)) - 1)
    x = np.asarray(x, dtype=np.uint64)
    tweak = np.broadcast_to(np.asarray(tweak, dtype=np.uint64), x.shape)

    def feistel(x, tw):
        L, R = x >> h, x & m
        for i in range(4):
            f = _philox_x(key, R, tw, i + 1, 4) & m
            L, R = R, L ^ f
        return (L << h) | R

    y = feistel(x, tweak)
    while True:
        bad = y >= np.uint64(n)
        if not bad.any():
            return y
        y[bad] = feistel(y[bad], tweak[bad])


def _draw_ref(mode, n_views, H, W, R, seed, ctr, rank=0, world=1, precrop_iters=0, crop=(0, 0)):
    c0, t = ctr
    r = np.arange(R, dtype=np.uint64)
    if mode == 0:
        key = (seed + c0) % 2 ** 64
        v = int((int(_philox_x(key, 0, rank, 0, 4)) * n_views) >> 32)
        if t < precrop_iters:
            ch, cw, y0, x0 = 2 * crop[0], 2 * crop[1], H // 2 - crop[0], W // 2 - crop[1]
        else:
            ch, cw, y0, x0 = H, W, 0, 0
        q = _perm(key, rank, r, ch * cw).astype(np.int64)
        return v * H * W + (y0 + q // cw) * W + x0 + q % cw
    n = n_views * H * W
    pos = ((t - 1) * world + rank) * R + r.astype(np.int64)
    e = pos // n
    return _perm(seed, e & 0xFFFFFFFF, pos % n, n).astype(np.int64)


def _draw(cuda, images, n_views, H, W, R, seed, ctr, **kw):
    from ctxnerf import ops
    c = torch.tensor(ctr, dtype=torch.int64, device=cuda)
    return ops.draw_rays(n_views, H, W, R, c, images=images, seed=seed, **kw)


# ---------------------------------------------------------------- 1. raygen over a pose stack
def _ff_stack(n, H, W, focal, rows=3):
    poses = []
    for v in range(n):
        _, c = forward_facing_camera(H, W, focal, yaw=0.08 - 0.05 * v, pitch=-0.05 + 0.03 * v,
                                     eye=(0.05 * v, -0.03, 0.1 - 0.02 * v))
        poses.append(c)
    p = torch.stack(poses)
    if rows == 4:
        p = torch.cat([p, torch.tensor([0.0, 0.0, 0.0, 1.0]).expand(n, 1, 4)], 1)
    K, _ = forward_facing_camera(H, W, focal)
    return K, p


@pytest.mark.parametrize("rows", [3, 4])
@pytest.mark.parametrize("ndc", [False, True])
def test_raygen_over_a_pose_stack_equals_one_pose_per_view(cuda, rows, ndc):
    from ctxnerf import ops
    H, W, N, R, S = 40, 56, 4, 3000, 64
    K, poses = _ff_stack(N, H, W, 45.0, rows)
    poses = poses.to(cuda)
    ids = torch.randint(0, N * H * W, (R,), generator=torch.Generator().manual_seed(rows + 2 * ndc)).to(cuda)
    assert len(set((ids // (H * W)).tolist())) >= 3
    kw = dict(n_samples=S, near=0.0 if ndc else 0.5, far=1.0 if ndc else 4.0, perturb=True, seed=1234,
              ndc=(float(K[0][0]), 1.0) if ndc else None, want_viewdirs=True)
    got = ops.raygen(H, W, K, poses, ray_idx=ids, **kw)
    view, pix = ids // (H * W), ids % (H * W)
    for v in range(N):
        want = ops.raygen(H, W, K, poses[v], ray_idx=pix, **kw)      # the same batch rows: the same jitter
        rows_v = view == v
        for name in ("rays_o", "rays_d", "viewdirs", "z_vals"):
            assert torch.equal(got[name][rows_v], want[name][rows_v]), (v, name)


# ---------------------------------------------------------------- 2. the draw equals its restatement
@pytest.mark.parametrize("mode", [0, 1])
def test_draw_equals_the_restatement(cuda, mode):
    N, H, W, R = 5, 24, 40, 200                                    # (the centre crop has 12 x 20 pixels)
    g = torch.Generator().manual_seed(mode)
    images = torch.rand(N, H, W, 3, generator=g).to(cuda)
    seed = 0x5DEECE66D1234567
    crop = (6, 10)
    for t in (1, 2, 3, 7, 40):
        for rank in (0, 1):
            for precrop in ((0, 10) if mode == 0 else (0,)):
                ctr = (2 * t + 11, t)
                kw = dict(mode=mode, rank=rank, world=2, precrop_iters=precrop, crop=crop)
                idx, tgt = _draw(cuda, images, N, H, W, R, seed, ctr, **kw)
                want = _draw_ref(mode, N, H, W, R, seed, ctr, rank=rank, world=2, precrop_iters=precrop, crop=crop)
                assert np.array_equal(idx.cpu().numpy(), want), (t, rank, precrop)
                v, y, x = idx // (H * W), (idx % (H * W)) // W, idx % W
                assert torch.equal(tgt, images[v, y, x])
    ids, none = _draw(cuda, None, N, H, W, R, seed, (4, 2), mode=mode)           # ids only
    assert none is None and np.array_equal(ids.cpu().numpy(), _draw_ref(mode, N, H, W, R, seed, (4, 2)))


# ---------------------------------------------------------------- 3. draw properties
def test_one_view_draw_properties(cuda):
    N, H, W, R = 5, 32, 48, 384
    crop = (int(H // 2 * 0.5), int(W // 2 * 0.5))                # 8 x 12 half-extents: 16 x 24 = 384 pixels
    counts = np.zeros(N)
    outside = 0
    for t in range(1, 601):
        idx, _ = _draw(cuda, None, N, H, W, R, 99, (2 * t, t), precrop_iters=5, crop=crop)
        ids = idx.cpu().numpy()
        assert len(np.unique(ids)) == ids.size, t                  # without replacement
        v, y, x = ids // (H * W), (ids % (H * W)) // W, ids % W
        assert (v == v[0]).all()                                   # one image per step
        counts[v[0]] += 1
        inside = (y >= H // 2 - crop[0]) & (y < H // 2 + crop[0]) & (x >= W // 2 - crop[1]) & (x < W // 2 + crop[1])
        if t < 5:
            assert inside.all()                                    # the whole crop, each pixel once
        else:
            outside += int((~inside).sum())
    assert outside > 0.5 * 595 * R * (1 - 384 / (H * W))          # after precrop_iters the whole image is drawn
    chi2 = float(((counts - counts.mean()) ** 2 / counts.mean()).sum())
    _diag(f"mode 0 view counts over 600 steps: {counts.tolist()}, chi2 {chi2:.2f} (4 dof)")
    assert chi2 < 25.0                                              # p ~ 5e-5 for a fair draw


@pytest.mark.parametrize("R", [128, 100])
def test_epoch_stream_draws_every_ray_once_per_epoch(cuda, R):
    N, H, W = 3, 16, 16
    n = N * H * W
    for world in (1, 2):
        stream = []
        t = 1
        while len(stream) < 3 * n + 2 * R:
            for rank in range(world):
                idx, _ = _draw(cuda, None, N, H, W, R, 777, (2 * t, t), mode=1, rank=rank, world=world)
                stream.extend(idx.cpu().tolist())
            t += 1
        epochs = [stream[e * n:(e + 1) * n] for e in range(3)]
        for e in epochs:                                            # each ray once per epoch, over every rank
            assert sorted(e) == list(range(n)), (world, R)
        assert epochs[0] != epochs[1] and epochs[1] != epochs[2]    # reshuffled


# ---------------------------------------------------------------- 4. gradients against the oracle
def _mv_trainer(cuda, N=3, H=32, W=32, focal=30.0, images=None, **kw):
    from ctxnerf.train import NerfTrainer
    K, poses = _ff_stack(N, H, W, focal)
    args = dict(near=0.0, far=1.0, N_samples=64, N_importance=64, perturb=0.0, white_bkgd=False, ndc=True,
                device=cuda, seed=3)
    args.update(kw)
    return NerfTrainer(H, W, K, poses, images=images, **args), K, poses


def _params(net):
    return {k: v.detach().cpu().clone().requires_grad_(True) for k, v in net.state_dict().items()}


def _oracle_rays(tr, K, poses, ids):
    """upstream's per-view rays: get_rays with the pose of each ray's view, view directions, then the NDC warp"""
    HW = tr.H * tr.W
    o = torch.empty(ids.numel(), 3)
    d = torch.empty(ids.numel(), 3)
    for v in range(poses.shape[0]):
        sel = (ids // HW) == v
        ro, rd = orc.get_rays(tr.H, tr.W, K, poses[v])
        o[sel] = ro.reshape(-1, 3)[ids[sel] % HW]
        d[sel] = rd.reshape(-1, 3)[ids[sel] % HW]
    vd = d / torch.norm(d, dim=-1, keepdim=True)
    o, d = orc.ndc_rays(tr.H, tr.W, K[0][0], 1.0, o, d)
    return o, d, vd


def _check_step_against_oracle(tr, K, poses, ids, tgt, loss, prc, prf, what):
    R, S, Ni = ids.numel(), tr.N_samples, tr.N_importance
    o, d, vd = _oracle_rays(tr, K, poses, ids)
    batch = torch.cat([o, d, torch.zeros(R, 1), torch.ones(R, 1), vd], -1)
    q = lambda pts, v, prm: orc.run_network(pts, v, prm, bf16_operands=True)
    ref = orc.render_rays(batch, prc, q, S, N_importance=Ni, network_fine=prf, white_bkgd=False)
    ref_loss = orc.img2mse(ref["rgb_map"], tgt) + orc.img2mse(ref["rgb0"], tgt)
    ref_loss.backward()
    _diag(f"{what}: loss {loss:.6f} vs oracle {ref_loss.item():.6f}")
    assert abs(loss - ref_loss.item()) < 2e-2 * abs(ref_loss.item())
    for tag, net, pr in (("coarse", tr.coarse, prc), ("fine", tr.fine, prf)):
        got = torch.cat([p.grad.reshape(-1).cpu() for _, p in net.named_parameters()])
        want = torch.cat([pr[name].grad.reshape(-1) for name, _ in net.named_parameters()])
        l2 = (got - want).norm().item() / want.norm().item()
        cos = torch.nn.functional.cosine_similarity(got, want, dim=0).item()
        _diag(f"{what} {tag}: whole-gradient l2-rel err {l2:.3e}, cosine {cos:.6f}")
        assert l2 < 2e-2 and cos > 0.999, (tag, l2, cos)


def test_multiview_steps_against_the_oracle(cuda):
    """step(global ids) and step_random (the batch it drew, from the plan) vs autograd through the oracle chain with
    each ray's own pose (the bars of test_ndc_step_against_the_oracle)."""
    N, H, W, R = 3, 32, 32, 256
    images = torch.rand(N, H, W, 3, generator=torch.Generator().manual_seed(5))
    torch.manual_seed(4)
    tr, K, poses = _mv_trainer(cuda, N, H, W, images=images)
    with torch.no_grad():            # a density the coarse pass resolves (see test_ndc_step_against_the_oracle)
        for net in (tr.coarse, tr.fine):
            net.alpha_linear.bias.fill_(2.0)
        tr._repack()
    ids = torch.randperm(N * H * W, generator=torch.Generator().manual_seed(1))[:R]
    tgt = torch.rand(R, 3, generator=torch.Generator().manual_seed(2))
    prc, prf = _params(tr.coarse), _params(tr.fine)
    loss = tr.step(ids.to(cuda), tgt.to(cuda), optimizer_step=False).item()
    _check_step_against_oracle(tr, K, poses, ids, tgt, loss, prc, prf, "multi-view step")

    prc, prf = _params(tr.coarse), _params(tr.fine)
    loss = tr.step_random(R, optimizer_step=False).item()
    pl = tr._plans[(R, "draw")]
    ids, tgt = pl.idx.cpu(), pl.target.cpu()
    v = ids // (H * W)
    assert (v == v[0]).all() and len(set(ids.tolist())) == R
    assert torch.equal(tgt, images[v, (ids % (H * W)) // W, ids % W])
    _check_step_against_oracle(tr, K, poses, ids, tgt, loss, prc, prf, "step_random")


# ---------------------------------------------------------------- 5. captured == eager
@pytest.mark.parametrize("no_batching", [True, False])
def test_captured_step_random_equals_eager(cuda, no_batching):
    N, H, W, R = 3, 48, 48, 512                                     # (the centre crop has 24 x 24 pixels)
    images = torch.rand(N, H, W, 3, generator=torch.Generator().manual_seed(9))
    res = {}
    for mode in ("graph", "eager"):
        os.environ["CTXNERF_GRAPH"] = "1" if mode == "graph" else "0"
        try:
            torch.manual_seed(7)
            tr, _, _ = _mv_trainer(cuda, N, H, W, 40.0, images=images, N_importance=128, perturb=1.0,
                                   raw_noise_std=1.0, lrate_decay=250, no_batching=no_batching,
                                   precrop_iters=2 if no_batching else 0)
        finally:
            del os.environ["CTXNERF_GRAPH"]
        p0 = tr.bucket.flat.clone()
        pl = tr._plan(R, draw=True)
        batches, losses, snap = [], [], None
        for s in range(5):
            losses.append(tr.step_random(R).item())
            batches.append((pl.idx.clone(), pl.target.clone()))
            if s == 1:
                torch.cuda.synchronize()
                snap = (tr.bucket.grad.clone(), tr.exp_avg.clone(), tr.bucket.flat.clone())
        torch.cuda.synchronize()
        assert (pl.graph is not None) == (mode == "graph")
        assert tr._ctr.tolist() == [10, 5]
        assert all(l == l for l in losses) and torch.isfinite(tr.bucket.flat).all()
        res[mode] = (losses, batches, snap, p0)
    (gl, gb, (gg, gm, gp), p0), (el, eb, (eg, em, ep), _) = res["graph"], res["eager"]
    for (gi, gt), (ei, et) in zip(gb, eb):       # the same draws: two trainers built under one torch seed
        assert torch.equal(gi, ei) and torch.equal(gt, et)
    for a, b in zip(gb, gb[1:]):                  # every replay draws a fresh batch
        assert not torch.equal(a[0], b[0])
    assert abs(gl[0] - el[0]) <= 1e-6 * abs(el[0]) and abs(gl[1] - el[1]) <= 1e-5 * abs(el[1]), (gl, el)
    gerr = (gg - eg).abs().max().item() / eg.abs().max().item()
    merr = (gm - em).abs().max().item() / em.abs().max().item()
    step_size = (ep - p0).abs().max().item()
    off = ((gp - ep).abs() > 0.05 * step_size).float().mean().item()
    _diag(f"captured vs eager step_random (no_batching={no_batching}): grad max rel diff {gerr:.3e}, exp_avg "
          f"{merr:.3e}; {100 * off:.3f} % of the parameters differ by more than 5 % of the update size")
    assert gerr < 1e-4 and merr < 1e-4
    assert off < 0.05


# ---------------------------------------------------------------- 6. one pose changes nothing
def test_a_single_pose_stack_changes_nothing(cuda, monkeypatch):
    from ctxnerf import ops, train
    from ctxnerf.train import NerfTrainer
    H = W = 32
    K, c2w = orbit_camera(H, W, focal=40.0)
    idx = torch.arange(0, H * W, 2, device=cuda)
    tgts = [torch.rand(idx.numel(), 3, generator=torch.Generator().manual_seed(s)).to(cuda) for s in range(3)]
    out = []
    for pose in (c2w, c2w[None]):
        names = []
        real = train.call

        def rec(name, *a):
            names.append(name)
            return real(name, *a)

        monkeypatch.setattr(train, "call", rec)
        monkeypatch.setattr(ops, "call", rec)
        torch.manual_seed(5)
        tr = NerfTrainer(H, W, K, pose, N_samples=32, N_importance=32, device=cuda, seed=2)
        losses = [tr.step(idx, t).item() for t in tgts]
        monkeypatch.undo()
        assert "ctx_raygen_fwd" in names and "ctx_raygen_views" not in names
        r = tr.render(idx)
        torch.cuda.synchronize()
        out.append((names, losses, tr.bucket.flat.clone(), r["rgb_map"], r["depth_map"], tuple(tr.c2w.shape)))
    (n1, l1, p1, rgb1, d1, s1), (n2, l2, p2, rgb2, d2, s2) = out
    assert n1 == n2 and l1 == l2 and s1 == s2 == (3, 4)
    assert torch.equal(p1, p2) and torch.equal(rgb1, rgb2) and torch.equal(d1, d2)


# ---------------------------------------------------------------- 7. render(c2w=...)
def test_render_of_a_pose_equals_the_kernel_sequence(cuda):
    from ctxnerf import ops
    from ctxnerf.mlp import launch_fwd
    for ndc in (True, False):
        tr, K, poses = _mv_trainer(cuda, 3, 48, 64, 50.0, N_importance=128, ndc=ndc,
                                   **({} if ndc else dict(near=0.5, far=4.0)))
        _, held_out = forward_facing_camera(48, 64, 50.0, yaw=-0.1, pitch=0.02)
        idx = torch.randint(0, 48 * 64, (1500,), device=cuda)
        S, Ni = tr.N_samples, tr.N_importance
        nd = (float(K[0][0]), 1.0) if ndc else None
        for pose in (poses[2], held_out, None):
            got = tr.render(idx, c2w=pose)
            p = tr.c2w if pose is None else pose.to(cuda)
            r = ops.raygen(tr.H, tr.W, tr.K, p, ray_idx=idx, n_samples=S, near=tr.near, far=tr.far, ndc=nd,
                           want_viewdirs=True)
            o, d, v, z_c = r["rays_o"], r["rays_d"], r["viewdirs"], r["z_vals"]
            raw_c = torch.empty(1500 * S, 4, device=cuda)
            launch_fwd(tr.coarse, tr._pk[tr.coarse], raw_c, rays=(o, d, v, z_c))
            comp_c = ops.composite(raw_c.view(1500, S, 4), z_c, d, white_bkgd=tr.white_bkgd)
            zs, z_f = ops.resample_merge(z_c, comp_c[3], Ni, det=True, seed=1)
            raw_f = torch.empty(1500 * (S + Ni), 4, device=cuda)
            launch_fwd(tr.fine, tr._pk[tr.fine], raw_f, rays=(o, d, v, z_f))
            rgb, disp, acc, _, depth = ops.composite(raw_f.view(1500, S + Ni, 4), z_f, d, white_bkgd=tr.white_bkgd)
            torch.cuda.synchronize()
            assert torch.equal(got["rgb_map"], rgb) and torch.equal(got["acc_map"], acc)
            assert torch.equal(got["depth_map"], depth) and torch.equal(got["rgb0"], comp_c[0])
        a, b = tr.render(idx, c2w=poses[1]), tr.render(idx, c2w=poses[2])
        assert not torch.equal(a["rgb_map"], b["rgb_map"])


# ---------------------------------------------------------------- 8. fitting a scene
def _sphere_image(H, W, K, c2w, radius=1.0):
    """a coloured sphere at the origin (colour 0.5 + 0.5 * normal) on white, rendered analytically"""
    ro, rd = orc.get_rays(H, W, K, c2w)
    ro, rd = ro.double(), rd.double()
    a = (rd * rd).sum(-1)
    b = (ro * rd).sum(-1)
    c = (ro * ro).sum(-1) - radius ** 2
    disc = b * b - a * c
    hit = disc > 0
    t = (-b - disc.clamp_min(0).sqrt()) / a
    nrm = (ro + t[..., None] * rd) / radius
    col = torch.where(hit[..., None], 0.5 + 0.5 * nrm, torch.ones_like(nrm))
    return col.clamp(0, 1).float()


def _psnr(tr, img, pose):
    rgb = tr.render(c2w=pose)["rgb_map"].reshape(img.shape).cpu()
    return -10.0 * torch.log10(((rgb - img) ** 2).mean()).item()


def test_step_random_fits_a_small_scene(cuda):
    """A coloured sphere at 32 x 32 from 5 orbit poses, 4 for training (azimuths 0, 90, 180, 270) and 1 held out
    (azimuth 45); 400 step_random steps of 512 rays (upstream's Blender recipe: one image per step, 50 steps of a
    24 x 24 centre crop first).

    Measured on a B200: training views 7.74 -> 28.13 dB, held-out view 7.85 -> 15.77 dB (four views are few: the
    held-out view gains far less than the training views).  The bars (+10 dB and +4 dB) leave a wide margin."""
    from ctxnerf.train import NerfTrainer
    H = W = 32
    cams = [orbit_camera(H, W, focal=40.0, azim_deg=a) for a in (0.0, 90.0, 180.0, 270.0, 45.0)]
    K = cams[0][0]
    poses = torch.stack([c for _, c in cams])
    images = torch.stack([_sphere_image(H, W, K, c) for _, c in cams])
    torch.manual_seed(1)
    tr = NerfTrainer(H, W, K, poses[:4], images=images[:4], N_samples=64, N_importance=64, precrop_iters=50,
                     precrop_frac=0.75, device=cuda, seed=1)

    def psnrs():
        train = sum(_psnr(tr, images[v], poses[v]) for v in range(4)) / 4
        return train, _psnr(tr, images[4], poses[4])

    t0, h0 = psnrs()
    for _ in range(400):
        tr.step_random(512)
    torch.cuda.synchronize()
    t1, h1 = psnrs()
    _diag(f"fitting: training views {t0:.2f} -> {t1:.2f} dB, held-out view {h0:.2f} -> {h1:.2f} dB")
    assert t1 > t0 + 10.0 and h1 > h0 + 4.0
