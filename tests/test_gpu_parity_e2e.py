"""End-to-end and glue-kernel parity (VERDICT r1, "Next round" item 1).

* render_rays coarse 64 + fine 128 on the cfg-3 shapes against the fp32 oracle at the north-star tolerance
  (2e-2 in bf16-MLP mode) with a PRINCIPLED exclusion: raw2outputs is discontinuous in exactly one place -- the last
  sample's distance is 1e10, so its alpha jumps 0 -> 1 where sigma_last crosses 0 -- and a ray is excluded from the
  2e-2 bound only if the kernel's and the oracle's sigma_last lie on different sides of 0.  Every excluded ray must
  be explained: |sigma_last| of the oracle is within the measured bf16 error of the raw output, and its error is
  bounded by the transmittance that reaches the last sample.
* MLP backward against autograd through the fp32 reference forward (not only the bf16 emulation).
* ctx_adam_step against torch.optim.Adam, ctx_mse_fwd_bwd against img2mse + autograd.
* N-rank all-reduced gradients == single-process sum (SURVEY.md 8e), spawned here when >= 2 GPUs are visible.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import nerf_oracle as orc
from conftest import ROOT

pytestmark = pytest.mark.gpu


def _diag(msg):
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/diag.log", "a") as fh:
        fh.write(msg + "\n")
    print(msg)


def _nets(cuda, seed):
    from ctxnerf import run_nerf_helpers as rh
    torch.manual_seed(seed)
    nets = []
    for _ in range(2):
        n = rh.NeRF()
        with torch.no_grad():
            for p in n.parameters():
                if p.dim() == 1:
                    p.uniform_(-0.1, 0.1)
        nets.append((n.to(cuda), {k: v.detach().clone().cpu() for k, v in n.state_dict().items()}))
    return nets


def _cfg3_rays(R, seed):
    """R rays of the cfg-2/3 camera (800x800, f=1111.1, radius 4.03, near 2, far 6) as an upstream [R,11] batch."""
    K, c2w = orc.lego_like_camera()
    _, rd = orc.get_rays(800, 800, K, c2w)
    idx = torch.randint(0, 800 * 800, (R,), generator=torch.Generator().manual_seed(seed))
    d = rd.reshape(-1, 3)[idx]
    o = c2w[:3, -1].expand(R, 3)
    vd = d / d.norm(dim=-1, keepdim=True)
    return torch.cat([o, d, torch.full((R, 1), 2.0), torch.full((R, 1), 6.0), vd], -1).contiguous()


@pytest.mark.parametrize("perturb", [0.0, 1.0])
def test_render_rays_end_to_end_against_fp32_oracle(cuda, perturb):
    from ctxnerf import ops, run_nerf_helpers as rh
    R, S, Ni, far = 4096, 64, 128, 6.0
    TOL = 2e-2                                         # north_star: bf16-MLP mode
    (coarse, pc), (fine, pf) = _nets(cuda, seed=11)
    rays = _cfg3_rays(R, seed=5)
    ro, rd_, vdir = rays[:, 0:3], rays[:, 3:6], rays[:, 8:11]
    jitter = u = None
    if perturb > 0:                                    # the numbers render_rays(pytest=True) draws (upstream hook)
        np.random.seed(0)
        jitter = torch.Tensor(np.random.rand(R, S))
        np.random.seed(0)
        u = torch.Tensor(np.random.rand(R, Ni))
    q32 = lambda pts, vd, prm: orc.run_network(pts, vd, prm)
    with torch.no_grad():
        out = rh.render_rays(rays.to(cuda), coarse, rh.FusedQuery(), S, N_importance=Ni, network_fine=fine,
                             perturb=perturb, white_bkgd=True, retraw=True, pytest=perturb > 0)
        ref = orc.render_rays(rays, pc, q32, S, N_importance=Ni, network_fine=pf, perturb=perturb, white_bkgd=True,
                              jitter=jitter, u=u, retraw=True)
        # ---- stage 1, coarse pass: the depths are bit-identical by construction (stratified_z is bit-exact) ----
        o, d, vd = ro.to(cuda), rd_.to(cuda), vdir.to(cuda)
        z_c = orc.stratified_z(rays[:, 6:7], rays[:, 7:8], S, jitter=jitter)
        raw_c = coarse.forward_rays(o, d, vd, z_c.to(cuda))
        comp_c = [t.cpu() for t in rh.raw2outputs(raw_c, z_c.to(cuda), d, white_bkgd=True)]
        raw_c_ref = orc.run_network(ro[:, None] + rd_[:, None] * z_c[..., None], vdir, pc)
        ref_c = orc.raw2outputs(raw_c_ref, z_c, rd_, white_bkgd=True)
        # ---- stage 2, hierarchical sampling on the PRODUCT's coarse weights: bit-exact against the oracle ----
        zs_g, zall_g = ops.resample_merge(z_c.to(cuda), comp_c[3].to(cuda), Ni, det=(perturb == 0.0),
                                          u=u.to(cuda) if u is not None else None)
        zs_g, zall_g = zs_g.cpu(), zall_g.cpu()
        z_mid = 0.5 * (z_c[..., 1:] + z_c[..., :-1])
        zs_o = orc.sample_pdf(z_mid, comp_c[3][..., 1:-1], Ni, det=(perturb == 0.0), u=u)
        zall_o = torch.sort(torch.cat([z_c, zs_o], -1), -1)[0]
        # ---- stage 3, fine pass on the product's own merged depths ----
        raw_f_ref = orc.run_network(ro[:, None] + rd_[:, None] * zall_g[..., None], vdir, pf)
        ref_f = orc.raw2outputs(raw_f_ref, zall_g, rd_, white_bkgd=True)
        raw_f = out["raw"].cpu()
        comp_f = [t.cpu() for t in rh.raw2outputs(out["raw"], zall_g.to(cuda), d, white_bkgd=True)]
    raw_c = raw_c.cpu()
    n_bad = int((zs_g != zs_o).sum())
    _diag(f"render_rays perturb={perturb}: importance samples on the product's coarse weights: {n_bad} of {zs_o.numel()} "
          f"differ from the oracle's; merged depths equal: {torch.equal(zall_g, zall_o)}")
    assert n_bad == 0 and torch.equal(zall_g, zall_o)          # north_star: sample positions bit-exact

    def explained_flips(tag, raw_gpu, raw_ref, weights_ref):
        """rays whose last-sample alpha sits on the other side of the 0 -> 1 jump, each one explained"""
        s_gpu, s_ref = raw_gpu[:, -1, 3], raw_ref[:, -1, 3]
        flip = (s_gpu > 0) != (s_ref > 0)
        tau = (raw_gpu[..., 3] - raw_ref[..., 3]).abs().max().item()        # measured bf16 error of sigma
        scale = raw_ref[..., 3].abs().max().item()
        e_rgbraw = (raw_gpu[..., :3] - raw_ref[..., :3]).abs().max().item() / raw_ref[..., :3].abs().max().item()
        _diag(f"render_rays perturb={perturb} {tag}: raw sigma err max {tau:.3e} (scale {scale:.3f}, rel {tau / scale:.3e}), "
              f"raw rgb rel err {e_rgbraw:.3e}; {int(flip.sum())}/{R} rays flip alpha_last")
        assert tau <= TOL * scale and e_rgbraw <= TOL
        assert (s_ref[flip].abs() <= tau).all(), "a flipped ray is not within the bf16 error of the discontinuity"
        assert flip.float().mean().item() < 0.03
        # what a flip can add or remove: the transmittance that reaches the last sample
        t_last = 1.0 - weights_ref[:, :-1].sum(-1)
        return flip, torch.maximum(t_last, weights_ref[:, -1]).clamp_min(0.0)

    def check(tag, got, want, flip, t_last):
        rgb, disp, acc, w, depth = got
        rgb_r, disp_r, acc_r, w_r, depth_r = want
        errs = {"rgb": (rgb - rgb_r).abs().amax(-1), "acc": (acc - acc_r).abs(),
                "depth": (depth - depth_r).abs() / far, "weights": (w - w_r).abs().amax(-1)}
        keep = ~flip
        for name, e in errs.items():
            _diag(f"render_rays perturb={perturb} {tag} {name}: max err {e[keep].max().item():.3e} on {int(keep.sum())} rays"
                  f" (excluded {int(flip.sum())}: max {e[flip].max().item() if flip.any() else 0.0:.3e})")
            assert e[keep].max().item() <= TOL, (tag, name)
            if flip.any():      # excluded rays: off by at most the weight the flipped last sample carries
                assert (e[flip] <= t_last[flip] + TOL).all(), (tag, name)
        # disp is NaN exactly when acc == 0 (0/0): the NaN sets may differ only on rays that are empty to within TOL
        nan_diff = keep & (torch.isnan(disp) != torch.isnan(disp_r))
        assert (torch.maximum(acc, acc_r)[nan_diff] <= TOL).all()
        # disp = acc/depth, a ratio of two quantities each within TOL: first-order bound TOL*(far/depth + 1/acc),
        # checked where the ray is solid enough for the ratio to be conditioned
        solid = keep & ~torch.isnan(disp_r) & ~torch.isnan(disp) & (acc_r > 0.5)
        if solid.any():
            ed = (disp - disp_r).abs() / disp_r.abs().clamp_min(1e-6)
            bound = 1.5 * TOL * (far / depth_r.clamp_min(1e-3) + 1.0 / acc_r.clamp_min(1e-3))
            _diag(f"render_rays perturb={perturb} {tag} disp: max rel err {ed[solid].max().item():.3e} on {int(solid.sum())} rays")
            assert (ed[solid] <= bound[solid]).all()

    flip_c, t_c = explained_flips("coarse", raw_c, raw_c_ref, ref_c[3])
    check("coarse", comp_c, ref_c, flip_c, t_c)
    flip_f, t_f = explained_flips("fine (product's depths)", raw_f, raw_f_ref, ref_f[3])
    check("fine (product's depths)", comp_f, ref_f, flip_f, t_f)
    # render_rays returned exactly what the stages produce
    assert torch.equal(out["rgb0"].cpu(), comp_c[0]) and torch.equal(out["acc0"].cpu(), comp_c[2])
    assert torch.equal(out["rgb_map"].cpu(), comp_f[0]) and torch.equal(out["acc_map"].cpu(), comp_f[2])
    torch.testing.assert_close(out["z_std"].cpu(), torch.std(zs_g, dim=-1, unbiased=False), rtol=1e-4, atol=1e-6)

    # ---- end to end against the oracle's own chain (its coarse weights -> its importance samples) ----
    # The fine pass of the product runs on depths placed by ITS coarse weights.  sample_pdf divides by
    # sum(w) + 1e-5*B, so on rays whose coarse weights are small (every ray of a random-init network) a 1e-3 error in
    # one weight moves whole groups of samples: a property of the reference function, present between the fp32 oracle
    # and ANY bf16 evaluation of the coarse network.  It is measured on the oracle alone -- Q = |oracle fine pass on
    # the product's depths - oracle fine pass on its own depths|, fp32 on both sides -- and the end-to-end bound is
    # TOL + Q per ray; rays whose samples did not move (Q ~ 0) therefore meet TOL itself.
    keep = ~flip_f
    for name, got, a_ref, b_ref in (("rgb", out["rgb_map"].cpu(), ref["rgb_map"], ref_f[0]),
                                    ("acc", out["acc_map"].cpu(), ref["acc_map"], ref_f[2]),
                                    ("depth", comp_f[4] / far, ref["depth_map"] / far, ref_f[4] / far)):
        red = (lambda t: t.amax(-1)) if got.dim() > 1 else (lambda t: t)
        e = red((got - a_ref).abs())
        Q = red((b_ref - a_ref).abs())
        still = keep & (Q <= 1e-3)
        _diag(f"render_rays perturb={perturb} end-to-end {name}: max err {e[keep].max().item():.3e} (p99 "
              f"{e[keep].quantile(0.99).item():.3e}); oracle's own sensitivity to the sample shift Q max {Q[keep].max().item():.3e}; "
              f"{int(still.sum())} rays with Q <= 1e-3: max err {e[still].max().item() if still.any() else 0.0:.3e}")
        assert (e[keep] <= TOL + Q[keep]).all(), name
        assert (e[flip_f] <= t_f[flip_f] + TOL + Q[flip_f]).all(), name


@pytest.mark.parametrize("views,in_pts,out_ch,P", [(False, 42, 3, 4096), (True, 63, 4, 4096)])
def test_mlp_backward_against_fp32_autograd(cuda, views, in_pts, out_ch, P):
    """dgrad + wgrad kernels vs autograd through the fp32 REFERENCE forward (NeRF2D.forward semantics, no bf16
    emulation).  The loss is coherent (MSE to a target + a small penalty), the kind of loss the path trains with;
    the bound is the north star's 2e-2 on the whole gradient (L2) -- per-tensor figures are logged."""
    from ctxnerf import run_nerf_helpers as rh
    torch.manual_seed(50 + P + in_pts)
    net = (rh.NeRF(input_ch=in_pts, input_ch_views=27) if views else rh.NeRF2D(input_ch=in_pts, output_ch=out_ch))
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 1:
                p.uniform_(-0.1, 0.1)
    params = {k: v.detach().clone() for k, v in net.state_dict().items()}
    net = net.to(cuda)
    g = torch.Generator().manual_seed(3)
    v = 27 if views else 0
    x = torch.rand(P, in_pts + v, generator=g) * 2 - 1
    tgt = torch.rand(P, out_ch, generator=g)
    pr = {k: t.clone().requires_grad_(True) for k, t in params.items()}
    o32 = orc.mlp_forward(pr, x, input_ch_views=v)
    ((torch.sigmoid(o32) - tgt).pow(2).mean() + 1e-2 * o32.pow(2).mean()).backward()
    out = net(x.to(cuda))
    ((torch.sigmoid(out) - tgt.to(cuda)).pow(2).mean() + 1e-2 * out.pow(2).mean()).backward()
    got = torch.cat([p.grad.reshape(-1).cpu() for _, p in net.named_parameters()])
    ref = torch.cat([pr[n].grad.reshape(-1) for n, _ in net.named_parameters()])
    l2 = ((got - ref).norm() / ref.norm()).item()
    cos = torch.nn.functional.cosine_similarity(got, ref, dim=0).item()
    worst = max(((p.grad.cpu() - pr[n].grad).norm() / (pr[n].grad.norm() + 1e-20)).item()
                for n, p in net.named_parameters())
    _diag(f"mlp bwd vs fp32 autograd views={views} in={in_pts}: whole-gradient l2 {l2:.3e}, cosine {cos:.6f}, "
          f"worst tensor l2 {worst:.3e}")
    assert l2 < 2e-2 and cos > 0.9995


def test_adam_kernel_matches_torch_adam(cuda):
    """ctx_adam_step (csrc/optim.cu) vs torch.optim.Adam (the reference's optimiser, trainer.py:603) over 3 steps,
    with the 1/world gradient scale and a weight decay."""
    from ctxnerf._lib import call, ptr, stream_ptr
    n = 100003
    g = torch.Generator().manual_seed(0)
    p0 = torch.randn(n, generator=g)
    grads = [torch.randn(n, generator=g) * (10.0 ** (i - 2)) for i in range(3)]
    for wd, scale in ((0.0, 1.0), (1e-2, 0.25)):
        ref = torch.nn.Parameter(p0.clone().to(cuda))
        opt = torch.optim.Adam([ref], lr=5e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=wd)
        p = p0.clone().to(cuda)
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        for step, gr in enumerate(grads, 1):
            ref.grad = (gr * scale).to(cuda)
            opt.step()
            gd = gr.to(cuda)
            call("ctx_adam_step", ptr(p), ptr(gd), ptr(m), ptr(v), n, 5e-4, 0.9, 0.999, 1e-8, step, wd, scale,
                 stream_ptr(cuda))
            torch.cuda.synchronize()
            st = opt.state[ref]
            # (torch computes lerp / addcmul, the kernel b*m + (1-b)*g: a few ulps apart, measured 1.3e-5 relative)
            # (where b*m and (1-b)*g cancel the relative difference of the sum is unbounded: absolute floor of 1e-7 of
            #  the gradient scale)
            gs = float(gr.abs().max()) * scale
            torch.testing.assert_close(m, st["exp_avg"], rtol=5e-5, atol=1e-7 * gs)
            torch.testing.assert_close(v, st["exp_avg_sq"], rtol=5e-5, atol=1e-7 * gs * gs)
            # parameters: both subtract an update that agrees to ~1e-5 relative (<= 5e-9 absolute); what is left is
            # the rounding of the result, i.e. a couple of ulps of the parameter
            torch.testing.assert_close(p, ref.detach(), rtol=3e-7, atol=2e-8)


def test_mse_kernel_matches_img2mse_autograd(cuda):
    """ctx_mse_fwd_bwd: loss = img2mse(a,t) + img2mse(b,t) (reference :9) and both gradients in one pass."""
    from ctxnerf._lib import call, ptr, stream_ptr
    from ctxnerf import run_nerf_helpers as rh
    g = torch.Generator().manual_seed(1)
    for R in (4096, 37, 1):
        a = torch.rand(R, 3, generator=g).to(cuda).requires_grad_(True)
        b = torch.rand(R, 3, generator=g).to(cuda).requires_grad_(True)
        t = torch.rand(R, 3, generator=g).to(cuda)
        (rh.img2mse(a, t) + rh.img2mse(b, t)).backward()
        loss = torch.zeros(1, device=cuda)
        ga, gb = torch.empty(R, 3, device=cuda), torch.empty(R, 3, device=cuda)
        call("ctx_mse_fwd_bwd", ptr(a.detach()), ptr(b.detach()), ptr(t), R * 3, 1.0, ptr(loss), ptr(ga), ptr(gb),
             stream_ptr(cuda))
        torch.cuda.synchronize()
        want = (rh.img2mse(a, t) + rh.img2mse(b, t)).item()
        assert abs(loss.item() - want) <= 1e-6 * max(1.0, abs(want))
        torch.testing.assert_close(ga, a.grad, rtol=1e-6, atol=1e-9)
        torch.testing.assert_close(gb, b.grad, rtol=1e-6, atol=1e-9)
        # single-image form
        call("ctx_mse_fwd_bwd", ptr(a.detach()), None, ptr(t), R * 3, 1.0, ptr(loss), ptr(ga), None, stream_ptr(cuda))
        torch.cuda.synchronize()
        assert abs(loss.item() - rh.img2mse(a, t).item()) <= 1e-6


def test_render_rays_driver_equals_the_kernel_sequence(cuda):
    """ctx_render_rays (csrc/render.cu, the C-ABI driver behind NerfTrainer.render) enqueues the same six launches a
    host would issue one by one: every intermediate and every map must be bit-identical to that sequence -- for the
    deterministic render and for the jittered one (same Philox seeds)."""
    from ctxnerf import ops
    from ctxnerf.mlp import launch_fwd
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera
    K, c2w = orbit_camera()
    tr = NerfTrainer(800, 800, K, c2w, device=cuda, seed=3)
    idx = torch.randint(0, 640000, (1500,), device=cuda)
    S, Ni = tr.N_samples, tr.N_importance
    for perturb, seed in ((False, 0), (True, 1234)):
        got = tr._render(idx, perturb=perturb, seed=seed)
        r = ops.raygen(tr.H, tr.W, tr.K, tr.c2w, ray_idx=idx, n_samples=S, near=tr.near, far=tr.far,
                       lindisp=tr.lindisp, perturb=perturb, seed=seed, want_viewdirs=True)
        o, d, v, z_c = r["rays_o"], r["rays_d"], r["viewdirs"], r["z_vals"]
        R = o.shape[0]
        raw_c = torch.empty(R * S, 4, device=cuda)
        launch_fwd(tr.coarse, tr._pk[tr.coarse], raw_c, rays=(o, d, v, z_c))
        comp_c = ops.composite(raw_c.view(R, S, 4), z_c, d, white_bkgd=tr.white_bkgd)
        zs, z_f = ops.resample_merge(z_c, comp_c[3], Ni, det=not perturb, seed=seed + 1)
        raw_f = torch.empty(R * (S + Ni), 4, device=cuda)
        launch_fwd(tr.fine, tr._pk[tr.fine], raw_f, rays=(o, d, v, z_f))
        comp_f = ops.composite(raw_f.view(R, S + Ni, 4), z_f, d, white_bkgd=tr.white_bkgd)
        torch.cuda.synchronize()
        assert torch.equal(got["z_f"], z_f) and torch.equal(got["raw_f"], raw_f)
        for a, b in zip(got["comp_c"] + got["comp_f"], comp_c + comp_f):
            assert torch.equal(a, b) or (torch.isnan(a) == torch.isnan(b)).all() and torch.equal(
                torch.nan_to_num(a), torch.nan_to_num(b))
    # single-pass form (n_importance = 0) with the bounding-sphere interval: NerfTrainer.render_view (BASELINE config 4)
    from ctxnerf.workloads import multiview_cameras
    cams, sph = multiview_cameras()
    Kv, cv = cams[1]
    idx4 = torch.randint(0, 1024 * 1024, (3000,), device=cuda)
    got = tr.render_view(1024, 1024, Kv, cv, n_samples=192, sphere=sph, ray_idx=idx4)
    r = ops.raygen(1024, 1024, Kv, torch.as_tensor(cv, dtype=torch.float32).to(cuda), n_samples=192, near=tr.near,
                   far=tr.far, sphere=sph, want_viewdirs=True, ray_idx=idx4)
    raw = torch.empty(3000 * 192, 4, device=cuda)
    launch_fwd(tr.fine, tr._pk[tr.fine], raw, rays=(r["rays_o"], r["rays_d"], r["viewdirs"], r["z_vals"]))
    rgb, disp, acc, _, depth = ops.composite(raw.view(3000, 192, 4), r["z_vals"], r["rays_d"], white_bkgd=tr.white_bkgd)
    torch.cuda.synchronize()
    assert torch.equal(got["rgb_map"], rgb) and torch.equal(got["acc_map"], acc) and torch.equal(got["depth_map"], depth)
    assert torch.equal(torch.nan_to_num(got["disp_map"]), torch.nan_to_num(disp))
    # argument errors come back as codes, not crashes
    from ctxnerf import _lib
    assert _lib.lib().ctx_render_rays(None, None) == -1
    bad = _lib.CtxRenderArgs()
    bad.n_rays, bad.n_samples = 4, 64
    assert _lib.lib().ctx_render_rays(ctypes.byref(bad), None) == -1


def test_allreduced_gradients_of_two_ranks_equal_single_process_sum(cuda):
    """SURVEY.md 8e correctness contract: the gradient bucket after the one all-reduce of N ranks (each its own
    4096-ray batch) == the sum of the per-batch gradients computed by one process.  Needs >= 2 GPUs (skipped on a
    single-GPU box); tools/dist_check.py is the body, its N = 2 / 8 outputs are kept under profiles/."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    # both routes of the all-reduce: the library's NCCL binding (ctx_allreduce, a node of the step graph) and
    # torch.distributed between two graphs (CTXNERF_NCCL=0)
    for k, (nccl, route) in enumerate((("1", "ctx_allreduce (NCCL"), ("0", "torch.distributed"))):
        port = 29600 + (os.getpid() % 300) + k
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", str(port),
                            os.path.join(ROOT, "tools", "dist_check.py")], capture_output=True, text=True, timeout=900,
                           env=dict(os.environ, CTXNERF_NCCL=nccl))
        _diag(f"dist_check (2 ranks, CTXNERF_NCCL={nccl}):\n" + r.stdout[-1500:])
        assert r.returncode == 0, r.stderr[-3000:]
        assert r.stdout.count("all-reduced vs single-process sum") == 2
        assert r.stdout.count(route) == 2
        assert r.stdout.count("identical on all ranks: True") == 2


def test_drop_in_mlp_survives_nn_dataparallel(cuda):
    """The reference wraps the texture MLP in nn.DataParallel whenever more than one GPU is visible
    (/root/reference/src/training/trainer.py:129-135) -- i.e. always on the 8-GPU target.  Build the model exactly as
    it does, run forward + backward through the wrapper (scatter of the [N,42] embedding, per-device replicas of the
    parameters, gather, reduce-add of the gradients) and compare with the unwrapped module on one GPU; the fused
    get_texture_map must accept the wrapper too.  Needs >= 2 GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    from ctxnerf import run_nerf_helpers as rh
    from ctxnerf.texture import get_texture_map
    device = torch.device("cuda", 0)
    embed_fn, embedder_out_dim = rh.get_embedder(multires=10)                     # trainer.py:129
    torch.manual_seed(3)
    texture_mlp = rh.NeRF2D(D=8, W=256, input_ch=embedder_out_dim, output_ch=3, skips=[4]).to(device)   # :133
    single = rh.NeRF2D(D=8, W=256, input_ch=embedder_out_dim, output_ch=3, skips=[4]).to(device)
    single.load_state_dict(texture_mlp.state_dict())
    wrapped = torch.nn.DataParallel(texture_mlp)                                  # :134-135
    g = torch.Generator().manual_seed(0)
    uv = torch.rand(20000, 2, generator=g).to(device)
    tgt = torch.rand(20000, 3, generator=g).to(device)
    for step in range(2):       # twice: the replicas are re-broadcast every call (no stale packed weights)
        out_w = wrapped(embed_fn(uv))
        out_s = single(embed_fn(uv))
        assert out_w.shape == out_s.shape == (20000, 3)
        torch.testing.assert_close(out_w, out_s, rtol=0, atol=1e-6)
        for m in (texture_mlp, single):
            m.zero_grad(set_to_none=True)
        ((torch.tanh(out_w) + 1) / 2 - tgt).pow(2).mean().backward()
        ((torch.tanh(out_s) + 1) / 2 - tgt).pow(2).mean().backward()
        for (n, pw), (_, ps) in zip(texture_mlp.named_parameters(), single.named_parameters()):
            assert pw.grad is not None, n
            scale = ps.grad.abs().max().item() + 1e-20
            assert (pw.grad - ps.grad).abs().max().item() <= 2e-5 * scale, (n, step)   # fp32 atomics: order only
        with torch.no_grad():   # an optimizer step in place, as Adam does (trainer.py:603)
            for pw, ps in zip(texture_mlp.parameters(), single.parameters()):
                pw.add_(pw.grad, alpha=-1e-3)
                ps.add_(ps.grad, alpha=-1e-3)
    tex_w, _ = get_texture_map(wrapped, 64)
    tex_s, _ = get_texture_map(single, 64)
    torch.testing.assert_close(tex_w, tex_s, rtol=0, atol=1e-6)


def test_captured_step_equals_eager_step(cuda):
    """NerfTrainer.step replays ONE CUDA graph per batch size (device-side seed / Adam step counters, static buffers,
    SURVEY.md 8f row 3).  The first step of a batch size runs eagerly, the second is captured and replayed: after the
    same first step, the captured second step must produce the gradient bucket, loss and Adam moments of an eager
    second step (perturb = 0: no random numbers; fp32 atomics give order-level noise).  Parameters are compared in
    bulk only: Adam normalises every update to ~lr, so a parameter whose gradient is summation noise moves by +-lr
    whichever sign the noise has."""
    import os
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera
    H = W = 64
    K, c2w = orbit_camera(H, W, focal=80.0)
    idx = torch.arange(0, H * W, 3, device=cuda, dtype=torch.int64)[:1024]
    tgts = [torch.rand(idx.numel(), 3, generator=torch.Generator().manual_seed(s)).to(cuda) for s in range(4)]
    res = {}
    for mode in ("graph", "eager"):
        os.environ["CTXNERF_GRAPH"] = "1" if mode == "graph" else "0"
        try:
            tr = NerfTrainer(H, W, K, c2w, perturb=0.0, device=cuda, seed=3, lr=5e-4)
        finally:
            del os.environ["CTXNERF_GRAPH"]
        p0 = tr.bucket.flat.clone()
        l1 = tr.step(idx, tgts[0]).item()
        l2 = tr.step(idx, tgts[1]).item()
        torch.cuda.synchronize()
        plan = tr._plans[idx.numel()]
        assert (plan.graph is not None) == (mode == "graph")
        snap = (l1, l2, tr.bucket.grad.clone(), tr.exp_avg.clone(), tr.bucket.flat.clone())
        more = [tr.step(idx, t).item() for t in tgts[2:]]          # two more replays
        torch.cuda.synchronize()
        assert tr._ctr.tolist() == [8, 4]                  # seed offset += 2 and Adam step += 1 per step, on the device
        assert all(l == l for l in more) and torch.isfinite(tr.bucket.flat).all()
        res[mode] = snap + (p0,)
    (g1, g2, gg, gm, gp, p0), (e1, e2, eg, em, ep, _) = res["graph"], res["eager"]
    assert abs(g1 - e1) <= 1e-6 * abs(e1) and abs(g2 - e2) <= 1e-5 * abs(e2), (g1, e1, g2, e2)
    gscale = eg.abs().max().item()
    gerr = (gg - eg).abs().max().item() / gscale
    merr = (gm - em).abs().max().item() / em.abs().max().item()
    step_size = (ep - p0).abs().max().item()
    off = ((gp - ep).abs() > 0.05 * step_size).float().mean().item()
    _diag(f"captured vs eager second step: grad max rel diff {gerr:.3e}, exp_avg {merr:.3e}; {100 * off:.3f} % of the "
          f"parameters differ by more than 5 % of the update size ({step_size:.3e})")
    assert gerr < 1e-4 and merr < 1e-4
    assert off < 0.05


def test_jitter_changes_between_replays_and_is_reproducible(cuda):
    """perturb = 1: the stratified jitter and the importance uniforms come from Philox(seed0 + device counter), so two
    replays of the captured step draw different depths, and two trainers built under the same torch seed agree."""
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera
    H = W = 32
    K, c2w = orbit_camera(H, W, focal=40.0)
    idx = torch.arange(H * W, device=cuda)[:512]
    tgt = torch.rand(512, 3, device=cuda)
    runs = []
    for _ in range(2):
        torch.manual_seed(11)
        tr = NerfTrainer(H, W, K, c2w, perturb=1.0, device=cuda, seed=1)
        zs = []
        for _ in range(3):
            tr.step(idx, tgt)
            zs.append(tr._plans[512].z_c.clone())
        runs.append(zs)
    assert not torch.equal(runs[0][0], runs[0][1]) and not torch.equal(runs[0][1], runs[0][2])   # fresh numbers per step
    for a, b in zip(*runs):
        assert torch.equal(a, b)                                                             # reproducible
    z = runs[0][2]
    assert (z[:, 1:] >= z[:, :-1]).all() and z.min() >= 2.0 and z.max() <= 6.0


def test_inputs_that_ask_for_unsupported_gradients_raise(cuda):
    """The hand-written backward differentiates w.r.t. the parameters (MLP) / raw (raw2outputs) only: an input that
    requires a gradient it would silently not get raises instead (ADVICE r1); float64 / strided inputs are converted,
    never reinterpreted."""
    from ctxnerf import run_nerf_helpers as rh
    from ctxnerf._lib import CtxNerfError
    net = rh.NeRF2D(D=8, W=256, input_ch=42, output_ch=3, skips=[4]).to(cuda)
    x = torch.rand(64, 42, device=cuda, requires_grad=True)
    with pytest.raises(CtxNerfError):
        net(x)
    raw = torch.randn(8, 16, 4, device=cuda, requires_grad=True)
    z = torch.sort(torch.rand(8, 16, device=cuda) * 4 + 2, -1)[0]
    d = torch.randn(8, 3, device=cuda)
    with pytest.raises(CtxNerfError):
        rh.raw2outputs(raw, z.clone().requires_grad_(True), d)
    for p in net.parameters():                    # every parameter frozen: forward works, backward is a no-op
        p.requires_grad_(False)
    out = net(torch.rand(64, 42, device=cuda))
    assert not out.requires_grad
    # float64 ray batch (numpy-built rays, as upstream tolerates): converted
    nerf = rh.NeRF().to(cuda)
    rays64 = torch.cat([torch.zeros(16, 3), torch.randn(16, 3), torch.full((16, 1), 2.0), torch.full((16, 1), 6.0),
                        torch.nn.functional.normalize(torch.randn(16, 3), dim=-1)], -1).double().to(cuda)
    with torch.no_grad():
        a = rh.render_rays(rays64, nerf, rh.FusedQuery(), 64, N_importance=32, network_fine=nerf)
        b = rh.render_rays(rays64.float(), nerf, rh.FusedQuery(), 64, N_importance=32, network_fine=nerf)
    assert torch.equal(a["rgb_map"], b["rgb_map"])
