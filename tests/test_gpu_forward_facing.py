"""Forward-facing training (upstream nerf-pytorch's LLFF recipe) in NerfTrainer: NDC rays, density noise drawn inside
the fused compositing kernels, learning-rate decay on the device, and the NDC form of the render driver."""
import ctypes
import os

import pytest
import torch

from ctxnerf.workloads import forward_facing_camera
from oracle import nerf_oracle as orc

pytestmark = pytest.mark.gpu


def _diag(msg):
    print(msg)        # measured figures: shown with pytest -s


def _density_noise(cuda, R, S, std, seed, seed_dev, stream_id):
    from ctxnerf._lib import call, ptr, stream_ptr
    out = torch.empty(R, S, device=cuda)
    call("ctx_density_noise", ptr(out), R, S, std, seed, ptr(seed_dev), stream_id, stream_ptr(cuda))
    return out


def _comp_train(cuda, raw, z, d, target, white, weights=True, noise=None, rng=None):
    """ctx_composite_train with a noise tensor (rng None) or ctx_composite_train_noise (rng = (std, seed, seed_dev,
    stream)) -> (loss, g_raw, weights, rgb_map)"""
    from ctxnerf._lib import call, ptr, stream_ptr
    R, S = z.shape
    loss = torch.zeros(1, device=cuda)
    g_raw = torch.full((R * S, 4), float("nan"), device=cuda)
    w = torch.full((R, S), float("nan"), device=cuda) if weights else None
    rgb = torch.full((R, 3), float("nan"), device=cuda)
    if rng is None:
        call("ctx_composite_train", ptr(raw), ptr(z), ptr(d), ptr(noise), R, S, int(white), ptr(target),
             1.0 / (3.0 * R), ptr(loss), ptr(g_raw), ptr(w), ptr(rgb), stream_ptr(cuda))
    else:
        std, seed, seed_dev, stream_id = rng
        call("ctx_composite_train_noise", ptr(raw), ptr(z), ptr(d), R, S, int(white), ptr(target), 1.0 / (3.0 * R),
             ptr(loss), ptr(g_raw), ptr(w), ptr(rgb), std, seed, ptr(seed_dev), stream_id, stream_ptr(cuda))
    return loss, g_raw, w, rgb


@pytest.mark.parametrize("S", [32, 64, 77, 96, 128, 192, 256, 384, 512, 1024])
def test_noise_kernel_equals_the_tensor_path(cuda, S):
    """ctx_composite_train_noise == ctx_composite_train fed the ctx_density_noise tensor, bit for bit, for every
    single-pass instantiation (S <= 512) and the chunked path (1024); R is not a multiple of the rays per warp."""
    g = torch.Generator().manual_seed(S)
    R = 1003
    raw = torch.randn(R * S, 4, generator=g).to(cuda)
    z = torch.sort(torch.rand(R, S, generator=g) * 4 + 2, -1)[0].to(cuda)
    d = torch.randn(R, 3, generator=g).to(cuda)
    tgt = torch.rand(R, 3, generator=g).to(cuda)
    ctr = torch.tensor([6, 3], dtype=torch.int64, device=cuda)
    seed = 0x123456789AB
    for white in (False, True):
        for std, stream_id in ((1.0, 2), (0.3, 3)):
            noise = _density_noise(cuda, R, S, std, seed, ctr, stream_id)
            want = _comp_train(cuda, raw, z, d, tgt, white, noise=noise)
            got = _comp_train(cuda, raw, z, d, tgt, white, rng=(std, seed, ctr, stream_id))
            clean = _comp_train(cuda, raw, z, d, tgt, white)
            torch.cuda.synchronize()
            for name, a, b in zip(("loss", "g_raw", "weights", "rgb_map"), got, want):
                assert torch.equal(a, b), (S, white, std, name)
            assert not torch.equal(got[1], clean[1])       # the noise does reach the gradients
    # without weights (the fine pass) and with noise_std == 0 (the launches of ctx_composite_train)
    noise = _density_noise(cuda, R, S, 1.0, seed, None, 2)
    want = _comp_train(cuda, raw, z, d, tgt, False, weights=False, noise=noise)
    got = _comp_train(cuda, raw, z, d, tgt, False, weights=False, rng=(1.0, seed, None, 2))
    zero = _comp_train(cuda, raw, z, d, tgt, False, rng=(0.0, seed, ctr, 2))
    clean = _comp_train(cuda, raw, z, d, tgt, False)
    torch.cuda.synchronize()
    for a, b in zip(got, want):
        assert a is None and b is None or torch.equal(a, b)
    for a, b in zip(zero, clean):
        assert torch.equal(a, b)


def test_density_noise_statistics(cuda):
    R, S, std, seed = 4096, 192, 0.7, 987654321
    ctr = torch.tensor([10, 5], dtype=torch.int64, device=cuda)
    n2 = _density_noise(cuda, R, S, std, seed, ctr, 2).double()
    n3 = _density_noise(cuda, R, S, std, seed, ctr, 3).double()
    ctr_next = ctr.clone()
    ctr_next[0] += 1
    n2b = _density_noise(cuda, R, S, std, seed, ctr_next, 2).double()
    again = _density_noise(cuda, R, S, std, seed, ctr, 2).double()
    N = R * S
    mean, sd = n2.mean().item(), n2.std().item()

    def corr(a, b):
        a, b = a.reshape(-1) - a.mean(), b.reshape(-1) - b.mean()
        return ((a * b).sum() / (a.norm() * b.norm())).item()

    c23, cnext, clag = corr(n2, n3), corr(n2, n2b), corr(n2[:, 1:], n2[:, :-1])
    _diag(f"density noise {R}x{S} std {std}: mean {mean:.3e} (bound {5 * std / N ** 0.5:.3e}), std {sd:.6f}, "
          f"corr streams 2/3 {c23:.2e}, successive seed_dev {cnext:.2e}, neighbouring samples {clag:.2e}")
    assert torch.isfinite(n2).all() and torch.isfinite(n3).all()
    assert abs(mean) < 5 * std / N ** 0.5
    assert abs(sd - std) < 0.01 * std
    assert abs(c23) < 0.01 and abs(cnext) < 0.01 and abs(clag) < 0.01
    assert torch.equal(n2, again)
    # the four moments of a normal, loosely: fourth standardised moment 3
    k4 = (((n2 - mean) / sd) ** 4).mean().item()
    assert abs(k4 - 3.0) < 0.06, k4


def _trainer(cuda, H=32, W=32, focal=30.0, **kw):
    from ctxnerf.train import NerfTrainer
    K, c2w = forward_facing_camera(H, W, focal)
    args = dict(near=0.0, far=1.0, N_samples=64, N_importance=64, perturb=0.0, white_bkgd=False, ndc=True,
                device=cuda, seed=3)
    args.update(kw)
    return NerfTrainer(H, W, K, c2w, **args), K, c2w


def _oracle_rays(tr, K, c2w, idx):
    """get_rays -> view directions -> ndc_rays(H, W, K[0][0], 1.) as upstream render() does, for the pixels idx"""
    ro, rd = orc.get_rays(tr.H, tr.W, K, c2w)
    ro, rd = ro.reshape(-1, 3)[idx].contiguous(), rd.reshape(-1, 3)[idx].contiguous()
    vd = rd / torch.norm(rd, dim=-1, keepdim=True)
    o, d = orc.ndc_rays(tr.H, tr.W, K[0][0], 1.0, ro, rd)
    return o, d, vd


def _compare_step(tr, loss, ref_loss, prc, prf, what):
    _diag(f"{what}: loss {loss:.6f} vs oracle {ref_loss:.6f}")
    assert abs(loss - ref_loss) < 2e-2 * abs(ref_loss)
    for tag, net, pr in (("coarse", tr.coarse, prc), ("fine", tr.fine, prf)):
        got = torch.cat([p.grad.reshape(-1).cpu() for _, p in net.named_parameters()])
        ref = torch.cat([pr[name].grad.reshape(-1) for name, _ in net.named_parameters()])
        l2 = (got - ref).norm().item() / ref.norm().item()
        cos = torch.nn.functional.cosine_similarity(got, ref, dim=0).item()
        _diag(f"{what} {tag}: whole-gradient l2-rel err {l2:.3e}, cosine {cos:.6f}")
        assert l2 < 2e-2 and cos > 0.999, (tag, l2, cos)


def _params(net):
    return {k: v.detach().cpu().clone().requires_grad_(True) for k, v in net.state_dict().items()}


def test_ndc_step_against_the_oracle(cuda):
    """NerfTrainer(ndc=True) step gradients vs autograd through the oracle chain with bf16 operands (the bars of
    test_mlp_backward_fused_rays_training_step)."""
    tr, K, c2w = _trainer(cuda)
    # A density the coarse pass resolves (sigma ~ 2 instead of a random-init network's +-0.3, half of it cut by the
    # relu): sample_pdf divides by sum(w) + 1e-5 (B - 2), so on near-empty rays a bf16-sized change of one coarse weight
    # moves whole groups of fine samples -- a property of the reference function, present between the oracle and any
    # bf16 evaluation (test_render_rays_end_to_end_against_fp32_oracle measures it), not of the NDC path.
    with torch.no_grad():
        for net in (tr.coarse, tr.fine):
            net.alpha_linear.bias.fill_(2.0)
        tr._repack()
    R, S, Ni = 256, tr.N_samples, tr.N_importance
    idx = torch.randperm(tr.H * tr.W, generator=torch.Generator().manual_seed(1))[:R]
    tgt = torch.rand(R, 3, generator=torch.Generator().manual_seed(2))
    prc, prf = _params(tr.coarse), _params(tr.fine)
    loss = tr.step(idx.to(cuda), tgt.to(cuda), optimizer_step=False).item()
    o, d, vd = _oracle_rays(tr, K, c2w, idx)
    batch = torch.cat([o, d, torch.zeros(R, 1), torch.ones(R, 1), vd], -1)
    q = lambda pts, v, prm: orc.run_network(pts, v, prm, bf16_operands=True)
    ref = orc.render_rays(batch, prc, q, S, N_importance=Ni, network_fine=prf, white_bkgd=False)
    ref_loss = orc.img2mse(ref["rgb_map"], tgt) + orc.img2mse(ref["rgb0"], tgt)
    ref_loss.backward()
    # the step's rays are upstream's NDC rays, its view directions the metric ones
    pl = tr._plans[R]
    for name, a, b in (("rays_o", pl.o, o), ("rays_d", pl.d, d), ("viewdirs", pl.v, vd)):
        e = (a.cpu() - b).abs().max().item()
        _diag(f"ndc step {name}: max |step - oracle| {e:.3e}")
        assert e <= 1e-5 * max(1.0, b.abs().max().item()), name
    _compare_step(tr, loss, ref_loss.item(), prc, prf, "ndc step")


def test_noisy_step_against_the_oracle(cuda):
    """raw_noise_std = 1: the oracle's raw2outputs(noise=...) gets the coarse / fine noise ctx_density_noise makes
    from the step's key (seed0 + counter) on streams 2 and 3."""
    torch.manual_seed(21)
    tr, K, c2w = _trainer(cuda, raw_noise_std=1.0)
    R, S, Ni = 256, tr.N_samples, tr.N_importance
    idx = torch.randperm(tr.H * tr.W, generator=torch.Generator().manual_seed(3))[:R]
    tgt = torch.rand(R, 3, generator=torch.Generator().manual_seed(4))
    prc, prf = _params(tr.coarse), _params(tr.fine)
    loss = tr.step(idx.to(cuda), tgt.to(cuda), optimizer_step=False).item()
    assert tr._seed0 != 0 and tr._ctr.tolist() == [2, 1]
    nc = _density_noise(cuda, R, S, 1.0, tr._seed0, tr._ctr, 2).cpu()
    nf = _density_noise(cuda, R, S + Ni, 1.0, tr._seed0, tr._ctr, 3).cpu()
    o, d, vd = _oracle_rays(tr, K, c2w, idx)
    q = lambda pts, prm: orc.run_network(pts, vd, prm, bf16_operands=True)
    z = orc.stratified_z(torch.zeros(R, 1), torch.ones(R, 1), S)
    rgb0, _, _, w, _ = orc.raw2outputs(q(o[:, None] + d[:, None] * z[..., None], prc), z, d, noise=nc)
    z_new = orc.sample_pdf(0.5 * (z[..., 1:] + z[..., :-1]), w[..., 1:-1], Ni, det=True).detach()
    zf, _ = torch.sort(torch.cat([z, z_new], -1), -1)
    rgb, _, _, _, _ = orc.raw2outputs(q(o[:, None] + d[:, None] * zf[..., None], prf), zf, d, noise=nf)
    ref_loss = orc.img2mse(rgb, tgt) + orc.img2mse(rgb0, tgt)
    ref_loss.backward()
    _compare_step(tr, loss, ref_loss.item(), prc, prf, "noisy ndc step")


def test_captured_step_equals_eager_step_with_every_option(cuda):
    """ndc + raw_noise_std + lrate_decay (+ jitter): the replayed graph computes what the eager sequence computes (the
    bars of test_captured_step_equals_eager_step)."""
    H = W = 64
    idx = torch.arange(0, H * W, 3, device=cuda, dtype=torch.int64)[:1024]
    tgts = [torch.rand(idx.numel(), 3, generator=torch.Generator().manual_seed(s)).to(cuda) for s in range(4)]
    res = {}
    for mode in ("graph", "eager"):
        os.environ["CTXNERF_GRAPH"] = "1" if mode == "graph" else "0"
        try:
            torch.manual_seed(7)
            tr, _, _ = _trainer(cuda, H, W, 60.0, N_importance=128, perturb=1.0, raw_noise_std=1.0, lrate_decay=250,
                                lr=5e-4)
        finally:
            del os.environ["CTXNERF_GRAPH"]
        p0 = tr.bucket.flat.clone()
        l1 = tr.step(idx, tgts[0]).item()
        l2 = tr.step(idx, tgts[1]).item()
        torch.cuda.synchronize()
        assert (tr._plans[idx.numel()].graph is not None) == (mode == "graph")
        snap = (l1, l2, tr.bucket.grad.clone(), tr.exp_avg.clone(), tr.bucket.flat.clone())
        more = [tr.step(idx, t).item() for t in tgts[2:]]
        torch.cuda.synchronize()
        assert tr._ctr.tolist() == [8, 4]
        assert all(l == l for l in more) and torch.isfinite(tr.bucket.flat).all()
        res[mode] = snap + (p0,)
    (g1, g2, gg, gm, gp, p0), (e1, e2, eg, em, ep, _) = res["graph"], res["eager"]
    assert abs(g1 - e1) <= 1e-6 * abs(e1) and abs(g2 - e2) <= 1e-5 * abs(e2), (g1, e1, g2, e2)
    gerr = (gg - eg).abs().max().item() / eg.abs().max().item()
    merr = (gm - em).abs().max().item() / em.abs().max().item()
    step_size = (ep - p0).abs().max().item()
    off = ((gp - ep).abs() > 0.05 * step_size).float().mean().item()
    _diag(f"captured vs eager second step (ndc + noise + decay): grad max rel diff {gerr:.3e}, exp_avg {merr:.3e}; "
          f"{100 * off:.3f} % of the parameters differ by more than 5 % of the update size")
    assert gerr < 1e-4 and merr < 1e-4
    assert off < 0.05


def test_noise_changes_between_replays_and_is_reproducible(cuda):
    """lr = 0 and perturb = 0: only the density noise moves rgb0 from step to step.  Every replay draws fresh noise,
    two trainers built under the same torch seed draw the same, and a replay's noise is the ctx_density_noise tensor
    of the step's key on stream 2."""
    runs = []
    for _ in range(2):
        torch.manual_seed(11)
        tr, _, _ = _trainer(cuda, raw_noise_std=1.0, lr=0.0)
        idx = torch.arange(tr.H * tr.W, device=cuda)[:512]
        tgt = torch.rand(512, 3, generator=torch.Generator().manual_seed(5)).to(cuda)
        rgb0 = []
        for _ in range(3):
            tr.step(idx, tgt)
            rgb0.append(tr._plans[512].rgb0.clone())
        runs.append(rgb0)
    assert tr._plans[512].graph is not None
    assert not torch.equal(runs[0][0], runs[0][1]) and not torch.equal(runs[0][1], runs[0][2])
    for a, b in zip(*runs):
        assert torch.equal(a, b)
    pl = tr._plans[512]
    noise = _density_noise(cuda, 512, tr.N_samples, 1.0, tr._seed0, tr._ctr, 2)
    _, _, _, rgb = _comp_train(cuda, pl.raw_c, pl.z_c, pl.d, pl.target, False, noise=noise)
    torch.cuda.synchronize()
    assert torch.equal(rgb, pl.rgb0)


def _torch_adam_upstream_loop(p0, grads, lrate, decay_steps, cuda):
    """torch.optim.Adam driven as upstream's training loop drives it: step, then lr from global_step, then count"""
    ref = torch.nn.Parameter(p0.clone().to(cuda))
    opt = torch.optim.Adam([ref], lr=lrate, betas=(0.9, 0.999), eps=1e-8)
    global_step = 0
    out = []
    for gr in grads:
        ref.grad = gr.to(cuda).clone()
        opt.step()
        new_lrate = lrate * (0.1 ** (global_step / decay_steps))
        for pg in opt.param_groups:
            pg["lr"] = new_lrate
        global_step += 1
        out.append((ref.detach().clone(), opt.state[ref]["exp_avg"].clone()))
    return out


def test_adam_learning_rate_decay(cuda):
    """ctx_adam_step_dev_decay over t = 1..6 == torch.optim.Adam under upstream's decay loop; then a trainer with
    lrate_decay applies that rate: its parameters after 4 steps equal a host replay of the gradients it used."""
    from ctxnerf._lib import call, ptr, stream_ptr
    n, lrate, decay_steps = 100003, 5e-4, 3.0
    g = torch.Generator().manual_seed(0)
    p0 = torch.randn(n, generator=g)
    grads = [torch.randn(n, generator=g) * (10.0 ** (i % 3 - 2)) for i in range(6)]
    want = _torch_adam_upstream_loop(p0, grads, lrate, decay_steps, cuda)
    p = p0.clone().to(cuda)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    ctr = torch.zeros(2, dtype=torch.int64, device=cuda)
    for t, (gr, (wp, wm)) in enumerate(zip(grads, want), 1):
        call("ctx_step_tick", ptr(ctr), None, stream_ptr(cuda))
        call("ctx_adam_step_dev_decay", ptr(p), ptr(gr.to(cuda)), ptr(m), ptr(v), n, lrate, 0.9, 0.999, 1e-8,
             ptr(ctr), 0.0, 1.0, decay_steps, stream_ptr(cuda))
        torch.cuda.synchronize()
        # (atol: a few ulps of parameters near zero; the update itself is ~lr, see test_adam_kernel_matches_torch_adam)
        torch.testing.assert_close(p, wp, rtol=1e-6, atol=2e-8)
        torch.testing.assert_close(m, wm, rtol=5e-5, atol=1e-7 * float(gr.abs().max()))
    # a constant rate is far from the decayed one by t = 6: the comparison above would see it
    assert lrate * 0.1 ** (4 / decay_steps) < 0.1 * lrate

    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera
    H = W = 32
    K, c2w = orbit_camera(H, W, focal=40.0)
    tr = NerfTrainer(H, W, K, c2w, N_samples=32, N_importance=32, perturb=0.0, device=cuda, seed=1,
                     lrate_decay=0.002)                           # decay_steps = 2
    idx = torch.arange(H * W, device=cuda)[:512]
    p_start = tr.bucket.flat.detach().clone()
    used = []
    for s in range(4):
        tr.step(idx, torch.rand(512, 3, generator=torch.Generator().manual_seed(s)).to(cuda))
        used.append(tr.bucket.grad.clone())
    torch.cuda.synchronize()
    assert tr._plans[512].graph is not None
    replay = _torch_adam_upstream_loop(p_start, used, tr.lr, 2.0, cuda)
    torch.testing.assert_close(tr.bucket.flat, replay[-1][0], rtol=1e-6, atol=2e-8)


def test_ndc_render_equals_the_kernel_sequence(cuda):
    """NerfTrainer.render / render_view of an NDC trainer (ctx_render_rays_ndc) == the launches a host would issue, bit
    for bit; ctx_render_rays without NDC is unchanged; the metric sphere interval is refused."""
    from ctxnerf import _lib, ops
    from ctxnerf._lib import CtxNerfError
    from ctxnerf.mlp import launch_fwd
    tr, K, c2w = _trainer(cuda, 48, 64, 50.0, N_importance=128)
    flat, _, _ = _trainer(cuda, 48, 64, 50.0, N_importance=128, ndc=False, near=0.5, far=4.0)
    idx = torch.randint(0, 48 * 64, (1500,), device=cuda)
    S, Ni = tr.N_samples, tr.N_importance
    for t, nd in ((tr, (float(K[0][0]), 1.0)), (flat, None)):
        got = t.render(idx)
        r = ops.raygen(t.H, t.W, t.K, t.c2w, ray_idx=idx, n_samples=S, near=t.near, far=t.far, ndc=nd,
                       want_viewdirs=True)
        o, d, v, z_c = r["rays_o"], r["rays_d"], r["viewdirs"], r["z_vals"]
        raw_c = torch.empty(1500 * S, 4, device=cuda)
        launch_fwd(t.coarse, t._pk[t.coarse], raw_c, rays=(o, d, v, z_c))
        comp_c = ops.composite(raw_c.view(1500, S, 4), z_c, d, white_bkgd=t.white_bkgd)
        zs, z_f = ops.resample_merge(z_c, comp_c[3], Ni, det=True, seed=1)
        raw_f = torch.empty(1500 * (S + Ni), 4, device=cuda)
        launch_fwd(t.fine, t._pk[t.fine], raw_f, rays=(o, d, v, z_f))
        rgb, disp, acc, _, depth = ops.composite(raw_f.view(1500, S + Ni, 4), z_f, d, white_bkgd=t.white_bkgd)
        torch.cuda.synchronize()
        assert torch.equal(got["rgb_map"], rgb) and torch.equal(got["acc_map"], acc)
        assert torch.equal(got["depth_map"], depth) and torch.equal(got["rgb0"], comp_c[0])
        assert torch.equal(torch.nan_to_num(got["disp_map"]), torch.nan_to_num(disp))
        if nd is not None:        # NDC origins lie on the near plane, z = -1
            assert torch.allclose(o[:, 2], torch.full_like(o[:, 2], -1.0))
    # single pass (render_view): the view's own focal
    Kv, cv = forward_facing_camera(40, 40, 35.0)
    idx2 = torch.randint(0, 1600, (700,), device=cuda)
    got = tr.render_view(40, 40, Kv, cv, n_samples=96, near=0.0, far=1.0, ray_idx=idx2)
    r = ops.raygen(40, 40, Kv, cv.to(cuda), ray_idx=idx2, n_samples=96, near=0.0, far=1.0, ndc=(35.0, 1.0),
                   want_viewdirs=True)
    raw = torch.empty(700 * 96, 4, device=cuda)
    launch_fwd(tr.fine, tr._pk[tr.fine], raw, rays=(r["rays_o"], r["rays_d"], r["viewdirs"], r["z_vals"]))
    rgb, _, acc, _, _ = ops.composite(raw.view(700, 96, 4), r["z_vals"], r["rays_d"], white_bkgd=tr.white_bkgd)
    torch.cuda.synchronize()
    assert torch.equal(got["rgb_map"], rgb) and torch.equal(got["acc_map"], acc)
    with pytest.raises(CtxNerfError):
        tr.render_view(40, 40, Kv, cv, n_samples=96, sphere=(0.0, 0.0, -2.0, 1.0))
    bad = _lib.CtxRenderArgs()
    bad.n_rays, bad.n_samples = 4, 64
    assert _lib.lib().ctx_render_rays_ndc(ctypes.byref(bad), 35.0, 1.0, None) == -1
