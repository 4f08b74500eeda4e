"""Test-split evaluation on the GPU: ctx_image_metrics (ops.image_metrics) against the fp64 oracle and its bit-level
properties, and NerfTrainer.evaluate against render(c2w=) + the oracle, leaving training undisturbed, tracking a fit,
and under two ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from ctxnerf.workloads import forward_facing_camera, orbit_camera
from oracle import image_metrics as om
from oracle import nerf_oracle as orc

pytestmark = pytest.mark.gpu


def _diag(msg):
    print(msg)        # measured figures: shown with pytest -s


def _images(kind, B, H, W, seed):
    """(pred fp32, target fp32) host pairs: independent noise, or smooth images and a noisy copy"""
    g = torch.Generator().manual_seed(seed)
    if kind == "random":
        return torch.rand(B, H, W, 3, generator=g), torch.rand(B, H, W, 3, generator=g)
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    ph = torch.rand(B, 1, 1, 3, generator=g, dtype=torch.float64) * 6.0
    base = 0.5 + 0.4 * torch.sin(xx[None, ..., None] / 9.0 + ph) * torch.cos(yy[None, ..., None] / 13.0 + 2 * ph)
    noisy = base + 0.03 * torch.randn(B, H, W, 3, generator=g, dtype=torch.float64)
    return base.float(), noisy.clamp(0, 1).float()


# ---------------------------------------------------------------- 1. the kernel against the oracle
WORST = {"mse_rel": 0.0, "ssim_abs": 0.0}


@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("kind", ["random", "smooth"])
@pytest.mark.parametrize("H,W,B", [(11, 11, 8), (37, 53, 5), (37, 53, 1), (378, 504, 3), (800, 800, 2)])
def test_metrics_against_the_oracle(cuda, H, W, B, kind, u8):
    from ctxnerf import ops
    pred, tgt = _images(kind, B, H, W, seed=H + W + B + 2 * u8)
    if u8:
        tgt = (tgt * 255.0).round().to(torch.uint8)
    mse, psnr, ssim = ops.image_metrics(pred.to(cuda), tgt.to(cuda))
    assert mse.dtype == psnr.dtype == ssim.dtype == torch.float64 and mse.shape == (B,)
    m_ref, p_ref, s_ref = om.image_metrics(pred.numpy(), tgt.numpy())
    mse, psnr, ssim = mse.cpu().numpy(), psnr.cpu().numpy(), ssim.cpu().numpy()
    mse_rel = float(np.max(np.abs(mse - m_ref) / m_ref))
    ssim_abs = float(np.max(np.abs(ssim - s_ref)))
    WORST["mse_rel"], WORST["ssim_abs"] = max(WORST["mse_rel"], mse_rel), max(WORST["ssim_abs"], ssim_abs)
    _diag(f"{H}x{W} B={B} {kind} {'u8' if u8 else 'fp32'}: mse rel err {mse_rel:.2e}, ssim abs err {ssim_abs:.2e}; "
          f"worst so far {WORST}")
    assert mse_rel <= 1e-10
    assert ssim_abs <= 1e-5
    assert np.allclose(psnr, p_ref, rtol=1e-10, atol=0)


def test_identical_images_and_a_single_image(cuda):
    from ctxnerf import ops
    x = torch.rand(40, 60, 3, generator=torch.Generator().manual_seed(0)).to(cuda)
    mse, psnr, ssim = ops.image_metrics(x, x)                  # [H,W,3]: a batch of one
    assert mse.shape == (1,) and mse.item() == 0.0 and psnr.item() == float("inf")
    assert abs(ssim.item() - 1.0) <= 1e-12
    a, b = torch.full((1, 20, 25, 3), 0.25, device=cuda), torch.full((1, 20, 25, 3), 0.75, device=cuda)
    mse, _, ssim = ops.image_metrics(a, b)
    assert mse.item() == 0.25
    assert abs(ssim.item() - (2 * 0.25 * 0.75 + om.C1) / (0.25 ** 2 + 0.75 ** 2 + om.C1)) <= 1e-12


# ---------------------------------------------------------------- 2. bit-level properties
def test_metrics_bit_properties(cuda):
    from ctxnerf import ops
    B, H, W = 5, 123, 201
    g = torch.Generator().manual_seed(11)
    pred = torch.rand(B, H, W, 3, generator=g).to(cuda)
    u8 = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, generator=g)
    f32 = torch.from_numpy(om.as_unit_float(u8.numpy())).to(cuda)       # u8 / 255 in fp32, IEEE division
    u8 = u8.to(cuda)
    a, b, c = ops.image_metrics(pred, u8), ops.image_metrics(pred, f32), ops.image_metrics(pred, u8)
    for x, y, z in zip(a, b, c):
        assert torch.equal(x, y), "a uint8 target and its fp32 u8 / 255 copy differ"
        assert torch.equal(x, z), "two calls differ"
    for i in range(B):                                                    # alone == inside the batch of 5
        alone = ops.image_metrics(pred[i], u8[i])
        for x, y in zip(alone, a):
            assert torch.equal(x, y[i:i + 1]), i


# ---------------------------------------------------------------- 3. evaluate == render + the oracle
@pytest.mark.parametrize("ndc", [False, True])
def test_evaluate_equals_render_and_the_oracle(cuda, ndc):
    from ctxnerf import ops
    from ctxnerf.train import NerfTrainer
    if ndc:
        H, W = 48, 64
        K, c2w = forward_facing_camera(H, W, 50.0)
        test = [forward_facing_camera(H, W, 50.0, yaw=0.1 - 0.07 * v, eye=(0.02 * v, -0.03, 0.1))[1] for v in range(3)]
        kw = dict(near=0.0, far=1.0, ndc=True, white_bkgd=False)
    else:
        H, W = 56, 40
        K, c2w = orbit_camera(H, W, focal=60.0)
        test = [orbit_camera(H, W, focal=60.0, azim_deg=25.0 + 100.0 * v)[1] for v in range(3)]
        kw = dict(near=2.0, far=6.0, white_bkgd=True)
    torch.manual_seed(2)
    tr = NerfTrainer(H, W, K, c2w, N_samples=32, N_importance=64, device=cuda, seed=4, **kw)
    poses = torch.stack(test)
    g = torch.Generator().manual_seed(7)
    for images in (torch.rand(3, H, W, 3, generator=g), torch.randint(0, 256, (3, H, W, 3), dtype=torch.uint8,
                                                                       generator=g)):
        for where in ("cpu", cuda):
            res = tr.evaluate(poses, images.to(where))
            assert all(v.device.type == "cpu" and v.dtype == torch.float64 and v.shape == (3,) for v in res.values())
            for v in range(3):
                rgb = tr.render(c2w=poses[v])["rgb_map"].reshape(H, W, 3)
                m, p, s = om.image_metrics(rgb.cpu().numpy(), images[v].numpy())
                assert abs(res["mse"][v].item() - m) <= 1e-10 * m
                assert abs(res["psnr"][v].item() - p) <= 1e-9
                assert abs(res["ssim"][v].item() - s) <= 1e-5
                got = ops.image_metrics(rgb, images[v].to(cuda))            # evaluate is exactly these two calls
                assert [res[k][v].item() for k in ("mse", "psnr", "ssim")] == [t.item() for t in got]
    _diag(f"evaluate (ndc={ndc}): psnr {res['psnr'].tolist()}, ssim {res['ssim'].tolist()}")


# ---------------------------------------------------------------- 4. training is undisturbed
def test_evaluate_does_not_disturb_training(cuda):
    from ctxnerf.train import NerfTrainer
    H = W = 32
    cams = [orbit_camera(H, W, focal=40.0, azim_deg=a) for a in (0.0, 120.0, 240.0)]
    poses = torch.stack([c for _, c in cams])
    images = torch.rand(3, H, W, 3, generator=torch.Generator().manual_seed(1))
    test_poses = torch.stack([orbit_camera(H, W, focal=40.0, azim_deg=a)[1] for a in (60.0, 180.0)])
    test_images = torch.randint(0, 256, (2, H, W, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(2))
    runs = []
    for with_eval in (True, False):
        torch.manual_seed(6)
        tr = NerfTrainer(H, W, cams[0][0], poses, images=images, N_samples=32, N_importance=32, precrop_iters=2,
                         device=cuda, seed=5)
        losses = [tr.step_random(256).item() for _ in range(3)]
        if with_eval:
            pl = tr._plans[(256, "draw")]
            assert pl.graph is not None
            torch.cuda.synchronize()
            before = dict(ctr=tr._ctr.clone(), loss=tr._loss.clone(), m=tr.exp_avg.clone(), v=tr.exp_avg_sq.clone(),
                          flat=tr.bucket.flat.clone(), rng=torch.random.get_rng_state(),
                          cuda_rng=torch.cuda.get_rng_state(cuda), graph=pl.graph, plans=dict(tr._plans),
                          pk={n: [t.clone() for t in tr._pk[n]] for n in (tr.coarse, tr.fine)})
            res = tr.evaluate(test_poses, test_images)
            torch.cuda.synchronize()
            assert torch.isfinite(res["psnr"]).all()
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


# ---------------------------------------------------------------- 5. a fit shows in the held-out metrics
def _sphere_image(H, W, K, c2w, radius=1.0):
    """a coloured sphere at the origin (colour 0.5 + 0.5 * normal) on white, rendered analytically (the scene of
    test_gpu_multiview.py)"""
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


def test_evaluate_tracks_a_fit(cuda):
    """The small sphere scene of test_gpu_multiview.py: 4 orbit views for training, the view at azimuth 45 held out;
    400 step_random steps of 512 rays.  The held-out view's PSNR and SSIM from evaluate both rise.

    Measured on a B200: held-out view 7.85 -> 15.77 dB, SSIM 0.101 -> 0.251; training views 7.74 -> 28.13 dB, SSIM
    0.082 -> 0.920 (the PSNRs equal the host computation of test_gpu_multiview.py's fitting test)."""
    from ctxnerf.train import NerfTrainer
    H = W = 32
    cams = [orbit_camera(H, W, focal=40.0, azim_deg=a) for a in (0.0, 90.0, 180.0, 270.0, 45.0)]
    K = cams[0][0]
    poses = torch.stack([c for _, c in cams])
    images = torch.stack([_sphere_image(H, W, K, c) for _, c in cams])
    torch.manual_seed(1)
    tr = NerfTrainer(H, W, K, poses[:4], images=images[:4], N_samples=64, N_importance=64, precrop_iters=50,
                     precrop_frac=0.75, device=cuda, seed=1)
    r0 = tr.evaluate(poses[4:], images[4:])
    t0 = tr.evaluate(poses[:4], images[:4])
    for _ in range(400):
        tr.step_random(512)
    r1 = tr.evaluate(poses[4:], images[4:])
    t1 = tr.evaluate(poses[:4], images[:4])
    _diag(f"fitting: held-out view psnr {r0['psnr'].item():.2f} -> {r1['psnr'].item():.2f} dB, ssim "
          f"{r0['ssim'].item():.4f} -> {r1['ssim'].item():.4f}; training views psnr {t0['psnr'].mean().item():.2f} -> "
          f"{t1['psnr'].mean().item():.2f} dB, ssim {t0['ssim'].mean().item():.4f} -> {t1['ssim'].mean().item():.4f}")
    assert r1["psnr"].item() > r0["psnr"].item() + 4.0
    assert r1["ssim"].item() > r0["ssim"].item()
    assert t1["psnr"].mean().item() > t0["psnr"].mean().item() + 10.0 and t1["ssim"].mean() > t0["ssim"].mean()


# ---------------------------------------------------------------- 6. two ranks
def test_evaluate_over_two_ranks_equals_one_process(cuda, tmp_path):
    """tools/eval_dist_check.py under 2 ranks: both ranks return the same vectors, bit for bit equal to the
    single-process evaluate of the same scene.  Needs >= 2 GPUs (skipped on a single-GPU box)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    tool = os.path.join(ROOT, "tools", "eval_dist_check.py")
    port = 29900 + (os.getpid() % 300)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), tool, str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    _diag("eval_dist_check (2 ranks):\n" + r.stdout[-1500:])
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stdout.count("identical on all ranks: True") == 2
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        from eval_dist_check import scene
    finally:
        sys.path.pop(0)
    tr, poses, images = scene(cuda)
    res = tr.evaluate(poses, images)
    single = torch.stack([res["mse"], res["psnr"], res["ssim"]]).numpy()
    for rank in (0, 1):
        got = np.load(os.path.join(tmp_path, f"rank{rank}.npy"))
        assert got.tobytes() == single.tobytes(), rank
