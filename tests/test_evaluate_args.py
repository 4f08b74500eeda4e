"""Test-split evaluation without a GPU: the fp64 metric oracle (oracle/image_metrics.py) against a second derivation
and known answers, and the argument checks of ctx_image_metrics, ops.image_metrics and NerfTrainer.evaluate, which
reject bad input before any launch or device work."""
import ctypes

import numpy as np
import pytest

from oracle import image_metrics as om

K = [[30.0, 0.0, 16.0], [0.0, 30.0, 16.0], [0.0, 0.0, 1.0]]
C2W = [[1.0, 0.0, 0.0, 0.0], [0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0]]


def _ssim_map_2d(x, y):
    """the SSIM map by scipy's 2-D convolution with the outer-product window, valid mode (the window is symmetric,
    so convolution and correlation agree)"""
    from scipy.signal import convolve2d
    g = om.gaussian_taps()
    win = np.outer(g, g)
    f = lambda a: convolve2d(a, win, mode="valid")
    maps = []
    for c in range(3):
        a, b = x[..., c].astype(np.float64), y[..., c].astype(np.float64)
        mu_a, mu_b = f(a), f(b)
        s_aa = np.maximum(0.0, f(a * a) - mu_a ** 2)
        s_bb = np.maximum(0.0, f(b * b) - mu_b ** 2)
        s_ab = f(a * b) - mu_a * mu_b
        s_ab = np.sign(s_ab) * np.minimum(np.sqrt(s_aa * s_bb), np.abs(s_ab))
        maps.append(((2 * mu_a * mu_b + om.C1) * (2 * s_ab + om.C2)) /
                    ((mu_a ** 2 + mu_b ** 2 + om.C1) * (s_aa + s_bb + om.C2)))
    return np.stack(maps)


@pytest.mark.parametrize("shape", [(11, 11), (23, 17), (40, 64)])
def test_separable_oracle_equals_the_2d_convolution(shape):
    rng = np.random.default_rng(sum(shape))
    H, W = shape
    yy, xx = np.mgrid[0:H, 0:W]
    smooth = 0.5 + 0.4 * np.sin(xx[..., None] / 5.0 + np.arange(3)) * np.cos(yy[..., None] / 7.0)
    for x, y in ((rng.random((H, W, 3)), rng.random((H, W, 3))),
                 (smooth, smooth + 0.05 * rng.standard_normal((H, W, 3)))):
        x, y = x.astype(np.float32), y.astype(np.float32)
        got = om.ssim_map(x, y)
        want = _ssim_map_2d(x, y)
        assert got.shape == (3, H - 10, W - 10)
        assert np.abs(got - want).max() <= 1e-12
        assert abs(om.ssim(x, y) - want.mean()) <= 1e-12


def test_oracle_known_answers():
    rng = np.random.default_rng(0)
    x = rng.random((2, 30, 40, 3)).astype(np.float32)
    m, p, s = om.image_metrics(x, x)
    assert np.all(m == 0.0) and np.all(np.isinf(p)) and np.allclose(s, 1.0, rtol=0, atol=1e-12)
    for a, b in ((0.25, 0.75), (0.875, 0.125), (0.5, 0.5), (0.0, 1.0)):     # fp32 differences are exact here
        xa, xb = np.full((20, 25, 3), a, np.float32), np.full((20, 25, 3), b, np.float32)
        m, p, s = om.image_metrics(xa, xb)
        assert abs(m - (a - b) ** 2) <= 1e-15
        assert abs(s - (2 * a * b + om.C1) / (a ** 2 + b ** 2 + om.C1)) <= 1e-12
    u8 = rng.integers(0, 256, (12, 13, 3), dtype=np.uint8)
    f = (u8.astype(np.float32) / np.float32(255.0)).astype(np.float32)      # a uint8 target reads as u8 / 255
    assert om.mse(x[0, :12, :13], u8) == om.mse(x[0, :12, :13], f)
    assert om.ssim(x[0, :12, :13], u8) == om.ssim(x[0, :12, :13], f)


def test_image_metrics_rejects_bad_arguments(libpath):
    from ctxnerf import _lib
    lib = _lib.lib()
    buf = ctypes.c_void_p(16)            # never dereferenced: every call below fails its checks first

    def metrics(pred=buf, target=buf, u8=0, B=2, H=16, W=16, mse=buf, ssim=buf, partials=buf):
        return lib.ctx_image_metrics(pred, target, u8, B, H, W, mse, ssim, partials, None)

    assert metrics(B=-1) == -1
    assert metrics(H=0) == -1 and metrics(W=0) == -1
    assert metrics(H=8, W=8) == -1                            # SSIM asked for, no valid window position
    assert metrics(H=10, W=64) == -1 and metrics(H=64, W=10) == -1
    assert metrics(u8=2) == -1
    assert metrics(pred=None) == -1 and metrics(target=None) == -1 and metrics(partials=None) == -1
    assert metrics(B=0) == 0                                  # nothing to do
    assert metrics(B=0, pred=None, target=None, partials=None) == 0
    assert lib.ctx_image_metrics_partials(2, 800, 800) == 2 * 2 * 25 * 25
    assert lib.ctx_image_metrics_partials(1, 11, 33) == 2 * 1 * 2
    assert lib.ctx_image_metrics_partials(0, 8, 8) == 0
    assert lib.ctx_image_metrics_partials(-1, 8, 8) == -1 and lib.ctx_image_metrics_partials(1, 0, 8) == -1


def test_image_metrics_op_needs_cuda_tensors():
    import torch
    from ctxnerf import ops
    from ctxnerf._lib import CtxNerfError
    with pytest.raises(CtxNerfError):
        ops.image_metrics(torch.zeros(2, 16, 16, 3), torch.zeros(2, 16, 16, 3))


def _bare_trainer(H=16, W=16):
    """evaluate checks its arguments before any device work: a bare instance that owns no device state at all"""
    from ctxnerf.train import NerfTrainer
    tr = object.__new__(NerfTrainer)
    tr.H, tr.W = H, W
    return tr


def test_evaluate_rejects_bad_input():
    import torch
    from ctxnerf._lib import CtxNerfError
    tr = _bare_trainer()
    poses = torch.tensor(C2W)[None].repeat(3, 1, 1)
    for images in (torch.zeros(3, 16, 17, 3), torch.zeros(3, 17, 16, 3), torch.zeros(3, 16, 16, 4),
                   torch.zeros(16, 16, 3)):
        with pytest.raises(CtxNerfError, match="images must be"):          # wrong image shape
            tr.evaluate(poses, images)
    for n in (2, 4):
        with pytest.raises(CtxNerfError, match="images must be"):          # pose / image count mismatch
            tr.evaluate(poses, torch.zeros(n, 16, 16, 3))
    for dt in (torch.float64, torch.float16, torch.int32, torch.bool):
        with pytest.raises(CtxNerfError, match="fp32 or uint8"):
            tr.evaluate(poses, torch.zeros(3, 16, 16, 3, dtype=dt))
    for bad in (torch.tensor(C2W), torch.zeros(3, 3, 3), torch.zeros(3, 2, 4)):
        with pytest.raises(CtxNerfError, match="c2w"):
            tr.evaluate(bad, torch.zeros(3, 16, 16, 3))


def test_evaluate_of_no_view_is_empty():
    import torch
    res = _bare_trainer().evaluate(torch.zeros(0, 3, 4), torch.zeros(0, 16, 16, 3, dtype=torch.uint8))
    assert set(res) == {"mse", "psnr", "ssim"}
    for v in res.values():
        assert v.shape == (0,) and v.dtype == torch.float64 and v.device.type == "cpu"
