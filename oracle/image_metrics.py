"""fp64 NumPy restatement of the evaluation metrics of ``ctx_image_metrics`` (csrc/metrics.cu).
TEST INFRASTRUCTURE ONLY (imported by tests/ only).

* MSE and PSNR: upstream's ``img2mse`` / ``mse2psnr`` (src/run_nerf_helpers.py:9-10), the squared difference of the
  fp32 images summed in fp64.
* SSIM: the ``compute_ssim`` of Google's mip-NeRF / MultiNeRF code with ``max_val = 1``, written out in the
  repository (DESIGN.md §4) because the reference has no SSIM: an 11-tap Gaussian window (sigma 1.5) applied
  separably, along x and then along y, in valid mode, to x, y, x^2, y^2 and xy of each channel.  Parity is unpinned:
  this file restates a third-party definition, and tests/test_evaluate_args.py checks it against a second derivation
  (scipy's 2-D convolution with the outer-product window).
"""
from __future__ import annotations

import numpy as np

C1, C2 = 0.01 * 0.01, 0.03 * 0.03


def gaussian_taps(size=11, sigma=1.5):
    """g_i = exp(-0.5 ((i - size//2) / sigma)^2), normalised to sum 1"""
    i = np.arange(size, dtype=np.float64)
    g = np.exp(-0.5 * ((i - size // 2) / sigma) ** 2)
    return g / g.sum()


def _filter_valid(img, g):
    """img [..., H, W] -> [..., H-10, W-10]: along x, then along y"""
    n = g.size
    H, W = img.shape[-2:]
    h = sum(g[k] * img[..., :, k:W - n + 1 + k] for k in range(n))
    return sum(g[k] * h[..., k:H - n + 1 + k, :] for k in range(n))


def as_unit_float(target):
    """a uint8 target as u8 / 255 in fp32 (IEEE division, as the kernel reads it), or the fp32 target itself"""
    t = np.asarray(target)
    if t.dtype == np.uint8:
        return (t.astype(np.float32) / np.float32(255.0)).astype(np.float32)
    return t.astype(np.float32)


def mse(pred, target):
    """[..., H, W, 3] -> [...]: mean of (pred - target)^2, the difference in fp32, squares and sums in fp64"""
    d = (np.asarray(pred, dtype=np.float32) - as_unit_float(target)).astype(np.float64)
    return (d * d).mean(axis=(-3, -2, -1))


def psnr(m):
    with np.errstate(divide="ignore"):
        return -10.0 * np.log10(np.asarray(m, dtype=np.float64))


def ssim_map(pred, target):
    """[..., H, W, 3] -> [..., 3, H-10, W-10]: the SSIM map of each channel"""
    x = np.moveaxis(np.asarray(pred, dtype=np.float32).astype(np.float64), -1, -3)
    y = np.moveaxis(as_unit_float(target).astype(np.float64), -1, -3)
    g = gaussian_taps()
    mu_x, mu_y = _filter_valid(x, g), _filter_valid(y, g)
    s_xx = np.maximum(0.0, _filter_valid(x * x, g) - mu_x ** 2)
    s_yy = np.maximum(0.0, _filter_valid(y * y, g) - mu_y ** 2)
    s_xy = _filter_valid(x * y, g) - mu_x * mu_y
    s_xy = np.sign(s_xy) * np.minimum(np.sqrt(s_xx * s_yy), np.abs(s_xy))
    return ((2 * mu_x * mu_y + C1) * (2 * s_xy + C2)) / ((mu_x ** 2 + mu_y ** 2 + C1) * (s_xx + s_yy + C2))


def ssim(pred, target):
    """[..., H, W, 3] -> [...]: the mean of the SSIM map over the three channels and the valid positions"""
    return ssim_map(pred, target).mean(axis=(-3, -2, -1))


def image_metrics(pred, target):
    """(mse, psnr, ssim) of one image [H, W, 3] or a batch [B, H, W, 3], fp64"""
    m = mse(pred, target)
    return m, psnr(m), ssim(pred, target)
