"""torch.autograd.Function wrappers around the C-ABI launchers.

Every backward calls the hand-written ``*_bwd`` kernel; nothing here falls
back to autograd through eager ops, and nothing runs on the CPU: inputs must
be CUDA tensors (a CPU tensor raises).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import call, ptr, stream_ptr


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.CtxNerfError(
                "ctxnerf ops run on CUDA tensors only (no CPU fallback); got a tensor on "
                f"{t.device}")


def _f32c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def new_seed() -> int:
    """A 63-bit Philox seed drawn from torch's global generator (so that
    torch.manual_seed makes the in-kernel random numbers reproducible)."""
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


# ------------------------------------------------------------------ posenc ---
class _PosEnc(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, L, include_input, log_sampling):
        _need_cuda(x)
        shape = x.shape
        d = shape[-1]
        xf = _f32c(x).reshape(-1, d)
        n = xf.shape[0]
        C = d * ((1 if include_input else 0) + 2 * L)
        out = torch.empty(n, C, device=x.device, dtype=torch.float32)
        with torch.cuda.device(x.device):
            call("ctx_posenc_fwd", ptr(xf), ptr(out), n, d, L, int(include_input), int(log_sampling),
                 stream_ptr(x.device))
        ctx.save_for_backward(xf)
        ctx.meta = (shape, d, L, include_input, log_sampling)
        return out.reshape(*shape[:-1], C)

    @staticmethod
    def backward(ctx, g):
        (xf,) = ctx.saved_tensors
        shape, d, L, inc, logs = ctx.meta
        g = _f32c(g).reshape(xf.shape[0], -1)
        gx = torch.empty_like(xf)
        with torch.cuda.device(xf.device):
            call("ctx_posenc_bwd", ptr(xf), ptr(g), ptr(gx), xf.shape[0], d, L, int(inc), int(logs),
                 stream_ptr(xf.device))
        return gx.reshape(shape), None, None, None


def posenc(x: torch.Tensor, L: int, include_input: bool = True, log_sampling: bool = True) -> torch.Tensor:
    return _PosEnc.apply(x, int(L), bool(include_input), bool(log_sampling))


# --------------------------------------------------------------- composite ---
class _Composite(torch.autograd.Function):
    @staticmethod
    def forward(ctx, raw, z_vals, rays_d, noise, white_bkgd):
        _need_cuda(raw, z_vals, rays_d, noise)
        for name, t in (("z_vals", z_vals), ("rays_d", rays_d), ("noise", noise)):
            if t is not None and t.requires_grad:
                raise _lib.CtxNerfError(
                    f"raw2outputs: the hand-written backward differentiates with respect to raw only; {name} has "
                    "requires_grad=True and would silently get no gradient.  Detach it (DESIGN.md section 7)")
        raw_c, z_c, d_c, n_c = _f32c(raw), _f32c(z_vals), _f32c(rays_d), _f32c(noise)
        S = raw_c.shape[-2]
        lead = raw_c.shape[:-2]
        R = raw_c.numel() // (S * 4) if S > 0 else 0
        if raw_c.shape[-1] != 4:
            raise _lib.CtxNerfError("raw2outputs expects raw[..., S, 4]")
        dev = raw.device
        rgb = torch.empty(*lead, 3, device=dev, dtype=torch.float32)
        disp = torch.empty(*lead, device=dev, dtype=torch.float32)
        acc = torch.empty(*lead, device=dev, dtype=torch.float32)
        weights = torch.empty(*lead, S, device=dev, dtype=torch.float32)
        depth = torch.empty(*lead, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            call("ctx_composite_fwd", ptr(raw_c), ptr(z_c), ptr(d_c), ptr(n_c), R, S, int(white_bkgd),
                 ptr(rgb), ptr(disp), ptr(acc), ptr(weights), ptr(depth), stream_ptr(dev))
        ctx.save_for_backward(raw_c, z_c, d_c, n_c if n_c is not None else torch.empty(0, device=dev))
        ctx.meta = (R, S, bool(white_bkgd), n_c is not None, raw.shape)
        ctx.mark_non_differentiable()
        return rgb, disp, acc, weights, depth

    @staticmethod
    def backward(ctx, g_rgb, g_disp, g_acc, g_weights, g_depth):
        raw_c, z_c, d_c, n_c = ctx.saved_tensors
        R, S, white, has_noise, raw_shape = ctx.meta
        g_raw = torch.empty_like(raw_c)
        dev = raw_c.device
        # keep every (possibly converted) gradient tensor referenced until the launch is enqueued
        gs = [_f32c(g_rgb), _f32c(g_disp), _f32c(g_acc), _f32c(g_weights), _f32c(g_depth)]
        with torch.cuda.device(dev):
            call("ctx_composite_bwd", ptr(raw_c), ptr(z_c), ptr(d_c), ptr(n_c if has_noise else None),
                 R, S, int(white), ptr(gs[0]), ptr(gs[1]), ptr(gs[2]), ptr(gs[3]), ptr(gs[4]), ptr(g_raw),
                 stream_ptr(dev))
        return g_raw.reshape(raw_shape), None, None, None, None


def composite(raw, z_vals, rays_d, noise=None, white_bkgd=False):
    """-> (rgb_map, disp_map, acc_map, weights, depth_map).  Gradients flow to
    ``raw`` only (z_vals / rays_d are data in the render step)."""
    return _Composite.apply(raw, z_vals, rays_d, noise, bool(white_bkgd))


# ---------------------------------------------------------------- resample ---
class _Resample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, bins, weights, n_samples, det, u, seed, mid_bins):
        _need_cuda(bins, weights, u)
        dev = bins.device
        lead = weights.shape[:-1]
        nw = weights.shape[-1]
        B = nw + 1
        b2 = bins.reshape(-1, bins.shape[-1]).float()
        w2 = weights.reshape(-1, nw).float()
        if b2.stride(-1) != 1:
            b2 = b2.contiguous()
        if w2.stride(-1) != 1:
            w2 = w2.contiguous()
        R = w2.shape[0]
        u2 = _f32c(u.reshape(R, n_samples)) if u is not None else None
        out = torch.empty(R, n_samples, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            call("ctx_resample_fwd", ptr(b2), b2.stride(0) if R > 1 else b2.shape[-1], int(mid_bins), ptr(w2),
                 w2.stride(0) if R > 1 else nw, None, ptr(u2), int(det), seed, None, R, B, n_samples, ptr(out),
                 None, None, 0, 0, None, stream_ptr(dev))
        ctx.save_for_backward(b2, w2, u2 if u2 is not None else torch.empty(0, device=dev))
        ctx.meta = (R, B, n_samples, det, seed, mid_bins, u2 is not None, weights.shape)
        return out.reshape(*lead, n_samples)

    @staticmethod
    def backward(ctx, g):
        b2, w2, u2 = ctx.saved_tensors
        R, B, N, det, seed, mid_bins, has_u, wshape = ctx.meta
        dev = b2.device
        gw = torch.empty(R, B - 1, device=dev, dtype=torch.float32)
        g2 = _f32c(g).reshape(R, N)
        with torch.cuda.device(dev):
            call("ctx_resample_bwd", ptr(b2), b2.stride(0) if R > 1 else b2.shape[-1], int(mid_bins), ptr(w2),
                 w2.stride(0) if R > 1 else B - 1, ptr(u2 if has_u else None), int(det), seed, R, B, N,
                 ptr(g2), ptr(gw), stream_ptr(dev))
        return None, gw.reshape(wshape), None, None, None, None, None


def resample(bins, weights, n_samples, det=False, u=None, seed=None, mid_bins=False):
    if seed is None:
        seed = 0 if (det or u is not None) else new_seed()
    return _Resample.apply(bins, weights, int(n_samples), bool(det), u, int(seed), bool(mid_bins))


def resample_merge(z_vals, weights, n_importance, det=False, u=None, seed=None, cdf=None,
                   return_inds=False, seed_dev=None, out=None):
    """Fused hierarchical step of upstream render_rays (no grad, as upstream
    detaches): bins = mid-points of z_vals, pdf = weights[...,1:-1];
    returns (z_samples [R,Ni], z_all [R,S+Ni] sorted[, inds])."""
    _need_cuda(z_vals, weights, u, cdf)
    dev = z_vals.device
    z2 = _f32c(z_vals.detach()).reshape(-1, z_vals.shape[-1])
    w2 = _f32c(weights.detach()).reshape(-1, weights.shape[-1])
    R, S = z2.shape
    B = S - 1
    if seed is None:
        seed = 0 if (det or u is not None or seed_dev is not None) else new_seed()
    u2 = _f32c(u.reshape(R, n_importance)) if u is not None else None
    c2 = _f32c(cdf.reshape(R, B)) if cdf is not None else None
    if out is not None:          # caller-owned (static) outputs: the captured training step
        zs, z_all = out
    else:
        zs = torch.empty(R, n_importance, device=dev, dtype=torch.float32)
        z_all = torch.empty(R, S + n_importance, device=dev, dtype=torch.float32)
    inds = torch.empty(R, n_importance, device=dev, dtype=torch.int64) if return_inds else None
    w_view = w2[:, 1:-1]  # stride S, offset 1: no copy
    with torch.cuda.device(dev):
        call("ctx_resample_fwd", ptr(z2), S, 1, ptr(w_view), S, ptr(c2), ptr(u2), int(det), int(seed), ptr(seed_dev),
             R, B, n_importance, ptr(zs), ptr(inds), ptr(z2), S, S, ptr(z_all), stream_ptr(dev))
    if return_inds:
        return zs, z_all, inds
    return zs, z_all


def resample_raw(bins, weights, n_samples, det=True, u=None, cdf=None, seed=0):
    """Un-differentiated call that also returns the searchsorted indices (tests)."""
    _need_cuda(bins, weights, u, cdf)
    dev = bins.device
    b2 = _f32c(bins).reshape(-1, bins.shape[-1])
    R, B = b2.shape
    w2 = _f32c(weights).reshape(R, B - 1) if weights is not None else None
    u2 = _f32c(u.reshape(R, n_samples)) if u is not None else None
    c2 = _f32c(cdf.reshape(R, B)) if cdf is not None else None
    out = torch.empty(R, n_samples, device=dev, dtype=torch.float32)
    inds = torch.empty(R, n_samples, device=dev, dtype=torch.int64)
    with torch.cuda.device(dev):
        call("ctx_resample_fwd", ptr(b2), B, 0, ptr(w2), B - 1, ptr(c2), ptr(u2), int(det), int(seed), None, R, B,
             n_samples, ptr(out), ptr(inds), None, 0, 0, None, stream_ptr(dev))
    return out, inds


# ------------------------------------------------------------------ raygen ---
def raygen(H, W, K, c2w, *, device=None, ray_idx=None, ndc=None, n_samples=0, near=0.0, far=1.0,
           lindisp=False, perturb=False, jitter=None, seed=None, sphere=None, want_viewdirs=False,
           want_near_far=False, seed_dev=None, out=None):
    """Fused get_rays (+ndc) (+viewdirs) (+stratified z_vals).  Returns a dict.

    ``c2w`` is one pose [3|4, 4] (``ray_idx``: pixel ids y*W + x) or a stack [N, 3|4, 4] (``ctx_raygen_views``:
    ``ray_idx`` holds global ids view*H*W + y*W + x, None = all N*H*W rays in that order)."""
    if torch.is_tensor(c2w):
        dev = c2w.device if c2w.is_cuda else torch.device(device or "cuda")
        c2w_d = c2w.to(device=dev, dtype=torch.float32)
    else:
        dev = torch.device(device or "cuda")
        c2w_d = torch.as_tensor(c2w, dtype=torch.float32).to(dev)
    if device is not None:
        dev = torch.device(device)
        c2w_d = c2w_d.to(dev)
    c2w_d = c2w_d.contiguous()
    ld = c2w_d.shape[-1]
    stack = c2w_d.dim() == 3
    if c2w_d.dim() not in (2, 3) or tuple(c2w_d.shape[-2:]) not in ((3, 4), (4, 4)):
        raise _lib.CtxNerfError(f"raygen: c2w must be [3|4, 4] or [N, 3|4, 4], got {tuple(c2w_d.shape)}")
    n_views = c2w_d.shape[0] if stack else 1
    fx, fy, cx, cy = float(K[0][0]), float(K[1][1]), float(K[0][2]), float(K[1][2])
    if ray_idx is not None:
        ray_idx = ray_idx.to(device=dev, dtype=torch.int64).contiguous()
        n = ray_idx.numel()
    else:
        n = n_views * H * W
    if out is not None:          # caller-owned (static) outputs: (rays_o, rays_d, viewdirs, z_vals)
        o, d, v, z = out
    else:
        o = torch.empty(n, 3, device=dev, dtype=torch.float32)
        d = torch.empty(n, 3, device=dev, dtype=torch.float32)
        v = torch.empty(n, 3, device=dev, dtype=torch.float32) if want_viewdirs else None
        z = torch.empty(n, n_samples, device=dev, dtype=torch.float32) if n_samples > 0 else None
    nf = torch.empty(n, 2, device=dev, dtype=torch.float32) if want_near_far else None
    if perturb and jitter is None and seed is None and seed_dev is None:
        seed = new_seed()
    import ctypes
    sph = (ctypes.c_float * 4)(*[float(s) for s in sphere]) if sphere is not None else None
    use_ndc, nfoc, nnear = (1, float(ndc[0]), float(ndc[1])) if ndc is not None else (0, 0.0, 0.0)
    jitter = _f32c(jitter)
    args = (int(H), int(W), fx, fy, cx, cy, ptr(c2w_d), int(ld), ptr(ray_idx), n, use_ndc, nfoc, nnear,
            int(n_samples), float(near), float(far), int(lindisp), int(bool(perturb)), ptr(jitter), int(seed or 0),
            ptr(seed_dev), int(sphere is not None), ctypes.cast(sph, ctypes.c_void_p) if sph is not None else None,
            ptr(o), ptr(d), ptr(v), ptr(z), ptr(nf))
    with torch.cuda.device(dev):
        if stack:
            call("ctx_raygen_views", *args, n_views, int(c2w_d.stride(0)), stream_ptr(dev))
        else:
            call("ctx_raygen_fwd", *args, stream_ptr(dev))
    return {"rays_o": o, "rays_d": d, "viewdirs": v, "z_vals": z, "near_far": nf}


def draw_rays(n_views, H, W, R, counters, *, images=None, mode=0, precrop_iters=0, crop=(0, 0), rank=0, world=1,
              seed=0, out=None):
    """Upstream train()'s ray batch drawn on the device (``ctx_draw_rays``): R global ray ids view*H*W + y*W + x and,
    with ``images`` [n_views, H, W, 3] fp32, their target colours.  ``counters`` is the step state ctx_step_tick
    advances ([0] Philox offset, [1] step count).  mode 0: one view per step, R distinct pixels of it (from the centre
    crop of half-extents ``crop`` = (dH, dW) while the step count is below ``precrop_iters``); mode 1: an epoch stream
    over every ray.  Returns (ray_idx [R] int64, target [R,3] or None)."""
    _need_cuda(counters, images)
    dev = counters.device
    if images is not None and (images.dtype != torch.float32 or not images.is_contiguous()):
        raise _lib.CtxNerfError("draw_rays: images must be a contiguous fp32 [n_views, H, W, 3] tensor")
    if out is not None:          # caller-owned (static) outputs: the captured training step
        idx, tgt = out
    else:
        idx = torch.empty(R, device=dev, dtype=torch.int64)
        tgt = torch.empty(R, 3, device=dev, dtype=torch.float32) if images is not None else None
    with torch.cuda.device(dev):
        call("ctx_draw_rays", ptr(images), int(n_views), int(H), int(W), int(R), int(mode), int(precrop_iters),
             int(crop[0]), int(crop[1]), int(rank), int(world), int(seed), ptr(counters), ptr(idx), ptr(tgt),
             stream_ptr(dev))
    return idx, tgt


def stratified(near, far, n_samples, lindisp=False, perturb=False, jitter=None, seed=None):
    """near/far: [R] or [R,1] (any stride) -> z_vals [R,n_samples]."""
    _need_cuda(near, far, jitter)
    dev = near.device
    R = near.shape[0]
    near = near.float()
    far = far.float()
    z = torch.empty(R, n_samples, device=dev, dtype=torch.float32)
    if perturb and jitter is None and seed is None:
        seed = new_seed()
    jitter = _f32c(jitter)
    with torch.cuda.device(dev):
        call("ctx_stratified_fwd", ptr(near), near.stride(0) if R > 1 else 1, ptr(far),
             far.stride(0) if R > 1 else 1, R, int(n_samples), int(lindisp), int(bool(perturb)),
             ptr(jitter), int(seed or 0), ptr(z), stream_ptr(dev))
    return z


class _Ndc(torch.autograd.Function):
    @staticmethod
    def forward(ctx, H, W, focal, near, rays_o, rays_d):
        _need_cuda(rays_o, rays_d)
        shape = rays_d.shape
        o = _f32c(rays_o.expand(shape)).reshape(-1, 3)
        d = _f32c(rays_d).reshape(-1, 3)
        oo, dd = torch.empty_like(o), torch.empty_like(d)
        with torch.cuda.device(d.device):
            call("ctx_ndc_fwd", int(H), int(W), float(focal), float(near), ptr(o), ptr(d), o.shape[0], ptr(oo),
                 ptr(dd), stream_ptr(d.device))
        ctx.save_for_backward(o, d)
        ctx.meta = (int(H), int(W), float(focal), float(near), shape)
        return oo.reshape(shape), dd.reshape(shape)

    @staticmethod
    def backward(ctx, g_o, g_d):
        o, d = ctx.saved_tensors
        H, W, focal, near, shape = ctx.meta
        go, gd = torch.empty_like(o), torch.empty_like(d)
        g_o, g_d = _f32c(g_o), _f32c(g_d)
        with torch.cuda.device(d.device):
            call("ctx_ndc_bwd", H, W, focal, near, ptr(o), ptr(d), ptr(g_o), ptr(g_d), o.shape[0],
                 ptr(go), ptr(gd), stream_ptr(d.device))
        return None, None, None, None, go.reshape(shape), gd.reshape(shape)


def ndc(H, W, focal, near, rays_o, rays_d):
    return _Ndc.apply(H, W, focal, near, rays_o, rays_d)


# ----------------------------------------------------------------- metrics ---
def image_metrics(pred: torch.Tensor, target: torch.Tensor):
    """Reconstruction metrics of rendered images (``ctx_image_metrics``): ``pred`` [B,H,W,3] or [H,W,3] fp32,
    ``target`` of the same shape, fp32 or uint8 (read as u8 / 255), on the same device.  Returns ``(mse, psnr,
    ssim)``, fp64 device tensors [B] (B = 1 for one image): upstream's img2mse and mse2psnr (psnr = -10 log10(mse),
    +inf at mse 0) and SSIM as mip-NeRF's compute_ssim (11-tap Gaussian window, sigma 1.5, max_val 1; H, W >= 11).
    Neither image is clamped."""
    _need_cuda(pred, target)
    if pred.dtype != torch.float32:
        raise _lib.CtxNerfError(f"image_metrics: pred must be fp32, got {pred.dtype}")
    if target.dtype not in (torch.float32, torch.uint8):
        raise _lib.CtxNerfError(f"image_metrics: target must be fp32 or uint8, got {target.dtype}")
    if pred.dim() not in (3, 4) or pred.shape[-1] != 3 or tuple(target.shape) != tuple(pred.shape):
        raise _lib.CtxNerfError(f"image_metrics: pred and target must both be [B,H,W,3] or [H,W,3], got "
                                f"{tuple(pred.shape)} and {tuple(target.shape)}")
    if target.device != pred.device:
        raise _lib.CtxNerfError(f"image_metrics: pred is on {pred.device}, target on {target.device}")
    B, H, W = (1, *pred.shape[:2]) if pred.dim() == 3 else pred.shape[:3]
    if min(H, W) < 11:
        raise _lib.CtxNerfError(f"image_metrics: SSIM's 11-tap window needs H, W >= 11, got {H}x{W}")
    dev = pred.device
    pred, target = pred.contiguous(), target.contiguous()
    mse = torch.empty(B, device=dev, dtype=torch.float64)
    ssim = torch.empty(B, device=dev, dtype=torch.float64)
    if B > 0:
        partials = torch.empty(int(_lib.lib().ctx_image_metrics_partials(B, H, W)), device=dev, dtype=torch.float64)
        with torch.cuda.device(dev):
            call("ctx_image_metrics", ptr(pred), ptr(target), int(target.dtype == torch.uint8), B, H, W, ptr(mse),
                 ptr(ssim), ptr(partials), stream_ptr(dev))
    return mse, mse.log10().mul_(-10.0), ssim
