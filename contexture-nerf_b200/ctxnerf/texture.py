"""Fused ``get_texture_map`` of the reference's TexturedMeshModel
(/root/reference/src/models/textured_mesh.py:266-301): UV grid -> 2-D L=10 positional encoding -> NeRF2D
42->3 -> (tanh+1)/2 -> [1,3,res,res], forward and backward, without materialising the grid or its encoding.

Drop-in use inside the reference::

    from ctxnerf.texture import get_texture_map
    TexturedMeshModel.get_texture_map = lambda self: get_texture_map(self.texture_mlp, self.texture_resolution)

(``self.texture_mlp`` may be the ``nn.DataParallel`` wrapper of trainer.py:134-135: it is unwrapped.)
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import call, ptr, stream_ptr
from .mlp import launch_fwd
from .mlp_bwd import mlp_backward


class _TextureMapFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, res, need_grad, *params):
        module._ensure()
        desc = module._desc
        if desc.in_views != 0 or desc.in_pts != 2 * (1 + 2 * module.L_pts):
            raise _lib.CtxNerfError("get_texture_map needs the 2-D texture MLP (input_ch = 2*(1+2*multires), no views)")
        dev = params[0].device
        P = res * res
        packed = module._packed.get(list(params))
        raw = torch.empty(P, desc.out_ch, device=dev, dtype=torch.float32)
        acts = torch.empty(desc.record_bytes(P), dtype=torch.uint8, device=dev) if need_grad else None
        tex = torch.empty(1, desc.out_ch, res, res, device=dev, dtype=torch.float32)
        launch_fwd(module, packed, raw, res=res, acts=acts)
        with torch.cuda.device(dev):
            call("ctx_tanh01_fwd", ptr(raw), ptr(tex), P, desc.out_ch, stream_ptr(dev))
        ctx.module, ctx.P, ctx.acts, ctx.packed, ctx.raw = module, P, acts, packed, raw
        return tex, raw

    @staticmethod
    def backward(ctx, g_tex, g_raw_in):
        desc = ctx.module._desc
        dev = ctx.raw.device
        g_raw = torch.empty_like(ctx.raw)
        gt = g_tex.float().contiguous() if g_tex is not None else None
        gi = g_raw_in.float().contiguous() if g_raw_in is not None else None
        with torch.cuda.device(dev):
            call("ctx_tanh01_bwd", ptr(ctx.raw), ptr(gt), ptr(gi), ptr(g_raw), ctx.P, desc.out_ch, stream_ptr(dev))
        grads = mlp_backward(ctx.module, ctx.packed, ctx.acts, ctx.P, g_raw)
        ctx.acts = None
        return (None, None, None) + tuple(grads)


def get_texture_map(texture_mlp, res: int):
    """-> (texture [1,3,res,res] in [0,1], mlp_output [res*res,3]) like the reference method.

    ``texture_mlp`` may be the ``nn.DataParallel`` wrapper the reference puts around the MLP on a multi-GPU box
    (/root/reference/src/training/trainer.py:134-135): the fused query generates its UV grid inside the kernel, there
    is no input batch to scatter, so it runs on the wrapped module's own device (the wrapper adds nothing here;
    scattered ``texture_mlp(embedding)`` calls go through DataParallel as usual)."""
    if isinstance(texture_mlp, torch.nn.DataParallel):
        texture_mlp = texture_mlp.module
    params = texture_mlp._param_list()
    need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
    return _TextureMapFn.apply(texture_mlp, int(res), need_grad, *params)


class _TextureValidFn(torch.autograd.Function):
    """MLP at the listed texels only + scatter into the [res*res, C] image (textured_mesh.py:331-347)."""

    @staticmethod
    def forward(ctx, module, uvs, idx, n_pix, scale, need_grad, *params):
        module._ensure()
        desc = module._desc
        if desc.in_views != 0 or desc.in_pts != 2 * (1 + 2 * module.L_pts):
            raise _lib.CtxNerfError("the valid-area texture query needs the 2-D texture MLP (no views)")
        dev = params[0].device
        M = idx.numel()
        packed = module._packed.get(list(params))
        raw = torch.empty(M, desc.out_ch, device=dev, dtype=torch.float32)
        acts = torch.empty(desc.record_bytes(M), dtype=torch.uint8, device=dev) if need_grad and M else None
        final = torch.empty(n_pix, desc.out_ch, device=dev, dtype=torch.float32)
        launch_fwd(module, packed, raw, x=uvs, gather=idx, acts=acts)
        with torch.cuda.device(dev):
            call("ctx_rows_scatter", ptr(raw), ptr(idx), float(scale), ptr(final), M, n_pix, desc.out_ch, stream_ptr(dev))
        ctx.module, ctx.M, ctx.acts, ctx.packed, ctx.idx, ctx.scale = module, M, acts, packed, idx, float(scale)
        return final

    @staticmethod
    def backward(ctx, g_final):
        desc = ctx.module._desc
        if ctx.acts is None:
            return (None,) * 6 + tuple(None for _ in ctx.needs_input_grad[6:])
        dev = g_final.device
        g_raw = torch.empty(ctx.M, desc.out_ch, device=dev, dtype=torch.float32)
        gf = g_final.float().contiguous()
        with torch.cuda.device(dev):
            call("ctx_rows_gather", ptr(gf), ptr(ctx.idx), ctx.scale, ptr(g_raw), ctx.M, desc.out_ch, stream_ptr(dev))
        grads = mlp_backward(ctx.module, ctx.packed, ctx.acts, ctx.M, g_raw)
        ctx.acts = None
        return (None,) * 6 + tuple(grads)


def get_texture_map_only_valid_areas(texture_mlp, interpolated_uvs, face_idx, res=None, scale=0.8 / 0.5):
    """The query + scatter half of the reference's ``get_texture_map_only_valid_areas``
    (/root/reference/src/models/textured_mesh.py:303-347): the MLP is evaluated ONLY at the texels the UV atlas
    covers.  ``interpolated_uvs`` [1,res,res,2] and ``face_idx`` [1,res,res] are what the rasteriser returns there
    (:321-326, kaolin: out of scope); the covered texels are compacted, their UVs gathered and encoded inside the MLP
    kernel (mode 3), and ``colors * scale`` (``unscale_image``, :336-338) scattered into a zero image.
    Returns [1, C, res, res].  Gradients flow to the MLP parameters."""
    from .view_weights import create_face_view_map
    if isinstance(texture_mlp, torch.nn.DataParallel):
        texture_mlp = texture_mlp.module
    if not (interpolated_uvs.is_cuda and face_idx.is_cuda):
        raise _lib.CtxNerfError("ctxnerf texture queries run on CUDA tensors only (no CPU fallback)")
    H, W = face_idx.shape[-2], face_idx.shape[-1]
    if res is not None and (H != res or W != res):
        raise _lib.CtxNerfError("face_idx does not match the texture resolution")
    rows = create_face_view_map(face_idx.reshape(1, 1, H, W))          # (face, view, i, j) of the covered texels
    idx = (rows[:, 2] * W + rows[:, 3]).contiguous()
    uvs = interpolated_uvs.detach().reshape(H * W, 2).float().contiguous()
    params = texture_mlp._param_list()
    need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
    final = _TextureValidFn.apply(texture_mlp, uvs, idx, H * W, scale, need_grad, *params)
    return final.reshape(H, W, -1).permute(2, 0, 1).unsqueeze(0)


class _TexMapFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, uv, texture, mask, bg, mode):
        if not (uv.is_cuda and texture.is_cuda):
            raise _lib.CtxNerfError("ctxnerf texture_mapping runs on CUDA tensors only (no CPU fallback)")
        dev = uv.device
        B = uv.shape[0]
        dims = tuple(uv.shape[1:-1])
        uv2 = uv.detach().reshape(B, -1, 2).float().contiguous()
        N = uv2.shape[1]
        tex = texture.float().contiguous()
        Bt, C, H, W = tex.shape
        if Bt != B and Bt != 1:
            raise _lib.CtxNerfError("texture batch must be 1 or match uv")
        m2 = mask.detach().reshape(B, N).float().contiguous() if mask is not None else None
        bg2 = bg.detach().reshape(C).float().contiguous() if bg is not None else None
        out = torch.empty(B, N, C, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            call("ctx_texmap_fwd", ptr(uv2), ptr(tex), ptr(m2), ptr(bg2), ptr(out), B, N, Bt, C, H, W, mode,
                 stream_ptr(dev))
        ctx.save_for_backward(uv2, m2 if m2 is not None else torch.empty(0, device=dev))
        ctx.meta = (B, N, Bt, C, H, W, mode, m2 is not None)
        return out.reshape(B, *dims, C)

    @staticmethod
    def backward(ctx, g):
        uv2, m2 = ctx.saved_tensors
        B, N, Bt, C, H, W, mode, has_mask = ctx.meta
        dev = uv2.device
        g2 = g.reshape(B, N, C).float().contiguous()
        g_tex = torch.zeros(Bt, C, H, W, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            call("ctx_texmap_bwd", ptr(uv2), ptr(m2 if has_mask else None), ptr(g2), ptr(g_tex), B, N, Bt, C, H, W,
                 mode, stream_ptr(dev))
        return None, g_tex, None, None, None


_MODES = {"nearest": 0, "bilinear": 1, "bicubic": 2}


def texture_mapping(texture_coordinates, texture_maps, mode="nearest", mask=None, background=None):
    """``kal.render.mesh.texture_mapping(uv, texture, mode)`` as used at /root/reference/src/models/render.py:135
    (uv [B,...,2] in [0,1], texture [B or 1, C, H, W] -> [B,...,C]); optionally fused with the two lines that follow
    it there: ``* mask`` and ``+ background * (1 - mask)`` (``mask`` [B,...,1], ``background`` scalar or C values).
    Only the texture receives a gradient (upstream detaches the coordinates).  Modes: the three render.py:9 allows
    ('nearest', 'bilinear', 'bicubic')."""
    if mode not in _MODES:
        raise _lib.CtxNerfError(f"texture_mapping mode {mode!r} not supported (nearest, bilinear, bicubic)")
    bg = None
    if mask is not None and background is not None:
        C = texture_maps.shape[1]
        bg = torch.as_tensor(background, dtype=torch.float32, device=texture_maps.device).reshape(-1)
        bg = bg.expand(C) if bg.numel() == 1 else bg
    return _TexMapFn.apply(texture_coordinates, texture_maps, mask, bg, _MODES[mode])
