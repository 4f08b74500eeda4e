"""Host side of the tcgen05 coordinate MLP: network description, weight
packing, the forward launcher (ctx_mlp_fwd_ex) and the autograd Function that
pairs it with the backward of mlp_bwd.py.

The modules keep the reference's parameter names and order
(/root/reference/src/run_nerf_helpers.py:81-97; trainer.py:888 indexes
``parameters()[-2]``), so ``state_dict`` round-trips with ``NeRF2D``.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib
from ._lib import call, ptr, stream_ptr

TILE = 128


class NetDesc:
    """Opaque CtxMlpNet blob (csrc/mlp_desc.h) + the few fields Python needs."""

    def __init__(self, D: int, skips: Sequence[int], in_pts: int, in_views: int, out_ch: int, W: int = 256):
        if W != 256:
            raise _lib.CtxNerfError(f"the tcgen05 MLP kernel is built for W=256 (got W={W})")
        lib = _lib.lib()
        n = lib.ctx_mlp_net_bytes()
        self.blob = (ctypes.c_uint8 * n)()
        mask = 0
        for s in skips:
            mask |= 1 << int(s)
        _lib.check(lib.ctx_mlp_describe(D, mask, in_pts, in_views, out_ch, ctypes.cast(self.blob, ctypes.c_void_p)),
                   "ctx_mlp_describe")
        ints = ctypes.cast(self.blob, ctypes.POINTER(ctypes.c_int32))
        (self.n_layers, self.in_pts, self.in_views, self.out_ch, self.head_off, self.w_bytes, self.wt_bytes,
         self.n_fparams, self.act_tile_bytes) = [ints[i] for i in range(9)]
        self.D = D

    @property
    def p(self):
        return ctypes.cast(self.blob, ctypes.c_void_p)

    def record_bytes(self, P: int) -> int:
        """Bytes of the activation records of P points (the dZ records take as many)."""
        ntiles = 4 * ((P + 4 * TILE - 1) // (4 * TILE))     # the 2-CTA kernels work on 4 tiles at a time
        return ntiles * self.act_tile_bytes

    def weight_buffers(self, dev):
        """Uninitialised (w, wt, fparams) buffers that ctx_mlp_pack fills: the bf16 forward and transposed weight
        streams and the fp32 bias/head block."""
        return (torch.empty(self.w_bytes, dtype=torch.uint8, device=dev),
                torch.empty(max(self.wt_bytes, 16), dtype=torch.uint8, device=dev),
                torch.empty(self.n_fparams, dtype=torch.float32, device=dev))


class PackedWeights:
    """bf16 weight streams (forward + transposed) and the fp32 bias/head block, per device.

    Cache discipline (ADVICE r1): an entry is keyed on the IDENTITY of the parameter tensors (``id`` of live leaf
    ``nn.Parameter`` objects, held by weak reference so that a recycled id cannot alias) plus their ``_version``
    counters, never on addresses.  Non-leaf parameters -- the per-iteration replicas ``nn.DataParallel`` broadcasts
    (/root/reference/src/training/trainer.py:134-135) -- are always re-packed.  Every pack writes FRESH buffers:
    a saved autograd graph keeps the buffers it ran with (``ctx.packed``), so a later re-pack (forward A, optimizer
    step, forward B, backward A) cannot change the transposed weights under a pending backward."""

    def __init__(self, desc: NetDesc):
        self.desc = desc
        self._per_dev = {}
        self.generation = 0          # number of packs performed (monotone; tests and the trainer read it)

    def invalidate(self):
        """Force a re-pack (parameters were updated in place by a non-torch kernel)."""
        self._per_dev.clear()

    def get(self, params: List[torch.Tensor]):
        import weakref
        dev = params[0].device
        cacheable = all(isinstance(p, torch.nn.Parameter) and p.is_leaf for p in params)
        ent = self._per_dev.get(dev) if cacheable else None
        if ent is not None:
            refs, versions, bufs = ent
            if (len(refs) == len(params) and all(r() is p for r, p in zip(refs, params))
                    and versions == tuple(p._version for p in params)):
                return bufs
        for p in params:
            if p.dtype != torch.float32 or not p.is_contiguous() or p.device != dev or not p.is_cuda:
                raise _lib.CtxNerfError("MLP parameters must be contiguous fp32 tensors on one CUDA device "
                                        "(ctxnerf has no CPU path)")
        bufs = self.desc.weight_buffers(dev)
        pack_into(self.desc, params, bufs)
        self.generation += 1
        if cacheable:
            self._per_dev[dev] = (tuple(weakref.ref(p) for p in params), tuple(p._version for p in params), bufs)
        return bufs


def pack_into(desc: NetDesc, params: List[torch.Tensor], bufs):
    """ctx_mlp_pack of ``params`` (reference order) into the given (w, wt, fparams) buffers on the current stream."""
    dev = params[0].device
    arr = (ctypes.c_void_p * len(params))(*[p.data_ptr() for p in params])
    with torch.cuda.device(dev):
        call("ctx_mlp_pack", desc.p, ctypes.cast(arr, ctypes.c_void_p), len(params), ptr(bufs[0]), ptr(bufs[1]),
             ptr(bufs[2]), stream_ptr(dev))


def launch_fwd(net, packed, out, *, x=None, rays=None, res=None, gather=None, acts=None):
    """The fused forward of ``net`` with the packed weights ``packed`` = (w, wt, fparams), on the current stream:
    ``out`` [P, out_ch] receives the raw output and ``acts`` (optional, ``record_bytes(P)`` bytes) the activation
    records of the backward.  The input picks the kernel's mode:

    * ``x`` [P, in_ch]: encoded inputs (mode 0);
    * ``rays`` = (rays_o, rays_d, viewdirs, z_vals [.., S]): the points o + d z, encoded in the kernel (mode 1);
    * ``res``: the res x res UV grid of get_texture_map, made and encoded in the kernel (mode 2);
    * ``x`` [*, 2|3] raw coordinates with ``gather`` [P] int64, the row of x each point reads (mode 3)."""
    desc, (w, _, f), P, dev = net._desc, packed, out.shape[0], out.device
    o = d = v = z = None
    x_ld = S = L_pts = L_dirs = 0
    if rays is not None:
        for t in rays:
            if t is not None and (not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous()):
                raise _lib.CtxNerfError("fused ray query needs contiguous fp32 CUDA tensors (rays_o, rays_d, viewdirs, "
                                        "z_vals); cast with .float().contiguous()")
        o, d, v, z = rays
        mode, S, L_pts, L_dirs = 1, z.shape[-1], net.L_pts, net.L_dirs
    elif res is not None:
        mode, S, L_pts = 2, res, net.L_pts
    else:
        if not x.is_cuda:
            raise _lib.CtxNerfError("ctxnerf MLP runs on CUDA tensors only (no CPU fallback)")
        x = x.reshape(-1, x.shape[-1]).float().contiguous()
        x_ld = x.shape[-1]
        mode, L_pts = (0, 0) if gather is None else (3, net.L_pts)
    with torch.cuda.device(dev):
        call("ctx_mlp_fwd_ex", desc.p, ptr(w), ptr(f), mode, ptr(x), x_ld, ptr(o), ptr(d), ptr(v), ptr(z), S, L_pts,
             L_dirs, P, ptr(out), ptr(acts), ptr(gather), 0, stream_ptr(dev))


def forward_raw(module, *, x=None, rays=None, save_acts=False):
    """Launch the fused forward.  Returns (out [P,out_ch], acts or None, P, packed)."""
    module._ensure()
    desc: NetDesc = module._desc
    packed = module._packed.get(module._param_list())
    P, dev = (x.shape[:-1].numel(), x.device) if x is not None else (rays[3].numel(), rays[3].device)
    out = torch.empty(P, desc.out_ch, device=dev, dtype=torch.float32)
    acts = torch.empty(desc.record_bytes(P), dtype=torch.uint8, device=dev) if save_acts else None
    launch_fwd(module, packed, out, x=x, rays=rays, acts=acts)
    return out, acts, P, packed


class _MlpFn(torch.autograd.Function):
    """out = MLP(x or rays).  Gradients flow to the parameters only (inputs are
    data: encodings of fixed coordinates)."""

    @staticmethod
    def forward(ctx, module, x, rays, need_grad, *params):
        # The kernels differentiate with respect to the parameters only.  An input that asks for a gradient would
        # silently get none (ADVICE r1): refuse instead, as loudly as the rest of the package.
        for t in ((x,) if x is not None else tuple(rays)):
            if t is not None and t.requires_grad:
                raise _lib.CtxNerfError(
                    "ctxnerf MLP: gradients flow to the parameters only; an input (x / rays_o / rays_d / viewdirs / "
                    "z_vals) has requires_grad=True.  Detach it (upstream never differentiates with respect to rays or "
                    "encodings) -- learnable coordinates are out of scope (DESIGN.md section 7)")
        lead = x.shape[:-1] if x is not None else rays[3].shape
        out, acts, P, packed = forward_raw(module, x=x, rays=rays, save_acts=need_grad)
        ctx.module, ctx.P, ctx.acts, ctx.packed = module, P, acts, packed
        return out.reshape(*lead, module._desc.out_ch)

    @staticmethod
    def backward(ctx, g_out):
        from .mlp_bwd import mlp_backward
        if ctx.acts is None:       # nothing asked for a gradient when the forward ran (all parameters frozen)
            return (None, None, None, None) + tuple(None for _ in ctx.needs_input_grad[4:])
        grads = mlp_backward(ctx.module, ctx.packed, ctx.acts, ctx.P, g_out)
        ctx.acts = None
        return (None, None, None, None) + tuple(grads)


class FusedMLPBase(nn.Module):
    """Shared machinery of NeRF2D / NeRF: parameters are ordinary nn.Linear
    modules (names/order of the reference); forward runs the fused kernel."""

    L_pts = 10
    L_dirs = 4

    def _setup(self, D, W, skips, in_pts, in_views, out_ch):
        self._desc_args = (D, tuple(skips), in_pts, in_views, out_ch, W)
        self.__dict__["_desc"] = None
        self.__dict__["_packed"] = None

    def _ensure(self):
        if self.__dict__.get("_desc") is None:
            D, skips, in_pts, in_views, out_ch, W = self._desc_args
            self.__dict__["_desc"] = NetDesc(D, skips, in_pts, in_views, out_ch, W)
            self.__dict__["_packed"] = PackedWeights(self._desc)

    def _param_list(self) -> List[torch.Tensor]:
        raise NotImplementedError

    def _run(self, x=None, rays=None):
        self._ensure()
        params = self._param_list()
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        return _MlpFn.apply(self, x, rays, need_grad, *params)
