"""Host side of the MLP backward: allocates the gradient tensors and the dZ
scratch records and calls ctx_mlp_bwd (dgrad + wgrad kernels)."""
from __future__ import annotations

import ctypes

import torch

from ._lib import call, ptr, stream_ptr


def _grad_targets(module, sinks, dev):
    params = module._param_list()
    if sinks is not None:
        return sinks, params
    sizes = [p.numel() for p in params]
    flat = torch.zeros(sum(sizes), device=dev, dtype=torch.float32)
    grads, off = [], 0
    for p, n in zip(params, sizes):
        grads.append(flat[off:off + n].view_as(p))
        off += n
    return grads, params


def mlp_dgrad(module, packed, acts, P, g_out, max_sms=0):
    """dZ records of every GEMM layer from g_out (ctx_mlp_dgrad_ex).  ``max_sms`` > 0 limits the SMs the kernel
    occupies so that another kernel can run beside it."""
    desc = module._desc
    _, wt, f = packed
    dev = g_out.device
    g = g_out.reshape(P, desc.out_ch).float().contiguous()
    dacts = torch.empty_like(acts)
    with torch.cuda.device(dev):
        call("ctx_mlp_dgrad_ex", desc.p, ptr(wt), ptr(f), ptr(g), ptr(acts), ptr(dacts), P, int(max_sms),
             stream_ptr(dev))
    return dacts


def wgrad_scratch(dev):
    """fp32 scratch of the wgrad kernels (ctx_mlp_wgrad_scratch_floats floats): the per-CTA partial sums and the
    view-direction head's G job."""
    from . import _lib
    return torch.empty(_lib.lib().ctx_mlp_wgrad_scratch_floats(), device=dev, dtype=torch.float32)


def mlp_wgrad(module, acts, dacts, P, sinks=None, max_sms=0, scratch=None):
    """Parameter gradients from the activation and dZ records (ctx_mlp_wgrad_ex); accumulates into ``sinks`` when
    given (returns None), else returns fresh tensors."""
    dev = acts.device
    grads, params = _grad_targets(module, sinks, dev)
    arr = (ctypes.c_void_p * len(grads))(*[t.data_ptr() for t in grads])
    parr = (ctypes.c_void_p * len(params))(*[t.data_ptr() for t in params])
    if scratch is None:
        scratch = wgrad_scratch(dev)
    with torch.cuda.device(dev):
        call("ctx_mlp_wgrad_ex", module._desc.p, ptr(acts), ptr(dacts), P, ctypes.cast(arr, ctypes.c_void_p),
             len(grads), ctypes.cast(parr, ctypes.c_void_p), ptr(scratch), int(max_sms), stream_ptr(dev))
    if sinks is not None:
        return None
    return [gr if p.requires_grad else None for gr, p in zip(grads, params)]


def mlp_backward(module, packed, acts, P, g_out, sinks=None, timed=None):
    """Gradients w.r.t. the module's parameters: dgrad then wgrad on the current stream.

    ``sinks`` (list of fp32 tensors, one per parameter, e.g. views into a flat
    all-reduce bucket): the wgrad kernel accumulates straight into them and
    ``None`` is returned; otherwise fresh zeroed tensors are returned.
    ``timed(name, fn)`` (optional) wraps the two kernel launches ("dgrad", "wgrad")."""
    run = timed if timed is not None else (lambda name, fn: fn())
    dacts = run("dgrad", lambda: mlp_dgrad(module, packed, acts, P, g_out))
    return run("wgrad", lambda: mlp_wgrad(module, acts, dacts, P, sinks))
