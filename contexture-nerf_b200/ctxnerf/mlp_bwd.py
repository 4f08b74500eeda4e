"""Host side of the MLP backward: the dgrad (ctx_mlp_dgrad_ex) and wgrad (ctx_mlp_wgrad_ex) launchers, which write
into buffers the caller owns, and the functions that allocate those buffers for one backward pass."""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from ._lib import call, ptr, stream_ptr


def launch_dgrad(net, packed, g_out, acts, dacts, P, max_sms=0):
    """dZ records ``dacts`` of every GEMM layer from g_out [P, out_ch] (fp32, contiguous) and the activation records
    ``acts``.  ``max_sms`` > 0 limits the SMs the kernel occupies so that another kernel can run beside it."""
    _, wt, f = packed
    dev = g_out.device
    with torch.cuda.device(dev):
        call("ctx_mlp_dgrad_ex", net._desc.p, ptr(wt), ptr(f), ptr(g_out), ptr(acts), ptr(dacts), P, int(max_sms),
             stream_ptr(dev))


def launch_wgrad(net, acts, dacts, P, grads, scratch, max_sms=0):
    """Accumulates (+=) the parameter gradients into ``grads`` (fp32 tensors in ``net._param_list()`` order) from the
    activation and dZ records; ``scratch`` is ``wgrad_scratch``."""
    params = net._param_list()
    garr = (ctypes.c_void_p * len(grads))(*[t.data_ptr() for t in grads])
    parr = (ctypes.c_void_p * len(params))(*[t.data_ptr() for t in params])
    if net._desc.in_views > 0:
        _lib.launch_count += 1     # the view-direction head's post kernel
    dev = acts.device
    with torch.cuda.device(dev):
        call("ctx_mlp_wgrad_ex", net._desc.p, ptr(acts), ptr(dacts), P, ctypes.cast(garr, ctypes.c_void_p), len(grads),
             ctypes.cast(parr, ctypes.c_void_p), ptr(scratch), int(max_sms), stream_ptr(dev))


def wgrad_scratch(dev):
    """fp32 scratch of the wgrad kernels (ctx_mlp_wgrad_scratch_floats floats): the per-CTA partial sums and the
    view-direction head's G job."""
    return torch.empty(_lib.lib().ctx_mlp_wgrad_scratch_floats(), device=dev, dtype=torch.float32)


def mlp_dgrad(module, packed, acts, P, g_out, max_sms=0):
    """Fresh dZ records from g_out (``launch_dgrad``)."""
    g = g_out.reshape(P, module._desc.out_ch).float().contiguous()
    dacts = torch.empty_like(acts)
    launch_dgrad(module, packed, g, acts, dacts, P, max_sms)
    return dacts


def mlp_wgrad(module, acts, dacts, P, max_sms=0):
    """Fresh parameter gradients from the activation and dZ records (``launch_wgrad``): one tensor per parameter,
    None for a parameter that does not require a gradient."""
    params = module._param_list()
    sizes = [p.numel() for p in params]
    flat = torch.zeros(sum(sizes), device=acts.device, dtype=torch.float32)
    grads = [t.view_as(p) for t, p in zip(flat.split(sizes), params)]
    launch_wgrad(module, acts, dacts, P, grads, wgrad_scratch(acts.device), max_sms)
    return [gr if p.requires_grad else None for gr, p in zip(grads, params)]


def mlp_backward(module, packed, acts, P, g_out):
    """Gradients w.r.t. the module's parameters: dgrad then wgrad on the current stream."""
    return mlp_wgrad(module, acts, mlp_dgrad(module, packed, acts, P, g_out), P)
