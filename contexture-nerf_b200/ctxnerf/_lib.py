"""ctypes binding of libctxnerf.so (include/ctxnerf.h).

There is deliberately no fallback: if the library is missing or a call fails
the wrapper raises.  The product path never routes through PyTorch eager math
or the CPU oracle.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libctxnerf.so")

_lib = None

P = c_void_p  # every device pointer


_SIGNATURES = {
    "ctx_abi_version": (c_int, []),
    "ctx_error_string": (c_char_p, [c_int]),
    "ctx_posenc_fwd": (c_int, [P, P, c_int64, c_int, c_int, c_int, c_int, P]),
    "ctx_posenc_bwd": (c_int, [P, P, P, c_int64, c_int, c_int, c_int, c_int, P]),
    "ctx_raygen_fwd": (c_int, [c_int, c_int, c_float, c_float, c_float, c_float, P, c_int, P, c_int64,
                               c_int, c_float, c_float, c_int, c_float, c_float, c_int, c_int, P,
                               c_uint64, P, c_int, P, P, P, P, P, P, P]),
    "ctx_raygen_views": (c_int, [c_int, c_int, c_float, c_float, c_float, c_float, P, c_int, P, c_int64,
                                 c_int, c_float, c_float, c_int, c_float, c_float, c_int, c_int, P,
                                 c_uint64, P, c_int, P, P, P, P, P, P, c_int, c_int, P]),
    "ctx_draw_rays": (c_int, [P, c_int, c_int, c_int, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_uint64, P,
                              P, P, P]),
    "ctx_stratified_fwd": (c_int, [P, c_int64, P, c_int64, c_int64, c_int, c_int, c_int, P, c_uint64, P, P]),
    "ctx_ndc_fwd": (c_int, [c_int, c_int, c_float, c_float, P, P, c_int64, P, P, P]),
    "ctx_ndc_bwd": (c_int, [c_int, c_int, c_float, c_float, P, P, P, P, c_int64, P, P, P]),
    "ctx_composite_fwd": (c_int, [P, P, P, P, c_int64, c_int, c_int, P, P, P, P, P, P]),
    "ctx_composite_bwd": (c_int, [P, P, P, P, c_int64, c_int, c_int, P, P, P, P, P, P, P]),
    "ctx_resample_fwd": (c_int, [P, c_int64, c_int, P, c_int64, P, P, c_int, c_uint64, P, c_int64, c_int,
                                 c_int, P, P, P, c_int64, c_int, P, P]),
    "ctx_resample_bwd": (c_int, [P, c_int64, c_int, P, c_int64, P, c_int, c_uint64, c_int64, c_int, c_int,
                                 P, P, P]),
    "ctx_mlp_net_bytes": (c_int, []),
    "ctx_mlp_describe": (c_int, [c_int, ctypes.c_uint32, c_int, c_int, c_int, P]),
    "ctx_mlp_pack": (c_int, [P, P, c_int, P, P, P, P]),
    "ctx_mlp_fwd": (c_int, [P, P, P, c_int, P, c_int, P, P, P, P, c_int, c_int, c_int, c_int64, P, P, P]),
    "ctx_mlp_fwd_ex": (c_int, [P, P, P, c_int, P, c_int, P, P, P, P, c_int, c_int, c_int, c_int64, P, P, P, c_int, P]),
    "ctx_rows_scatter": (c_int, [P, P, c_float, P, c_int64, c_int64, c_int, P]),
    "ctx_rows_gather": (c_int, [P, P, c_float, P, c_int64, c_int, P]),
    "ctx_mlp_dgrad": (c_int, [P, P, P, P, P, P, c_int64, P]),
    "ctx_mlp_wgrad": (c_int, [P, P, P, c_int64, P, c_int, P, P, P]),
    "ctx_mlp_bwd": (c_int, [P, P, P, P, P, P, c_int64, P, c_int, P, P, P]),
    "ctx_mlp_dgrad_ex": (c_int, [P, P, P, P, P, P, c_int64, c_int, P]),
    "ctx_mlp_wgrad_ex": (c_int, [P, P, P, c_int64, P, c_int, P, P, c_int, P]),
    "ctx_mlp_wgrad_scratch_floats": (c_int, []),
    "ctx_composite_train": (c_int, [P, P, P, P, c_int64, c_int, c_int, P, c_float, P, P, P, P, P]),
    "ctx_composite_train_noise": (c_int, [P, P, P, c_int64, c_int, c_int, P, c_float, P, P, P, P, c_float, c_uint64,
                                          P, c_int, P]),
    "ctx_density_noise": (c_int, [P, c_int64, c_int, c_float, c_uint64, P, c_int, P]),
    "ctx_texmap_fwd": (c_int, [P, P, P, P, P, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, P]),
    "ctx_texmap_bwd": (c_int, [P, P, P, P, c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, P]),
    "ctx_tanh01_fwd": (c_int, [P, P, c_int64, c_int, P]),
    "ctx_tanh01_bwd": (c_int, [P, P, P, P, c_int64, c_int, P]),
    "ctx_adam_step": (c_int, [P, P, P, P, c_int64, c_float, c_float, c_float, c_float, c_int, c_float, c_float, P]),
    "ctx_view_weight_masks": (c_int, [P, P, c_int, c_int, c_int, c_int, P, P, P, P]),
    "ctx_face_view_map_blocks": (c_int64, [c_int64]),
    "ctx_face_view_map": (c_int, [P, c_int, c_int, c_int, P, P, c_int, P]),
    "ctx_step_tick": (c_int, [P, P, P]),
    "ctx_adam_step_dev": (c_int, [P, P, P, P, c_int64, c_float, c_float, c_float, c_float, P, c_float, c_float, P]),
    "ctx_adam_step_dev_decay": (c_int, [P, P, P, P, c_int64, c_float, c_float, c_float, c_float, P, c_float, c_float,
                                        c_float, P]),
    "ctx_mse_fwd_bwd": (c_int, [P, P, P, c_int64, c_float, P, P, P, P]),
    "ctx_render_rays": (c_int, [P, P]),
    "ctx_render_rays_ndc": (c_int, [P, c_float, c_float, P]),
    "ctx_render_args_bytes": (c_int, []),
    "ctx_image_metrics": (c_int, [P, P, c_int, c_int, c_int, c_int, P, P, P, P]),
    "ctx_image_metrics_partials": (c_int64, [c_int, c_int, c_int]),
    "ctx_density_grid_workspace": (c_int64, [c_int, c_int, c_int]),
    "ctx_density_grid": (c_int, [P, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float,
                                 c_float, P, c_int64, P, P]),
    "ctx_marching_cubes_workspace": (c_int64, [c_int, c_int, c_int]),
    "ctx_marching_cubes": (c_int, [P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_float,
                                   c_float, P, c_int64, P, P, P, P, c_int, P]),
    "ctx_vertex_colors_workspace": (c_int64, [c_int64]),
    "ctx_vertex_colors": (c_int, [P, c_int, c_int, P, P, c_int64, P, c_int64, P, P]),
    "ctx_comm_load": (c_int, [ctypes.c_char_p]),
    "ctx_comm_version": (c_int, []),
    "ctx_comm_last_error": (ctypes.c_char_p, []),
    "ctx_comm_unique_id": (c_int, [P]),
    "ctx_comm_init": (c_int, [P, c_int, P, c_int]),
    "ctx_comm_destroy": (c_int, [P]),
    "ctx_allreduce": (c_int, [P, P, c_int64, P]),
}


class CtxNet(ctypes.Structure):
    """CtxNet of include/ctxnerf.h"""
    _fields_ = [("desc", c_void_p), ("wpacked", c_void_p), ("fparams", c_void_p)]


class CtxRenderArgs(ctypes.Structure):
    """CtxRenderArgs of include/ctxnerf.h (field for field; ctx_render_args_bytes() checks the layout)"""
    _fields_ = ([("H", c_int), ("W", c_int), ("fx", c_float), ("fy", c_float), ("cx", c_float), ("cy", c_float),
                 ("c2w", c_void_p), ("c2w_ld", c_int), ("ray_idx", c_void_p), ("n_rays", c_int64),
                 ("near", c_float), ("far", c_float), ("lindisp", c_int), ("perturb", c_int), ("seed", c_uint64),
                 ("seed_dev", c_void_p), ("sphere", c_void_p), ("n_samples", c_int), ("n_importance", c_int),
                 ("white_bkgd", c_int), ("L_pts", c_int), ("L_dirs", c_int), ("max_sms", c_int),
                 ("coarse", CtxNet), ("fine", CtxNet)]
                + [(n, c_void_p) for n in ("rays_o", "rays_d", "viewdirs", "z_coarse", "raw_coarse", "weights_coarse",
                                           "z_samples", "z_fine", "raw_fine", "weights_fine", "rgb0", "disp0", "acc0",
                                           "depth0", "rgb_map", "disp_map", "acc_map", "depth_map")])


# diagnostics build (libctxnerf_diag.so, include/ctxnerf_diag.h): tools/ and one GPU test only
_DIAG_SIGNATURES = {
    "ctx_mlp_set_prof_buffer": (c_int, [P]),
    "ctx_mlp_set_debug": (c_int, [c_int]),
    "ctx_mlp_set_hang_buffer": (c_int, [P]),
    "ctx_dgrad_set_prof": (c_int, [P]),
    "ctx_tcgen05_selftest": (c_int, [P, P, P, c_int, c_int, c_int, c_int, P]),
    "ctx_tcgen05_mma_rate": (c_int, [c_int, c_int, c_int, c_int, P, c_int, P, P]),
    "ctx_tcgen05_sync_cost": (c_int, [P, c_int, P]),
    "ctx_tcgen05_selftest2": (c_int, [P, P, P, c_int, c_int, P]),
}
DIAG_LIB_PATH = os.path.join(_HERE, "libctxnerf_diag.so")


class CtxNerfError(RuntimeError):
    pass


def use_diag_lib() -> ctypes.CDLL:
    """Switch this process to the diagnostics build (call before the first kernel launch): the same entry points
    plus the profiling / micro-benchmark hooks of include/ctxnerf_diag.h."""
    global _lib, LIB_PATH
    if not os.path.exists(DIAG_LIB_PATH):
        raise CtxNerfError(f"{DIAG_LIB_PATH} not found: python contexture-nerf_b200/ctxnerf/build.py --diag")
    LIB_PATH = DIAG_LIB_PATH
    _lib = None
    handle = lib()
    for name, (res, args) in _DIAG_SIGNATURES.items():
        fn = getattr(handle, name)
        fn.restype = res
        fn.argtypes = args
    return handle


def lib() -> ctypes.CDLL:
    """Load libctxnerf.so (once).  Raises loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CtxNerfError(
            f"{LIB_PATH} not found: build the CUDA extension first "
            "(python __graft_entry__.py build, or python contexture-nerf_b200/ctxnerf/build.py). "
            "ctxnerf has no CPU or eager-PyTorch fallback.")
    handle = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(handle, name)
        except AttributeError:
            continue  # reported by tests/test_abi_symbols.py; calling it raises below
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().ctx_error_string(int(code))
        text = msg.decode() if msg else "?"
        if code == -3:      # CTX_ERR_NO_NCCL: the detail lives in the communicator binding
            detail = lib().ctx_comm_last_error()
            text += f" [{detail.decode() if detail else ''}]"
        raise CtxNerfError(f"{what} failed with code {code}: {text}")


# kernels launched per ABI call (bench.py reports the total as gpu_launches)
KERNELS_PER_CALL = {"ctx_mlp_bwd": 3, "ctx_mlp_wgrad": 2, "ctx_mlp_wgrad_ex": 2, "ctx_composite_train": 2, "ctx_composite_train_noise": 2, "ctx_render_rays": 6, "ctx_render_rays_ndc": 6, "ctx_image_metrics": 2, "ctx_allreduce": 0, "ctx_comm_load": 0, "ctx_comm_unique_id": 0, "ctx_comm_init": 0, "ctx_comm_destroy": 0}     # (the view-direction wgrad also runs a small post kernel: +1, counted by mlp_bwd.launch_wgrad only)
launch_count = 0


def call(name: str, *args) -> None:
    global launch_count
    launch_count += KERNELS_PER_CALL.get(name, 1)
    fn = getattr(lib(), name, None)
    if fn is None:
        raise CtxNerfError(f"libctxnerf.so does not export {name}; rebuild the extension")
    check(fn(*args), name)


def ptr(t) -> c_void_p:
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return c_void_p(0)
    return c_void_p(t.data_ptr())


def stream_ptr(device=None) -> c_void_p:
    import torch
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)
