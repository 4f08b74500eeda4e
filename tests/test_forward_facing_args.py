"""The forward-facing entry points (density noise, decaying Adam, NDC render driver) reject bad arguments before any
launch, so these checks need no GPU."""
import ctypes

import pytest


def test_noise_entry_points_reject_bad_arguments(libpath):
    from ctxnerf import _lib
    lib = _lib.lib()
    buf = ctypes.c_void_p(16)            # never dereferenced: every call below fails its checks first

    def train_noise(R=4, S=64, std=1.0, stream_id=2, ptrs=True):
        p = buf if ptrs else None
        return lib.ctx_composite_train_noise(p, p, p, R, S, 0, p, 1.0, p, p, None, p, std, 7, None, stream_id, None)

    assert train_noise(ptrs=False) == -1                  # null pointers
    assert train_noise(R=-1) == -1
    assert train_noise(S=0) == -1
    assert train_noise(std=-0.5) == -1
    assert train_noise(std=float("nan")) == -1
    assert train_noise(stream_id=0) == -1                 # the stratified jitter's stream
    assert train_noise(stream_id=1) == -1                 # the sample_pdf uniforms' stream
    assert train_noise(R=0) == 0                          # no rays: nothing to do
    assert lib.ctx_density_noise(None, 4, 64, 1.0, 7, None, 2, None) == -1
    assert lib.ctx_density_noise(buf, -1, 64, 1.0, 7, None, 2, None) == -1
    assert lib.ctx_density_noise(buf, 4, 64, -1.0, 7, None, 2, None) == -1
    assert lib.ctx_density_noise(buf, 4, 64, 1.0, 7, None, 1, None) == -1
    assert lib.ctx_density_noise(buf, 0, 64, 1.0, 7, None, 2, None) == 0


def test_decaying_adam_rejects_bad_arguments(libpath):
    from ctxnerf import _lib
    lib = _lib.lib()
    buf = ctypes.c_void_p(16)
    args = (buf, buf, buf, buf, 8, 5e-4, 0.9, 0.999, 1e-8, buf, 0.0, 1.0)
    for decay_steps in (0.0, -1.0, float("nan")):
        assert lib.ctx_adam_step_dev_decay(*args, decay_steps, None) == -1
    assert lib.ctx_adam_step_dev_decay(buf, buf, buf, buf, 8, 5e-4, 0.9, 0.999, 1e-8, None, 0.0, 1.0, 250e3,
                                       None) == -1                # no step counters
    assert lib.ctx_adam_step_dev_decay(*args[:4], -1, *args[5:], 250e3, None) == -1


def test_ndc_render_driver_rejects_bad_arguments(libpath):
    from ctxnerf import _lib
    lib = _lib.lib()
    assert lib.ctx_render_rays_ndc(None, 30.0, 1.0, None) == -1
    a = _lib.CtxRenderArgs()
    a.n_rays, a.n_samples = 0, 64
    assert lib.ctx_render_rays_ndc(ctypes.byref(a), 30.0, 1.0, None) == 0          # no rays: nothing to do
    for focal, near in ((0.0, 1.0), (30.0, 0.0), (float("nan"), 1.0)):
        assert lib.ctx_render_rays_ndc(ctypes.byref(a), focal, near, None) == -1
    sph = (ctypes.c_float * 4)(0.0, 0.0, -2.0, 1.0)
    a.sphere = ctypes.addressof(sph)                                               # metric interval: refused
    assert lib.ctx_render_rays_ndc(ctypes.byref(a), 30.0, 1.0, None) == -1
    a.sphere, a.n_rays = None, 16
    assert lib.ctx_render_rays_ndc(ctypes.byref(a), 30.0, 1.0, None) == -1          # no network / buffers


def test_trainer_rejects_negative_options():
    from ctxnerf._lib import CtxNerfError
    from ctxnerf.train import NerfTrainer
    K = [[30.0, 0.0, 16.0], [0.0, 30.0, 16.0], [0.0, 0.0, 1.0]]
    c2w = [[1.0, 0.0, 0.0, 0.0], [0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0]]
    with pytest.raises(CtxNerfError):
        NerfTrainer(32, 32, K, c2w, raw_noise_std=-1.0, device="cpu")
    with pytest.raises(CtxNerfError):
        NerfTrainer(32, 32, K, c2w, lrate_decay=-250, device="cpu")
