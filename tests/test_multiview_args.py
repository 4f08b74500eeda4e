"""Multi-view training entry points (ctx_raygen_views, ctx_draw_rays) and NerfTrainer's multi-view arguments reject
bad input before any launch or device work, so these checks need no GPU."""
import ctypes

import pytest

K = [[30.0, 0.0, 16.0], [0.0, 30.0, 16.0], [0.0, 0.0, 1.0]]
C2W = [[1.0, 0.0, 0.0, 0.0], [0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0]]


def test_draw_rays_rejects_bad_arguments(libpath):
    from ctxnerf import _lib
    lib = _lib.lib()
    buf = ctypes.c_void_p(16)            # never dereferenced: every call below fails its checks first

    def draw(images=buf, n_views=3, H=16, W=16, R=64, mode=0, precrop_iters=0, dh=4, dw=4, rank=0, world=1,
             counters=buf, idx=buf, target=buf):
        return lib.ctx_draw_rays(images, n_views, H, W, R, mode, precrop_iters, dh, dw, rank, world, 7, counters, idx,
                                 target, None)

    assert draw(idx=None) == -1                               # null ray-id output
    assert draw(images=None) == -1                            # targets asked for, no images
    assert draw(counters=None) == -1                          # no step counters
    assert draw(R=-1) == -1
    assert draw(R=257) == -1                                  # mode 0: more distinct pixels than one image has
    assert draw(R=65, precrop_iters=10) == -1                 # ... than the 8 x 8 centre crop has
    assert draw(precrop_iters=10, dh=0) == -1                 # empty crop
    assert draw(precrop_iters=10, dw=0) == -1
    assert draw(precrop_iters=10, dh=9) == -1                 # crop larger than the image
    assert draw(rank=2, world=2) == -1                        # rank >= world
    assert draw(rank=-1, world=2) == -1
    assert draw(world=0) == -1
    assert draw(n_views=1 << 15, H=256, W=256) == -1          # n_views*H*W >= 2^31
    assert draw(mode=2) == -1
    assert draw(mode=1, precrop_iters=10) == -1               # the crop belongs to the one-image sampler
    assert draw(n_views=0) == -1
    assert draw(R=0) == 0                                     # nothing to draw
    assert draw(R=0, images=None, target=None) == 0           # ids only
    assert draw(mode=1, R=0) == 0


def test_raygen_views_rejects_bad_arguments(libpath):
    from ctxnerf import _lib
    lib = _lib.lib()
    buf = ctypes.c_void_p(16)

    def views(n_views=3, stride=12, H=16, W=16, n=8, poses=buf, ld=4, idx=buf, outs=True):
        o = buf if outs else None
        return lib.ctx_raygen_views(H, W, 30.0, 30.0, 8.0, 8.0, poses, ld, idx, n, 0, 0.0, 0.0, 16, 2.0, 6.0, 0, 0,
                                    None, 0, None, 0, None, o, o, None, None, None, n_views, stride, None)

    assert views(poses=None) == -1
    assert views(n_views=0) == -1
    assert views(stride=8) == -1                              # poses overlap: stride below 3 rows
    assert views(ld=3) == -1
    assert views(n_views=1 << 15, H=256, W=256) == -1         # n_views*H*W >= 2^31
    assert views(idx=None, n=3 * 16 * 16 + 1) == -1           # all rays of the stack, and one more
    assert views(outs=False) == -1
    assert views(n=-1) == -1
    assert views(n=0) == 0
    assert views(stride=16, n=0) == 0                         # [N,4,4] stacks


def test_trainer_rejects_bad_multiview_arguments():
    import torch
    from ctxnerf._lib import CtxNerfError
    from ctxnerf.train import NerfTrainer
    poses = torch.tensor(C2W)[None].repeat(3, 1, 1)
    for images in (torch.zeros(2, 32, 32, 3), torch.zeros(3, 16, 32, 3), torch.zeros(3, 32, 16, 3),
                   torch.zeros(3, 32, 32, 4)):
        with pytest.raises(CtxNerfError):
            NerfTrainer(32, 32, K, poses, images=images, device="cpu")
    with pytest.raises(CtxNerfError):                           # one pose, three images
        NerfTrainer(32, 32, K, C2W, images=torch.zeros(3, 32, 32, 3), device="cpu")
    for frac in (0.0, -0.5, 1.5, float("nan")):
        with pytest.raises(CtxNerfError):
            NerfTrainer(32, 32, K, poses, images=torch.zeros(3, 32, 32, 3), precrop_iters=10, precrop_frac=frac,
                        device="cpu")
    with pytest.raises(CtxNerfError):                           # a crop of no pixel
        NerfTrainer(2, 2, K, poses, precrop_iters=10, precrop_frac=0.4, device="cpu")
    with pytest.raises(CtxNerfError):                           # the crop is a one-image sampler's
        NerfTrainer(32, 32, K, poses, precrop_iters=10, no_batching=False, device="cpu")
    for bad in (torch.zeros(3, 3, 3), torch.zeros(2, 4), torch.zeros(0, 3, 4), torch.zeros(2, 2, 3, 4)):
        with pytest.raises(CtxNerfError):
            NerfTrainer(32, 32, K, bad, device="cpu")


def test_step_random_needs_images():
    """Checked before any device work: the method is called on a bare instance that owns no device state at all."""
    from ctxnerf._lib import CtxNerfError
    from ctxnerf.train import NerfTrainer
    tr = object.__new__(NerfTrainer)
    tr.images = None
    with pytest.raises(CtxNerfError, match="images"):
        tr.step_random(4096)
