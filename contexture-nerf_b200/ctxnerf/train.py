"""The coarse+fine NeRF training / rendering step built from the ctxnerf
kernels -- the hot path BASELINE.json measures.

One step = ray generation fused with stratified sampling -> coarse MLP (points
encoded in shared memory) -> raw2outputs fused with the loss and its own
backward -> sample_pdf + merge -> fine MLP -> fused raw2outputs/loss/backward ->
hand-written MLP backward (dgrad, wgrad) of both networks -> one gradient
all-reduce -> Adam -> re-pack of the bf16 weight streams.  It is upstream's
render()+train iteration (SURVEY.md 3.2) with the same hyper-parameter names;
every numeric stage is a libctxnerf.so kernel, orchestrated here without
autograd.

The step works on STATIC buffers (allocated once per batch size) and keeps its
per-step state -- Philox seed offset, Adam step count, loss -- on the device, so
the whole launch sequence is captured once into a CUDA graph and replayed
(SURVEY.md 8f row 3): no host-side argument changes between steps.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

from . import _lib, mesh, ops
from ._lib import CtxNerfError, call, ptr, stream_ptr
from .dist import BucketComm, FlatBucket, dist_backend, world
from .mlp import launch_fwd, pack_into
from .mlp_bwd import launch_dgrad, launch_wgrad, wgrad_scratch
from .run_nerf_helpers import NeRF


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return int(default)


class _Plan:
    """Static device buffers of the training step for one batch size R."""

    def __init__(self, tr: "NerfTrainer", R: int, draw: bool = False):
        dev, S, Sf = tr.device, tr.N_samples, tr.N_samples + tr.N_importance
        f32 = dict(device=dev, dtype=torch.float32)
        self.R = R
        self.draw = draw           # True: the step draws idx / target itself (ctx_draw_rays); False: the caller's batch
        self.idx = torch.zeros(R, device=dev, dtype=torch.int64)
        self.target = torch.zeros(R, 3, **f32)
        self.o, self.d, self.v = (torch.empty(R, 3, **f32) for _ in range(3))
        self.z_c, self.w_c = torch.empty(R, S, **f32), torch.empty(R, S, **f32)
        self.raw_c, self.g_raw_c = torch.empty(R * S, 4, **f32), torch.empty(R * S, 4, **f32)
        self.zs, self.z_f = torch.empty(R, tr.N_importance, **f32), torch.empty(R, Sf, **f32)
        self.raw_f, self.g_raw_f = torch.empty(R * Sf, 4, **f32), torch.empty(R * Sf, 4, **f32)
        self.rgb0, self.rgb = torch.empty(R, 3, **f32), torch.empty(R, 3, **f32)

        def records(P, net):
            n = net._desc.record_bytes(P)
            return (torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev))

        self.acts_c, self.dacts_c = records(R * S, tr.coarse)
        self.acts_f, self.dacts_f = records(R * Sf, tr.fine)
        self.graph = None          # torch.cuda.CUDAGraph of the step (None: not captured yet)
        self.graph_tail = None     # second graph (Adam + re-pack) when the all-reduce runs between the two
        self.eager_steps = 0
        self.kernels_per_step = 0


class NerfTrainer:
    """Upstream nerf-pytorch's training step on one camera or a set of posed images.  The defaults are its Blender
    recipe; its forward-facing (LLFF) recipe is ``ndc=True, near=0, far=1, raw_noise_std=1.0, lrate_decay=250,
    white_bkgd=False, no_batching=False``:

    * ``c2w``: one pose [3|4, 4] or a stack [N, 3|4, 4] (one K for every view, as upstream).  ``step`` takes global ray
      ids view*H*W + y*W + x (with one pose, the pixel ids y*W + x).  The stack lives on the device as ``poses``;
      ``c2w`` is its first pose.
    * ``images`` [N, H, W, 3] (float in [0, 1], or uint8), the training images of the poses, kept on the device as
      fp32.  ``step_random(N_rand)`` then draws each step's batch on the device, inside the captured step, as upstream's
      loop does: ``no_batching=True`` takes one random image per step and N_rand distinct pixels of it (from the
      centre crop ``precrop_frac`` for the first ``precrop_iters`` steps); ``no_batching=False`` walks a stream over
      every ray of every image, reshuffled each epoch (csrc/raybatch.cu gives the construction).

    * ``ndc``: rays are warped by ``ndc_rays(H, W, K[0][0], 1., ...)`` after the view directions are taken, so
      near / far are NDC depths.  Training, ``render`` and ``render_view`` all use the warped rays.
    * ``raw_noise_std``: the training step adds ``raw_noise_std * randn`` to every density, drawn inside the fused
      compositing kernels (Philox key ``seed0 + counter``, stream 2 coarse, 3 fine): fresh on every step, reproducible
      under ``torch.manual_seed``.  Renders stay noise-free, as upstream's ``render_kwargs_test``.
    * ``lrate_decay`` (thousands of steps): Adam's update ``t`` uses
      ``lr * 0.1 ** (max(t - 2, 0) / (lrate_decay * 1000))``, the rate upstream's loop sets; 0 keeps ``lr`` constant.
    """

    def __init__(self, H, W, K, c2w, near=2.0, far=6.0, N_samples=64, N_importance=128, perturb=1.0,
                 white_bkgd=True, lindisp=False, lr=5e-4, betas=(0.9, 0.999), eps=1e-8, device=None, seed=0,
                 multires=10, multires_views=4, ndc=False, raw_noise_std=0.0, lrate_decay=0, images=None,
                 no_batching=True, precrop_iters=0, precrop_frac=0.5):
        c2w_h = torch.as_tensor(c2w, dtype=torch.float32)
        if c2w_h.dim() not in (2, 3) or tuple(c2w_h.shape[-2:]) not in ((3, 4), (4, 4)):
            raise CtxNerfError(f"NerfTrainer: c2w must be [3|4, 4] or a stack [N, 3|4, 4], got {tuple(c2w_h.shape)}")
        n_views = c2w_h.shape[0] if c2w_h.dim() == 3 else 1
        if n_views < 1:
            raise CtxNerfError("NerfTrainer: the pose stack is empty")
        if n_views * H * W >= 2 ** 31:
            raise CtxNerfError("NerfTrainer: N*H*W must stay below 2^31 (global ray ids are split in 32 bits)")
        if images is not None:
            shape = tuple(images.shape)
            if shape != (n_views, H, W, 3):
                raise CtxNerfError(f"NerfTrainer: images must be [N, H, W, 3] = {(n_views, H, W, 3)} for {n_views} "
                                   f"pose(s) of {H}x{W}, got {shape}")
        if not (0.0 < precrop_frac <= 1.0):
            raise CtxNerfError("NerfTrainer: precrop_frac must lie in (0, 1]")
        if not precrop_iters >= 0:
            raise CtxNerfError("NerfTrainer: precrop_iters must be >= 0")
        if precrop_iters > 0 and not no_batching:
            raise CtxNerfError("NerfTrainer: precrop_iters crops the one image a step draws from (no_batching=True)")
        crop = (int(H // 2 * precrop_frac), int(W // 2 * precrop_frac))     # upstream's dH, dW
        if precrop_iters > 0 and min(crop) < 1:
            raise CtxNerfError(f"NerfTrainer: the centre crop of precrop_frac={precrop_frac} is empty at {H}x{W}")
        if not raw_noise_std >= 0.0:
            raise CtxNerfError("NerfTrainer: raw_noise_std must be >= 0")
        if not lrate_decay >= 0:
            raise CtxNerfError("NerfTrainer: lrate_decay must be >= 0 (thousands of steps; 0 = constant rate)")
        self.device = torch.device(device if device is not None else ("cuda", torch.cuda.current_device()))
        dev = self.device
        self.H, self.W, self.K = H, W, K
        self.n_views = n_views
        if c2w_h.dim() == 3:
            self.poses = c2w_h.to(dev).contiguous()
            self.c2w = self.poses[0]
        else:
            self.c2w = c2w_h.to(dev).contiguous()
            self.poses = self.c2w[None]
        self.no_batching, self.precrop_iters, self.precrop_frac = bool(no_batching), int(precrop_iters), precrop_frac
        self._crop = crop
        self.near, self.far = float(near), float(far)
        self.N_samples, self.N_importance = int(N_samples), int(N_importance)
        self.perturb, self.white_bkgd, self.lindisp = float(perturb), bool(white_bkgd), bool(lindisp)
        self.lr, self.betas, self.eps = lr, betas, eps
        self.ndc, self.raw_noise_std, self.lrate_decay = bool(ndc), float(raw_noise_std), lrate_decay
        # identical initial weights on every rank: construct under a fixed seed
        st = torch.random.get_rng_state()
        torch.manual_seed(seed)
        in_pts, in_views = 3 * (1 + 2 * multires), 3 * (1 + 2 * multires_views)
        self.coarse = NeRF(input_ch=in_pts, input_ch_views=in_views).to(dev)
        self.fine = NeRF(input_ch=in_pts, input_ch_views=in_views).to(dev)
        # key of the epoch stream (no_batching=False): from the same seed, so every rank walks the same permutation
        self._stream_key = ops.new_seed() if images is not None and not no_batching else 0
        torch.random.set_rng_state(st)
        for net in (self.coarse, self.fine):
            net.L_pts, net.L_dirs = multires, multires_views
            net._ensure()
        self.bucket = FlatBucket([self.coarse, self.fine])
        self.exp_avg = torch.zeros_like(self.bucket.flat)
        self.exp_avg_sq = torch.zeros_like(self.bucket.flat)
        self.rank, self.world_size = world()
        # gradient all-reduce through the library's own NCCL binding (ctx_allreduce on the step's stream: the whole
        # step is then one graph); CTXNERF_NCCL=0 or a non-NCCL process group -> torch.distributed between two graphs
        self.comm = None
        if self.world_size > 1 and os.environ.get("CTXNERF_NCCL", "1") != "0" and "nccl" in dist_backend():
            self.comm = self._make_comm(dev)
        self.reduce_gradients = True       # (tools/dist_check.py turns the exchange off for its single-process sums)
        # The bucket is all-reduced in one call after the join of the two backward chains.  bench.py reads this flag
        # to name the route; a two-halves route measured slower and was removed (DESIGN.md §5), so it is always False.
        self.split_reduce = False
        self._loss = torch.zeros(1, device=dev)
        # device-side step state: [0] Philox seed offset, [1] Adam step count (ctx_step_tick advances both)
        self._ctr = torch.zeros(2, device=dev, dtype=torch.int64)
        # the Philox base seed comes from torch's generator: torch.manual_seed makes a training run reproducible
        # (a trainer with images keys its per-step image and pixel draw with it too)
        self._seed0 = ops.new_seed() if self.perturb > 0.0 or self.raw_noise_std > 0.0 or images is not None else 0
        self.images = None
        if images is not None:
            im = torch.as_tensor(images)
            im = im.to(dev).float().div_(255.0) if im.dtype == torch.uint8 else im.to(dev, dtype=torch.float32)
            self.images = im.contiguous()
        # bf16 weight streams of both networks: trainer-owned static buffers, re-packed after every Adam update
        self._pk = {net: net._desc.weight_buffers(dev) for net in (self.coarse, self.fine)}
        self._scratch = {net: wgrad_scratch(dev) for net in (self.coarse, self.fine)}
        self._packed_version = -1
        self._plans = {}
        self.timers = None      # optional dict name -> list[(start_event, end_event)]; forces the eager path
        self.n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
        # Backward schedule: the two networks' chains are independent and their kernels bind on different resources
        # (dgrad: tensor pipe / epilogue; wgrad: HBM reads).  The coarse chain runs on a side stream inside an SM
        # budget while wgrad of the fine network streams its records through the other SMs.
        self.overlap_backward = os.environ.get("CTXNERF_OVERLAP", "1") != "0"
        self.side_sms = _env_int("CTXNERF_SIDE_SMS", 44)
        self.use_graph = os.environ.get("CTXNERF_GRAPH", "1") != "0"
        self._side = torch.cuda.Stream(device=dev)
        self._pack_stream = torch.cuda.Stream(device=dev)
        self._ev0, self._ev1, self._ev2, self._ev3 = (torch.cuda.Event() for _ in range(4))
        with torch.cuda.device(dev):
            self._repack()

    @staticmethod
    def _make_comm(dev):
        """The library's NCCL communicator, or None (-> torch.distributed's all-reduce) when it cannot be had on EVERY
        rank: the outcome is agreed through the existing process group so that no rank waits in a collective the
        others never enter.  A failure is reported, not hidden (stderr, once per rank)."""
        import sys
        import torch.distributed as dist
        comm, err = None, None
        try:
            comm = BucketComm(dev)
        except Exception as e:          # no NCCL shared object, version outside 2.x, init error
            err = e
        ok = torch.tensor([1 if comm is not None else 0], device=dev, dtype=torch.int32)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 1:
            return comm
        if comm is not None:
            comm.close()
        print(f"ctxnerf: ctx_allreduce unavailable on at least one rank ({err}); using torch.distributed for the "
              "gradient all-reduce", file=sys.stderr, flush=True)
        return None

    @property
    def step_count(self) -> int:
        return int(self._ctr[1].item())

    # ------------------------------------------------------------------ utils
    def _timed(self, name, fn):
        if self.timers is None:
            return fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        self.timers.setdefault(name, []).append((a, b))
        return r

    def _repack(self):
        """bf16 operand images of both networks from the fp32 bucket (two independent launches: the fine network's
        on a side stream)."""
        dev = self.device
        main = torch.cuda.current_stream(dev)
        self._ev2.record(main)
        self._pack_stream.wait_event(self._ev2)
        with torch.cuda.stream(self._pack_stream):
            pack_into(self.fine._desc, self.fine._param_list(), self._pk[self.fine])
            self._ev3.record(self._pack_stream)
        pack_into(self.coarse._desc, self.coarse._param_list(), self._pk[self.coarse])
        main.wait_event(self._ev3)

    def _comp_train(self, raw, z, d, R, S, target, g_raw, weights, rgb, noise_stream):
        # the noise has the raygen key (seed0 + counter) and its own Philox stream per pass; raw_noise_std == 0 runs
        # the launches of ctx_composite_train without noise
        call("ctx_composite_train_noise", ptr(raw), ptr(z), ptr(d), R, S, int(self.white_bkgd), ptr(target),
             1.0 / (3.0 * R), ptr(self._loss), ptr(g_raw), ptr(weights), ptr(rgb), self.raw_noise_std,
             self._seed0, ptr(self._ctr), noise_stream, stream_ptr(self.device))

    # --------------------------------------------------------- the step body
    def _enqueue_head(self, pl: _Plan):
        """Everything up to (and including) the weight gradients, on the current stream (+ the side stream)."""
        dev, R, S, Ni = self.device, pl.R, self.N_samples, self.N_importance
        Sf, Pc, Pf = S + Ni, pl.R * S, pl.R * (S + Ni)
        jit = self.perturb > 0.0
        main = torch.cuda.current_stream(dev)
        call("ctx_step_tick", ptr(self._ctr), ptr(self._loss), stream_ptr(dev))
        if pl.draw:
            ops.draw_rays(self.n_views, self.H, self.W, R, self._ctr, images=self.images,
                          mode=0 if self.no_batching else 1, precrop_iters=self.precrop_iters, crop=self._crop,
                          rank=self.rank, world=self.world_size,
                          seed=self._seed0 if self.no_batching else self._stream_key, out=(pl.idx, pl.target))
        self.bucket.zero_grad()
        # one pose: ctx_raygen_fwd; a stack: ctx_raygen_views (each ray the pose of its view)
        ops.raygen(self.H, self.W, self.K, self.c2w if self.n_views == 1 else self.poses, ray_idx=pl.idx, n_samples=S,
                   near=self.near, far=self.far, lindisp=self.lindisp, perturb=jit, seed=self._seed0, seed_dev=self._ctr if jit else None,
                   ndc=self._ndc_args(self.K), want_viewdirs=True, out=(pl.o, pl.d, pl.v, pl.z_c))
        c, f, pk, sinks = self.coarse, self.fine, self._pk, self.bucket.sinks_for
        self._timed("mlp_fwd_coarse", lambda: launch_fwd(c, pk[c], pl.raw_c, rays=(pl.o, pl.d, pl.v, pl.z_c),
                                                         acts=pl.acts_c))
        # raw2outputs + img2mse(rgb0, target) + their backward in one pass; the weights feed sample_pdf
        self._comp_train(pl.raw_c, pl.z_c, pl.d, R, S, pl.target, pl.g_raw_c, pl.w_c, pl.rgb0, 2)
        ops.resample_merge(pl.z_c, pl.w_c, Ni, det=not jit, seed=self._seed0 + 1, seed_dev=self._ctr if jit else None,
                           out=(pl.zs, pl.z_f))
        self._timed("mlp_fwd_fine", lambda: launch_fwd(f, pk[f], pl.raw_f, rays=(pl.o, pl.d, pl.v, pl.z_f),
                                                       acts=pl.acts_f))
        self._comp_train(pl.raw_f, pl.z_f, pl.d, R, Sf, pl.target, pl.g_raw_f, None, pl.rgb, 3)
        self._timed("mlp_dgrad_fine", lambda: launch_dgrad(f, pk[f], pl.g_raw_f, pl.acts_f, pl.dacts_f, Pf))

        def coarse_chain(dgrad_sms):
            self._timed("mlp_dgrad_coarse",
                        lambda: launch_dgrad(c, pk[c], pl.g_raw_c, pl.acts_c, pl.dacts_c, Pc, dgrad_sms))
            self._timed("mlp_wgrad_coarse",
                        lambda: launch_wgrad(c, pl.acts_c, pl.dacts_c, Pc, sinks(c), self._scratch[c]))

        def wgrad_fine(max_sms):
            self._timed("mlp_wgrad_fine",
                        lambda: launch_wgrad(f, pl.acts_f, pl.dacts_f, Pf, sinks(f), self._scratch[f], max_sms))

        if self.overlap_backward:
            self._ev0.record(main)
            self._side.wait_event(self._ev0)
            if self.timers is not None:
                g0 = torch.cuda.Event(enable_timing=True)
                g0.record(main)
            with torch.cuda.stream(self._side):
                coarse_chain(self.side_sms)
                self._ev1.record(self._side)
            wgrad_fine(self.n_sms - self.side_sms)
            main.wait_event(self._ev1)
            if self.timers is not None:   # span of the concurrent group on the main stream
                g1 = torch.cuda.Event(enable_timing=True)
                g1.record(main)
                self.timers.setdefault("bwd_overlap_group", []).append((g0, g1))
        else:
            wgrad_fine(0)
            coarse_chain(0)

    def _enqueue_tail(self):
        dev = self.device
        args = (ptr(self.bucket.flat), ptr(self.bucket.grad), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                self.bucket.numel, self.lr, self.betas[0], self.betas[1], self.eps, ptr(self._ctr), 0.0,
                1.0 / self.world_size)
        if self.lrate_decay > 0:
            call("ctx_adam_step_dev_decay", *args, float(self.lrate_decay) * 1000.0, stream_ptr(dev))
        else:
            call("ctx_adam_step_dev", *args, stream_ptr(dev))
        self._repack()

    def _plan(self, R: int, draw: bool = False) -> _Plan:
        """Static buffers (and graphs) of one batch size: ``_plans[R]`` for the caller's batches, ``_plans[(R, "draw")]``
        for batches the step draws itself."""
        key = (R, "draw") if draw else R
        pl = self._plans.get(key)
        if pl is None:
            pl = self._plans[key] = _Plan(self, R, draw)
        return pl

    def _ndc_args(self, K):
        """(focal, near) of the NDC warp upstream applies to forward-facing scenes, or None"""
        return (float(K[0][0]), 1.0) if self.ndc else None

    def _render_rays(self, H, W, K, pose, ray_idx, n_rays, near, far, nets, bufs, n_samples, n_importance=0,
                     lindisp=False, perturb=False, seed=0, sphere=None):
        """One ctx_render_rays (ctx_render_rays_ndc on an NDC trainer) of ``n_rays`` > 0 rays of the device pose
        ``pose``: ``nets`` holds the network of the first pass and, with ``n_importance`` > 0, the fine one; ``bufs``
        maps CtxRenderArgs buffer fields to device tensors (the others stay NULL); ``sphere``: (cx, cy, cz, r)."""
        a = _lib.CtxRenderArgs()
        a.H, a.W = int(H), int(W)
        a.fx, a.fy, a.cx, a.cy = float(K[0][0]), float(K[1][1]), float(K[0][2]), float(K[1][2])
        a.c2w, a.c2w_ld = pose.data_ptr(), pose.stride(0)
        a.ray_idx, a.n_rays = (None if ray_idx is None else ray_idx.data_ptr()), n_rays
        a.near, a.far, a.lindisp, a.perturb = float(near), float(far), int(lindisp), int(bool(perturb))
        a.seed = int(seed)
        sph = None      # the sphere array must outlive the call
        if sphere is not None:
            sph = (ctypes.c_float * 4)(*[float(x) for x in sphere])
            a.sphere = ctypes.addressof(sph)
        a.n_samples, a.n_importance, a.white_bkgd = int(n_samples), int(n_importance), int(self.white_bkgd)
        a.L_pts, a.L_dirs = nets[0].L_pts, nets[0].L_dirs
        for cn, net in zip((a.coarse, a.fine), nets):
            w, _, f = self._pk[net]
            cn.desc, cn.wpacked, cn.fparams = ctypes.addressof(net._desc.blob), w.data_ptr(), f.data_ptr()
        for name, t in bufs.items():
            setattr(a, name, t.data_ptr())
        nd = self._ndc_args(K)
        with torch.cuda.device(self.device):
            if nd is None:
                call("ctx_render_rays", ctypes.byref(a), stream_ptr(self.device))
            else:
                call("ctx_render_rays_ndc", ctypes.byref(a), nd[0], nd[1], stream_ptr(self.device))

    # ------------------------------------------------------------------- API
    @torch.no_grad()
    def step(self, ray_idx: torch.Tensor, target: torch.Tensor, optimizer_step: bool = True) -> torch.Tensor:
        """One training step on this rank's ray batch; returns the loss (device scalar, valid once the stream has
        reached the end of the step)."""
        dev = self.device
        if not (torch.is_tensor(target) and target.is_cuda and target.device == dev):
            raise CtxNerfError("NerfTrainer.step: target must be a CUDA tensor on the trainer's device "
                               "(use step_from_host for host buffers)")
        if not (torch.is_tensor(ray_idx) and ray_idx.is_cuda and ray_idx.device == dev):
            raise CtxNerfError("NerfTrainer.step: ray_idx must be a CUDA tensor on the trainer's device")
        R = ray_idx.numel()
        if target.numel() != 3 * R:
            raise CtxNerfError("NerfTrainer.step: target must hold one rgb triple per ray")
        if R == 0:
            return self._loss.zero_()
        with torch.cuda.device(dev):
            pl = self._plan(R)
            pl.idx.copy_(ray_idx.reshape(-1), non_blocking=True)
            pl.target.copy_(target.reshape(R, 3), non_blocking=True)     # (casts a non-fp32 target)
            self._run(pl, optimizer_step)
        return self._loss

    @torch.no_grad()
    def step_random(self, N_rand: int, optimizer_step: bool = True) -> torch.Tensor:
        """One training step on a batch of N_rand rays drawn on the device from the training images, as upstream's
        loop draws it (``no_batching``, ``precrop_iters``, ``precrop_frac``); returns the loss (device scalar).  The
        draw is part of the step: a captured step draws a fresh batch on every replay, and the batch of the last step
        is in ``_plans[(N_rand, "draw")].idx / .target``.  Under several ranks each rank draws its own share."""
        if self.images is None:
            raise CtxNerfError("NerfTrainer.step_random draws from the training images: build the trainer with images=")
        R = int(N_rand)
        if R < 1:
            raise CtxNerfError("NerfTrainer.step_random: N_rand must be >= 1")
        if self.no_batching:
            dom = self.H * self.W
            if self.precrop_iters > 0:
                dom = min(dom, 4 * self._crop[0] * self._crop[1])
            if R > dom:
                raise CtxNerfError(f"NerfTrainer.step_random: N_rand={R} distinct pixels of one image, but the "
                                   f"{'centre crop' if dom < self.H * self.W else 'image'} has {dom}")
        with torch.cuda.device(self.device):
            pl = self._plan(R, draw=True)
            self._run(pl, optimizer_step)
        return self._loss

    def _all_reduce(self):
        """The exchange step after the join of the two backward chains: the whole gradient bucket."""
        if not self.reduce_gradients:
            return
        if self.comm is not None:
            self.comm.all_reduce(self.bucket.grad)
        else:
            self.bucket.all_reduce()

    def _run(self, pl: _Plan, optimizer_step: bool):
        multi = self.world_size > 1 and self.comm is None      # all-reduce outside the graph (torch.distributed)
        if optimizer_step:     # the modules' own pack caches (direct net(x) calls) do not see the in-place Adam update
            self.coarse._packed.invalidate()
            self.fine._packed.invalidate()
        graphable = self.use_graph and self.timers is None and optimizer_step
        if not graphable or pl.eager_steps < 1:
            # eager launch sequence (first step of a batch size: sets the kernels' attributes; timed passes)
            l0 = _lib.launch_count
            self._enqueue_head(pl)
            self._all_reduce()
            if optimizer_step:
                self._enqueue_tail()
            if graphable:
                pl.eager_steps += 1
                pl.kernels_per_step = _lib.launch_count - l0
            return
        if pl.graph is None:
            self._capture(pl, multi)
        _lib.launch_count += pl.kernels_per_step
        pl.graph.replay()
        if multi:
            self._all_reduce()
            pl.graph_tail.replay()

    def _capture(self, pl: _Plan, multi: bool):
        """Capture the step into one CUDA graph (single process, or N processes with the library's NCCL binding: the
        all-reduce is a node of the graph) or two with torch.distributed's all-reduce between them."""
        dev = self.device
        torch.cuda.synchronize(dev)
        saved = _lib.launch_count
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._enqueue_head(pl)
                if not multi:
                    self._all_reduce()
                    self._enqueue_tail()
            tail = None
            if multi:
                tail = torch.cuda.CUDAGraph()
                with torch.cuda.graph(tail, capture_error_mode="thread_local"):
                    self._enqueue_tail()
        except Exception as e:                      # pragma: no cover - depends on driver / NCCL state
            raise CtxNerfError(f"CUDA-graph capture of the training step failed ({e}); set CTXNERF_GRAPH=0 to run the "
                               "eager launch sequence") from e
        finally:
            _lib.launch_count = saved
        pl.graph, pl.graph_tail = g, tail

    def step_from_host(self, ray_idx_pinned: torch.Tensor, target_pinned: torch.Tensor,
                       loss_pinned: torch.Tensor) -> "torch.cuda.Event":
        """End-to-end entry: host (pinned) inputs in, loss back to the host.  Asynchronous: the returned event marks
        the arrival of the loss in ``loss_pinned``, so a training loop can submit step i+1 before it reads the loss
        of step i (the launches of the next step then hide behind the GPU work of this one)."""
        dev = self.device
        R = ray_idx_pinned.numel()
        if target_pinned.numel() != 3 * R:
            raise CtxNerfError("NerfTrainer.step_from_host: target must hold one rgb triple per ray")
        with torch.cuda.device(dev):
            pl = self._plan(R)
            pl.idx.copy_(ray_idx_pinned.reshape(-1), non_blocking=True)              # host -> device, inside the step
            pl.target.copy_(target_pinned.reshape(R, 3), non_blocking=True)
            self._run(pl, True)
            loss_pinned.copy_(self._loss, non_blocking=True)
            done = torch.cuda.Event()
            done.record(torch.cuda.current_stream(dev))
        return done     # loss_pinned is valid once this event has completed

    # ------------------------------------------------------------ inference
    def _render(self, ray_idx, perturb, seed=0, c2w=None):
        """Forward-only coarse+fine render of the given pixels (None = the whole image): dynamic shapes, fresh
        outputs; shares the trainer's packed weights.  ONE C-ABI call: ctx_render_rays (csrc/render.cu) enqueues
        raygen -> MLP -> raw2outputs -> sample_pdf + merge -> MLP -> raw2outputs."""
        dev, S, Ni = self.device, self.N_samples, self.N_importance
        if ray_idx is not None:
            ray_idx = ray_idx.to(device=dev, dtype=torch.int64).reshape(-1).contiguous()
        R = self.H * self.W if ray_idx is None else ray_idx.numel()
        f32 = dict(device=dev, dtype=torch.float32)
        b = {n: torch.empty(R, 3, **f32) for n in ("rays_o", "rays_d", "viewdirs", "rgb0", "rgb_map")}
        b.update({n: torch.empty(R, **f32) for n in ("disp0", "acc0", "depth0", "disp_map", "acc_map", "depth_map")})
        b.update({n: torch.empty(R, S, **f32) for n in ("z_coarse", "weights_coarse")})
        b.update({n: torch.empty(R, S + Ni, **f32) for n in ("z_fine", "weights_fine")})
        b.update(raw_coarse=torch.empty(R * S, 4, **f32), z_samples=torch.empty(R, Ni, **f32),
                 raw_fine=torch.empty(R * (S + Ni), 4, **f32))
        if R > 0:
            pose = self.c2w
            if c2w is not None:
                pose = torch.as_tensor(c2w, dtype=torch.float32).to(dev).contiguous()
                if tuple(pose.shape) not in ((3, 4), (4, 4)):
                    raise CtxNerfError(f"NerfTrainer.render: c2w must be one pose [3|4, 4], got {tuple(pose.shape)}")
            self._render_rays(self.H, self.W, self.K, pose, ray_idx, R, self.near, self.far, (self.coarse, self.fine),
                              b, S, Ni, lindisp=self.lindisp, perturb=perturb, seed=seed)
        return dict(comp_c=tuple(b[n] for n in ("rgb0", "disp0", "acc0", "weights_coarse", "depth0")),
                    comp_f=tuple(b[n] for n in ("rgb_map", "disp_map", "acc_map", "weights_fine", "depth_map")),
                    z_f=b["z_fine"], raw_f=b["raw_fine"], R=R)

    @torch.no_grad()
    def render(self, ray_idx: Optional[torch.Tensor] = None, c2w=None):
        """Inference render of the given pixels (None = the whole H x W image) of the pose ``c2w`` [3|4, 4] (None = the
        first training pose), with the trainer's K: held-out test poses render through here.  Deterministic, as
        upstream's render_kwargs_test (perturb=False, raw_noise_std=0): linspace depths and det=True importance
        sampling."""
        with torch.cuda.device(self.device):
            fwd = self._render(ray_idx, perturb=False, c2w=c2w)
        rgb, disp, acc, _, depth = fwd["comp_f"]
        return dict(rgb_map=rgb, disp_map=disp, acc_map=acc, depth_map=depth, rgb0=fwd["comp_c"][0])

    @torch.no_grad()
    def evaluate(self, c2w, images):
        """Test-split metrics, as NeRF results are reported: each pose of ``c2w`` [N, 3|4, 4] renders through
        ``render(c2w=pose)`` (deterministic, with the trainer's K, NDC warp and ``white_bkgd``) and is compared with its
        image of ``images`` [N, H, W, 3] (fp32 in [0, 1] or uint8, on the host or the device, at the trainer's H x W) by
        ``ops.image_metrics``.  Returns ``dict(mse=, psnr=, ssim=)``, CPU fp64 tensors [N], one entry per pose:
        upstream's img2mse and mse2psnr, and SSIM as mip-NeRF's compute_ssim.

        The targets must already be composited the way the trainer renders, e.g. onto white for ``white_bkgd=True``
        (upstream's Blender loader does ``rgb * alpha + (1 - alpha)``): neither image is clamped or blended here.  A
        uint8 stack stays uint8 on the device (the kernel converts it); a host stack is copied to the device once, up
        front, and the results come back with one host synchronisation at the end.

        Under several ranks every rank calls ``evaluate`` with the same arguments: rank r renders the views
        v = r mod world, and one all-reduce of the [3, N] results (zero outside a rank's views, so the sum is exact)
        gives every rank the single-process vectors bit for bit.  The training state is left as it was: the step
        counters, the loss, the Adam moments, the weights and their packed images, the captured step graphs and torch's
        random number generator."""
        P = torch.as_tensor(c2w, dtype=torch.float32)
        if P.dim() != 3 or tuple(P.shape[1:]) not in ((3, 4), (4, 4)):
            raise CtxNerfError(f"NerfTrainer.evaluate: c2w must be a stack [N, 3|4, 4], got {tuple(P.shape)}")
        images = torch.as_tensor(images)
        N = P.shape[0]
        if tuple(images.shape) != (N, self.H, self.W, 3):
            raise CtxNerfError(f"NerfTrainer.evaluate: images must be [N, H, W, 3] = {(N, self.H, self.W, 3)} for {N} "
                               f"pose(s) of the trainer's {self.H}x{self.W}, got {tuple(images.shape)}")
        if images.dtype not in (torch.float32, torch.uint8):
            raise CtxNerfError(f"NerfTrainer.evaluate: images must be fp32 or uint8, got {images.dtype}")
        if N == 0:
            empty = torch.empty(0, dtype=torch.float64)
            return dict(mse=empty, psnr=empty.clone(), ssim=empty.clone())
        dev = self.device
        with torch.cuda.device(dev):
            vals = torch.zeros(3, N, device=dev, dtype=torch.float64)
            poses = P.to(dev)
            targets = images[self.rank::self.world_size].to(dev)
            for i, v in enumerate(range(self.rank, N, self.world_size)):
                rgb = self.render(c2w=poses[v])["rgb_map"].view(self.H, self.W, 3)
                vals[:, v] = torch.cat(ops.image_metrics(rgb, targets[i]))
            if self.world_size > 1:
                import torch.distributed as dist
                dist.all_reduce(vals)
            out = vals.cpu()
        return dict(mse=out[0], psnr=out[1], ssim=out[2])

    @torch.no_grad()
    def render_view(self, H, W, K, c2w, n_samples=192, sphere=None, near=None, far=None, ray_idx=None):
        """Single-pass render of a view (or of the pixels ``ray_idx`` of it) with the fine network (BASELINE config 4:
        per-ray near/far from the bounding sphere of the normalised mesh, `n_samples` depths per ray, no hierarchical
        pass).  Maps are [H,W,...] for a whole view, [n,...] for a pixel list.  An NDC trainer warps the view's rays
        with its K[0][0]; the sphere interval is metric and is refused there."""
        dev = self.device
        if self.ndc and sphere is not None:
            raise CtxNerfError("NerfTrainer.render_view: sphere= gives metric depths; an ndc=True trainer renders "
                               "between NDC depths near / far")
        f32 = dict(device=dev, dtype=torch.float32)
        c2w_d = torch.as_tensor(c2w, dtype=torch.float32).to(dev).contiguous()
        if ray_idx is not None:
            ray_idx = ray_idx.to(device=dev, dtype=torch.int64).reshape(-1).contiguous()
        n = H * W if ray_idx is None else ray_idx.numel()
        b = {k: torch.empty(n, 3, **f32) for k in ("rays_o", "rays_d", "viewdirs", "rgb_map")}
        b.update({k: torch.empty(n, **f32) for k in ("disp_map", "acc_map", "depth_map")})
        b.update({k: torch.empty(n, n_samples, **f32) for k in ("z_coarse", "weights_coarse")})
        b.update(raw_coarse=torch.empty(n * n_samples, 4, **f32))
        if n > 0:
            # the single-pass form of ctx_render_rays (n_importance = 0) with the fine network and the sphere interval
            self._render_rays(H, W, K, c2w_d, ray_idx, n, self.near if near is None else near,
                              self.far if far is None else far, (self.fine,), b, n_samples, sphere=sphere)
        rgb, disp, acc, depth = b["rgb_map"], b["disp_map"], b["acc_map"], b["depth_map"]
        if ray_idx is None:
            return dict(rgb_map=rgb.reshape(H, W, 3), disp_map=disp.reshape(H, W), acc_map=acc.reshape(H, W),
                        depth_map=depth.reshape(H, W))
        return dict(rgb_map=rgb, disp_map=disp, acc_map=acc, depth_map=depth)

    # ------------------------------------------------------------ geometry
    def _mesh_net(self, network, what):
        if self.ndc:
            raise CtxNerfError(f"NerfTrainer.{what}: an ndc=True trainer's field lives in NDC space, so a lattice over "
                               "world bounds would not sample it")
        nets = {"fine": self.fine, "coarse": self.coarse}
        if network not in nets:
            raise CtxNerfError(f"NerfTrainer.{what}: network must be 'fine' or 'coarse', got {network!r}")
        return nets[network]

    @torch.no_grad()
    def density_grid(self, resolution=256, bounds=mesh.DEFAULT_BOUNDS, network="fine"):
        """``relu(sigma)`` of the ``network`` ('fine' or 'coarse') on a lattice of ``resolution`` cells (an int or
        ``(nx, ny, nz)``) over ``bounds = (lo, hi)``, with zero view directions, as the original NeRF release's
        ``extract_mesh.ipynb``: fp32 ``[nx+1, ny+1, nz+1]`` on the device (``ctxnerf.mesh.density_grid`` on the
        trainer's packed weights).  The training state is left as it was, and no collective is entered."""
        net = self._mesh_net(network, "density_grid")
        with torch.cuda.device(self.device):
            return mesh.density_grid(net, self._pk[net], resolution, bounds)

    @torch.no_grad()
    def extract_mesh(self, resolution=256, bounds=mesh.DEFAULT_BOUNDS, threshold=50.0, network="fine", colors=True):
        """The surface ``sigma == threshold`` of ``density_grid(resolution, bounds, network)`` by marching cubes
        (upstream thresholds the relu'd density at 50), with a colour per vertex: ``sigmoid(rgb)`` of the same network
        seen along ``-normal``.  Returns ``dict(vertices [V,3], faces [F,3] int32, normals [V,3], colors [V,3] or
        None)`` on the device; ``ctxnerf.mesh.write_ply`` writes it.  The training state is left as it was."""
        net = self._mesh_net(network, "extract_mesh")
        if not float(threshold) > 0.0:
            raise CtxNerfError(f"NerfTrainer.extract_mesh: threshold must be > 0 (the density is relu'd), got "
                               f"{threshold}")
        mesh.lattice(bounds, mesh._cells(resolution))      # refuse bad bounds before any launch
        with torch.cuda.device(self.device):
            sigma = mesh.density_grid(net, self._pk[net], resolution, bounds)
            out = mesh.marching_cubes(sigma, threshold, bounds)
            out["colors"] = mesh.vertex_colors(net, self._pk[net], out["vertices"], out["normals"]) if colors else None
        return out
