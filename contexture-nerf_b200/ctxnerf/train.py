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

from . import _lib, ops
from ._lib import CtxNerfError, call, ptr, stream_ptr
from .dist import BucketComm, FlatBucket, dist_backend, world
from .mlp import TILE, forward_raw, pack_into
from .mlp_bwd import wgrad_scratch
from .run_nerf_helpers import NeRF


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return int(default)


class _Plan:
    """Static device buffers of the training step for one batch size R."""

    def __init__(self, tr: "NerfTrainer", R: int):
        dev, S, Sf = tr.device, tr.N_samples, tr.N_samples + tr.N_importance
        f32 = dict(device=dev, dtype=torch.float32)
        self.R = R
        self.idx = torch.zeros(R, device=dev, dtype=torch.int64)
        self.target = torch.zeros(R, 3, **f32)
        self.o, self.d, self.v = (torch.empty(R, 3, **f32) for _ in range(3))
        self.z_c, self.w_c = torch.empty(R, S, **f32), torch.empty(R, S, **f32)
        self.raw_c, self.g_raw_c = torch.empty(R * S, 4, **f32), torch.empty(R * S, 4, **f32)
        self.zs, self.z_f = torch.empty(R, tr.N_importance, **f32), torch.empty(R, Sf, **f32)
        self.raw_f, self.g_raw_f = torch.empty(R * Sf, 4, **f32), torch.empty(R * Sf, 4, **f32)
        self.rgb0, self.rgb = torch.empty(R, 3, **f32), torch.empty(R, 3, **f32)

        def records(P, net):
            ntiles = 4 * ((P + 4 * TILE - 1) // (4 * TILE))     # the 2-CTA kernels work on 4 tiles at a time
            n = ntiles * net._desc.act_tile_bytes
            return (torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev))

        self.acts_c, self.dacts_c = records(R * S, tr.coarse)
        self.acts_f, self.dacts_f = records(R * Sf, tr.fine)
        self.graph = None          # torch.cuda.CUDAGraph of the step (None: not captured yet)
        self.graph_tail = None     # second graph (Adam + re-pack) when the all-reduce runs between the two
        self.eager_steps = 0
        self.kernels_per_step = 0


class NerfTrainer:
    def __init__(self, H, W, K, c2w, near=2.0, far=6.0, N_samples=64, N_importance=128, perturb=1.0,
                 white_bkgd=True, lindisp=False, lr=5e-4, betas=(0.9, 0.999), eps=1e-8, device=None, seed=0,
                 multires=10, multires_views=4):
        self.device = torch.device(device if device is not None else ("cuda", torch.cuda.current_device()))
        dev = self.device
        self.H, self.W, self.K = H, W, K
        self.c2w = torch.as_tensor(c2w, dtype=torch.float32).to(dev).contiguous()
        self.near, self.far = float(near), float(far)
        self.N_samples, self.N_importance = int(N_samples), int(N_importance)
        self.perturb, self.white_bkgd, self.lindisp = float(perturb), bool(white_bkgd), bool(lindisp)
        self.lr, self.betas, self.eps = lr, betas, eps
        # identical initial weights on every rank: construct under a fixed seed
        st = torch.random.get_rng_state()
        torch.manual_seed(seed)
        in_pts, in_views = 3 * (1 + 2 * multires), 3 * (1 + 2 * multires_views)
        self.coarse = NeRF(input_ch=in_pts, input_ch_views=in_views).to(dev)
        self.fine = NeRF(input_ch=in_pts, input_ch_views=in_views).to(dev)
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
        self._seed0 = ops.new_seed() if self.perturb > 0.0 else 0
        # bf16 weight streams of both networks: trainer-owned static buffers, re-packed after every Adam update
        self._pk = {}
        for net in (self.coarse, self.fine):
            d = net._desc
            self._pk[net] = (torch.empty(d.w_bytes, dtype=torch.uint8, device=dev),
                             torch.empty(max(d.wt_bytes, 16), dtype=torch.uint8, device=dev),
                             torch.empty(d.n_fparams, dtype=torch.float32, device=dev))
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

    def _fwd(self, net, rays, P, out, acts):
        o, d, v, z = rays
        w, _, f = self._pk[net]
        call("ctx_mlp_fwd_ex", net._desc.p, ptr(w), ptr(f), 1, None, 0, ptr(o), ptr(d), ptr(v), ptr(z), z.shape[-1],
             net.L_pts, net.L_dirs, P, ptr(out), ptr(acts), None, 0, stream_ptr(self.device))

    def _dgrad(self, net, g_raw, acts, dacts, P, max_sms=0):
        _, wt, f = self._pk[net]
        call("ctx_mlp_dgrad_ex", net._desc.p, ptr(wt), ptr(f), ptr(g_raw), ptr(acts), ptr(dacts), P, int(max_sms),
             stream_ptr(self.device))

    def _wgrad(self, net, acts, dacts, P, max_sms=0):
        sinks, params = self.bucket.sinks_for(net), net._param_list()
        garr = (ctypes.c_void_p * len(sinks))(*[t.data_ptr() for t in sinks])
        parr = (ctypes.c_void_p * len(params))(*[t.data_ptr() for t in params])
        _lib.launch_count += 1     # the view-direction head's post kernel
        call("ctx_mlp_wgrad_ex", net._desc.p, ptr(acts), ptr(dacts), P, ctypes.cast(garr, ctypes.c_void_p), len(sinks),
             ctypes.cast(parr, ctypes.c_void_p), ptr(self._scratch[net]), int(max_sms), stream_ptr(self.device))

    def _comp_train(self, raw, z, d, R, S, target, g_raw, weights, rgb):
        call("ctx_composite_train", ptr(raw), ptr(z), ptr(d), None, R, S, int(self.white_bkgd), ptr(target),
             1.0 / (3.0 * R), ptr(self._loss), ptr(g_raw), ptr(weights), ptr(rgb), stream_ptr(self.device))

    # --------------------------------------------------------- the step body
    def _enqueue_head(self, pl: _Plan):
        """Everything up to (and including) the weight gradients, on the current stream (+ the side stream)."""
        dev, R, S, Ni = self.device, pl.R, self.N_samples, self.N_importance
        Sf, Pc, Pf = S + Ni, pl.R * S, pl.R * (S + Ni)
        jit = self.perturb > 0.0
        main = torch.cuda.current_stream(dev)
        call("ctx_step_tick", ptr(self._ctr), ptr(self._loss), stream_ptr(dev))
        self.bucket.zero_grad()
        ops.raygen(self.H, self.W, self.K, self.c2w, ray_idx=pl.idx, n_samples=S, near=self.near, far=self.far,
                   lindisp=self.lindisp, perturb=jit, seed=self._seed0, seed_dev=self._ctr if jit else None,
                   want_viewdirs=True, out=(pl.o, pl.d, pl.v, pl.z_c))
        rays_c, rays_f = (pl.o, pl.d, pl.v, pl.z_c), (pl.o, pl.d, pl.v, pl.z_f)
        self._timed("mlp_fwd_coarse", lambda: self._fwd(self.coarse, rays_c, Pc, pl.raw_c, pl.acts_c))
        # raw2outputs + img2mse(rgb0, target) + their backward in one pass; the weights feed sample_pdf
        self._comp_train(pl.raw_c, pl.z_c, pl.d, R, S, pl.target, pl.g_raw_c, pl.w_c, pl.rgb0)
        ops.resample_merge(pl.z_c, pl.w_c, Ni, det=not jit, seed=self._seed0 + 1, seed_dev=self._ctr if jit else None,
                           out=(pl.zs, pl.z_f))
        self._timed("mlp_fwd_fine", lambda: self._fwd(self.fine, rays_f, Pf, pl.raw_f, pl.acts_f))
        self._comp_train(pl.raw_f, pl.z_f, pl.d, R, Sf, pl.target, pl.g_raw_f, None, pl.rgb)
        self._timed("mlp_dgrad_fine", lambda: self._dgrad(self.fine, pl.g_raw_f, pl.acts_f, pl.dacts_f, Pf))

        def coarse_chain(dgrad_sms):
            self._timed("mlp_dgrad_coarse",
                        lambda: self._dgrad(self.coarse, pl.g_raw_c, pl.acts_c, pl.dacts_c, Pc, max_sms=dgrad_sms))
            self._timed("mlp_wgrad_coarse", lambda: self._wgrad(self.coarse, pl.acts_c, pl.dacts_c, Pc))

        if self.overlap_backward:
            self._ev0.record(main)
            self._side.wait_event(self._ev0)
            if self.timers is not None:
                g0 = torch.cuda.Event(enable_timing=True)
                g0.record(main)
            with torch.cuda.stream(self._side):
                coarse_chain(self.side_sms)
                self._ev1.record(self._side)
            self._timed("mlp_wgrad_fine", lambda: self._wgrad(self.fine, pl.acts_f, pl.dacts_f, Pf,
                                                              max_sms=self.n_sms - self.side_sms))
            main.wait_event(self._ev1)
            if self.timers is not None:   # span of the concurrent group on the main stream
                g1 = torch.cuda.Event(enable_timing=True)
                g1.record(main)
                self.timers.setdefault("bwd_overlap_group", []).append((g0, g1))
        else:
            self._timed("mlp_wgrad_fine", lambda: self._wgrad(self.fine, pl.acts_f, pl.dacts_f, Pf))
            coarse_chain(0)

    def _enqueue_tail(self):
        dev = self.device
        call("ctx_adam_step_dev", ptr(self.bucket.flat), ptr(self.bucket.grad), ptr(self.exp_avg),
             ptr(self.exp_avg_sq), self.bucket.numel, self.lr, self.betas[0], self.betas[1], self.eps, ptr(self._ctr),
             0.0, 1.0 / self.world_size, stream_ptr(dev))
        self._repack()

    def _plan(self, R: int) -> _Plan:
        pl = self._plans.get(R)
        if pl is None:
            pl = self._plans[R] = _Plan(self, R)
        return pl

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
    def _render(self, ray_idx, perturb, seed=0, max_sms=0):
        """Forward-only coarse+fine render of the given pixels (None = the whole image): dynamic shapes, fresh
        outputs; shares the trainer's packed weights.  ONE C-ABI call: ctx_render_rays (csrc/render.cu) enqueues
        raygen -> MLP -> raw2outputs -> sample_pdf + merge -> MLP -> raw2outputs."""
        dev, S, Ni = self.device, self.N_samples, self.N_importance
        if ray_idx is not None:
            ray_idx = ray_idx.to(device=dev, dtype=torch.int64).reshape(-1).contiguous()
        R = self.H * self.W if ray_idx is None else ray_idx.numel()
        f32 = dict(device=dev, dtype=torch.float32)
        o, d, v = (torch.empty(R, 3, **f32) for _ in range(3))
        z_c, raw_c, w_c = torch.empty(R, S, **f32), torch.empty(R * S, 4, **f32), torch.empty(R, S, **f32)
        zs, z_f = torch.empty(R, Ni, **f32), torch.empty(R, S + Ni, **f32)
        raw_f, w_f = torch.empty(R * (S + Ni), 4, **f32), torch.empty(R, S + Ni, **f32)
        maps_c = [torch.empty(R, 3, **f32)] + [torch.empty(R, **f32) for _ in range(3)]     # rgb, disp, acc, depth
        maps_f = [torch.empty(R, 3, **f32)] + [torch.empty(R, **f32) for _ in range(3)]
        if R == 0:
            return dict(comp_c=(maps_c[0], maps_c[1], maps_c[2], w_c, maps_c[3]),
                        comp_f=(maps_f[0], maps_f[1], maps_f[2], w_f, maps_f[3]), z_f=z_f, raw_f=raw_f, R=0)
        a = _lib.CtxRenderArgs()
        a.H, a.W = self.H, self.W
        a.fx, a.fy, a.cx, a.cy = (float(self.K[0][0]), float(self.K[1][1]), float(self.K[0][2]), float(self.K[1][2]))
        a.c2w, a.c2w_ld = self.c2w.data_ptr(), self.c2w.stride(0)
        a.ray_idx, a.n_rays = (None if ray_idx is None else ray_idx.data_ptr()), R
        a.near, a.far, a.lindisp, a.perturb = self.near, self.far, int(self.lindisp), int(bool(perturb))
        a.seed, a.seed_dev, a.sphere = int(seed), None, None
        a.n_samples, a.n_importance, a.white_bkgd = S, Ni, int(self.white_bkgd)
        a.L_pts, a.L_dirs, a.max_sms = self.coarse.L_pts, self.coarse.L_dirs, int(max_sms)
        for field, net in (("coarse", self.coarse), ("fine", self.fine)):
            w, _, f = self._pk[net]
            cn = getattr(a, field)
            cn.desc, cn.wpacked, cn.fparams = ctypes.addressof(net._desc.blob), w.data_ptr(), f.data_ptr()
        for name, t in (("rays_o", o), ("rays_d", d), ("viewdirs", v), ("z_coarse", z_c), ("raw_coarse", raw_c),
                        ("weights_coarse", w_c), ("z_samples", zs), ("z_fine", z_f), ("raw_fine", raw_f),
                        ("weights_fine", w_f), ("rgb0", maps_c[0]), ("disp0", maps_c[1]), ("acc0", maps_c[2]),
                        ("depth0", maps_c[3]), ("rgb_map", maps_f[0]), ("disp_map", maps_f[1]), ("acc_map", maps_f[2]),
                        ("depth_map", maps_f[3])):
            setattr(a, name, t.data_ptr())
        call("ctx_render_rays", ctypes.byref(a), stream_ptr(dev))
        return dict(comp_c=(maps_c[0], maps_c[1], maps_c[2], w_c, maps_c[3]),
                    comp_f=(maps_f[0], maps_f[1], maps_f[2], w_f, maps_f[3]), z_f=z_f, raw_f=raw_f, R=R)

    def _composite(self, raw, z, d, R, S):
        dev = self.device
        rgb = torch.empty(R, 3, device=dev)
        disp = torch.empty(R, device=dev)
        acc = torch.empty(R, device=dev)
        w = torch.empty(R, S, device=dev)
        depth = torch.empty(R, device=dev)
        call("ctx_composite_fwd", ptr(raw), ptr(z), ptr(d), None, R, S, int(self.white_bkgd), ptr(rgb), ptr(disp),
             ptr(acc), ptr(w), ptr(depth), stream_ptr(dev))
        return rgb, disp, acc, w, depth

    @torch.no_grad()
    def render(self, ray_idx: Optional[torch.Tensor] = None):
        """Inference render of the given pixels (None = the whole H x W image).  Deterministic, as upstream's
        render_kwargs_test (perturb=False, raw_noise_std=0): linspace depths and det=True importance sampling."""
        with torch.cuda.device(self.device):
            fwd = self._render(ray_idx, perturb=False)
        rgb, disp, acc, _, depth = fwd["comp_f"]
        return dict(rgb_map=rgb, disp_map=disp, acc_map=acc, depth_map=depth, rgb0=fwd["comp_c"][0])

    @torch.no_grad()
    def render_view(self, H, W, K, c2w, n_samples=192, sphere=None, near=None, far=None, ray_idx=None):
        """Single-pass render of a view (or of the pixels ``ray_idx`` of it) with the fine network (BASELINE config 4:
        per-ray near/far from the bounding sphere of the normalised mesh, `n_samples` depths per ray, no hierarchical
        pass).  Maps are [H,W,...] for a whole view, [n,...] for a pixel list."""
        dev = self.device
        f32 = dict(device=dev, dtype=torch.float32)
        c2w_d = torch.as_tensor(c2w, dtype=torch.float32).to(dev).contiguous()
        if ray_idx is not None:
            ray_idx = ray_idx.to(device=dev, dtype=torch.int64).reshape(-1).contiguous()
        n = H * W if ray_idx is None else ray_idx.numel()
        o, d, v = (torch.empty(n, 3, **f32) for _ in range(3))
        z, raw, w = torch.empty(n, n_samples, **f32), torch.empty(n * n_samples, 4, **f32), torch.empty(n, n_samples, **f32)
        rgb, disp, acc, depth = torch.empty(n, 3, **f32), torch.empty(n, **f32), torch.empty(n, **f32), torch.empty(n, **f32)
        if n > 0:
            # the single-pass form of ctx_render_rays (n_importance = 0) with the fine network and the sphere interval
            a = _lib.CtxRenderArgs()
            a.H, a.W = int(H), int(W)
            a.fx, a.fy, a.cx, a.cy = float(K[0][0]), float(K[1][1]), float(K[0][2]), float(K[1][2])
            a.c2w, a.c2w_ld = c2w_d.data_ptr(), c2w_d.stride(0)
            a.ray_idx, a.n_rays = (None if ray_idx is None else ray_idx.data_ptr()), n
            a.near, a.far = float(self.near if near is None else near), float(self.far if far is None else far)
            a.lindisp, a.perturb, a.seed, a.seed_dev = 0, 0, 0, None
            sph = None
            if sphere is not None:
                sph = (ctypes.c_float * 4)(*[float(x) for x in sphere])
                a.sphere = ctypes.addressof(sph)
            a.n_samples, a.n_importance, a.white_bkgd = int(n_samples), 0, int(self.white_bkgd)
            a.L_pts, a.L_dirs, a.max_sms = self.fine.L_pts, self.fine.L_dirs, 0
            wp, _, fp = self._pk[self.fine]
            a.coarse.desc, a.coarse.wpacked, a.coarse.fparams = ctypes.addressof(self.fine._desc.blob), wp.data_ptr(), fp.data_ptr()
            for name, t in (("rays_o", o), ("rays_d", d), ("viewdirs", v), ("z_coarse", z), ("raw_coarse", raw),
                            ("weights_coarse", w), ("rgb_map", rgb), ("disp_map", disp), ("acc_map", acc),
                            ("depth_map", depth)):
                setattr(a, name, t.data_ptr())
            with torch.cuda.device(dev):
                call("ctx_render_rays", ctypes.byref(a), stream_ptr(dev))
        if ray_idx is None:
            return dict(rgb_map=rgb.reshape(H, W, 3), disp_map=disp.reshape(H, W), acc_map=acc.reshape(H, W),
                        depth_map=depth.reshape(H, W))
        return dict(rgb_map=rgb, disp_map=disp, acc_map=acc, depth_map=depth)
