#!/usr/bin/env python
"""bench.py -- rays/s of the coarse(64)+fine(128) NeRF training step (fwd+bwd) on B200.

    python bench.py --gpus N --steps K --warmup W           (N > 1: launched by torchrun)
    python bench.py --impl reference ...                    (CPU arm: the oracle port on the host cores)
    python bench.py ... --dump-outputs DIR                  (+ the last timed step's outputs as DIR/<name>.npy)

Prints ONE JSON line (rank 0).  Workload = BASELINE.json configs[2]: 4096 rays per GPU
drawn from the 800x800 config-2 camera, two view-direction D=8/W=256 MLPs, L=10/4
encodings, stratified sampling (perturb=1), white background, MSE loss on rgb and rgb0,
gradient all-reduce, Adam.  Synthetic rays/targets, random-init weights.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "contexture-nerf_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

RAYS_PER_GPU = 4096
N_SAMPLES, N_IMPORTANCE = 64, 128
MACS_PER_EVAL = 593408                       # view-direction net, SURVEY.md 8d
EVALS_PER_RAY = N_SAMPLES + (N_SAMPLES + N_IMPORTANCE)
METRIC = "rays/sec fwd+bwd (64+128 samples)"
CONFIG = {"workload": "configs[2]: training step fwd+bwd, 4096-ray batch per GPU, coarse 64 + fine 128, "
                      "D=8/W=256 view-dir MLPs, L=10/4, gradient all-reduce + Adam",
          "rays_per_gpu": RAYS_PER_GPU, "n_samples": N_SAMPLES, "n_importance": N_IMPORTANCE,
          "image": "800x800 config-2 camera", "perturb": 1.0, "white_bkgd": True,
          "l2": "no explicit flush: each step streams ~15 GB of activation / dZ records through the 126 MB L2",
          "settle": "0.75 s of idle between the warm-up steps and every timed region (fixed; it used to be the random "
                    "start-up time of the clock sampler); `sustained` = the same loop held for 200 steps, by which the board's "
                    "power limiter has engaged (it does after ~40 steps of continuous work)",
          "schedule": "one CUDA graph per step (N > 1: the NCCL all-reduce of the gradient bucket is a node of it, issued "
                      "through the library's ctx_allreduce); backward of the coarse network "
                      "(dgrad -> wgrad) on a side stream beside wgrad of the fine network (SM budgets 44 / 104)"}


SETTLE_S = 0.75


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "tf_burst": p["bf16_tflops"], "tf_sustained": p["bf16_tflops_sustained"],
                "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_first_sample(self, timeout=5.0):
        """nvidia-smi needs a moment to start; block until it has produced a line."""
        t0 = time.time()
        while self.proc is not None and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.02)

    def mark(self):
        self.t_mark = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        t_lo = getattr(self, "t_mark", 0.0) - 0.06      # samples taken during the timed region
        for ts, ln in self.lines:
            if ts < t_lo:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_step_outputs(out_dir, tr):
    """What the last training step computed, as float32 DIR/<name>.npy (about 10 MB in all): its loss, the fine and
    coarse colours of the ray batch, the all-reduced gradient bucket and the parameters after its Adam update (the
    last two: coarse then fine network, named_parameters() order, flattened).  The rays, targets, initial weights and
    jitter seed are fixed, so two builds run with the same arguments can be compared array for array."""
    import numpy as np
    pl = tr._plans[RAYS_PER_GPU]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("loss", tr._loss), ("rgb_map", pl.rgb), ("rgb0", pl.rgb0), ("grads", tr.bucket.grad),
                    ("params", tr.bucket.flat)):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def cpu_step_sample(n_rays, threads, steps, warmup):
    """The oracle port (oracle/nerf_oracle.py) doing the same training step on the host cores."""
    from oracle import nerf_oracle as orc
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    K, c2w = orc.lego_like_camera()
    pc = {k: v.requires_grad_(True) for k, v in orc.init_mlp_params(63, 4, input_ch_views=27, generator=g).items()}
    pf = {k: v.requires_grad_(True) for k, v in orc.init_mlp_params(63, 4, input_ch_views=27, generator=g).items()}
    _, rd = orc.get_rays(800, 800, K, c2w)
    rd = rd.reshape(-1, 3)
    q = lambda pts, vd, prm: orc.run_network(pts, vd, prm)
    times = []
    for it in range(warmup + steps):
        idx = torch.randint(0, 800 * 800, (n_rays,), generator=g)
        d = rd[idx]
        o = c2w[:3, -1].expand(n_rays, 3)
        vd = d / d.norm(dim=-1, keepdim=True)
        rays = torch.cat([o, d, torch.full((n_rays, 1), 2.0), torch.full((n_rays, 1), 6.0), vd], -1)
        tgt = torch.rand(n_rays, 3, generator=g)
        t0 = time.perf_counter()
        out = orc.render_rays(rays, pc, q, N_SAMPLES, N_importance=N_IMPORTANCE, network_fine=pf, perturb=1.0,
                              white_bkgd=True)
        loss = orc.img2mse(out["rgb_map"], tgt) + orc.img2mse(out["rgb0"], tgt)
        for p in list(pc.values()) + list(pf.values()):
            p.grad = None
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return times


def run_reference(args, rank):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # the full 4096-ray batch of the benchmark config (about 5 s per step on 16 cores); --ref-rays bounds it further
    n_rays = args.ref_rays or RAYS_PER_GPU
    times = cpu_step_sample(n_rays, threads, args.steps, min(args.warmup, 2))
    total = sum(times)
    val = n_rays * len(times) / total
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(CONFIG, sample=(f"{n_rays} rays per step" + ("" if n_rays == RAYS_PER_GPU else
                                                                           " (bounded sample of the 4096-ray batch)"))),
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": threads, "kind": "port",
                             "sample": f"{n_rays}-ray coarse+fine fwd+bwd step, oracle/nerf_oracle.py (torch CPU fp32), "
                                       f"{len(times)} steps"},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_cfg1(args):
    """BASELINE configs[0] (the reference's own CPU-runnable case): the render-only chain on 4096 rays.  Not the
    bench line of the metric; prints its own JSON line with the GPU chain and the CPU oracle timed side by side."""
    from oracle import nerf_oracle as orc
    from ctxnerf import ops, run_nerf_helpers as rh
    dev = torch.device("cuda", 0)
    R, S, Ni = 4096, 64, 128
    raw, z, d = orc.cfg1_inputs(R, S)
    raw_f = orc.cfg1_inputs(R, S + Ni, seed=1)[0]
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        ref = orc.cfg1_chain(raw, z, d, raw_f, Ni)
    cpu_s = (time.perf_counter() - t0) / reps
    rc, zc, dc, rfc = raw.to(dev), z.to(dev), d.to(dev), raw_f.to(dev)

    def chain():
        c = rh.raw2outputs(rc, zc, dc)
        zs, z_all = ops.resample_merge(zc, c[3], Ni, det=True)
        return c, zs, z_all, rh.raw2outputs(rfc, z_all, dc)

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            out = chain()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            out = chain()
        b.record()
        torch.cuda.synchronize()
    ms = a.elapsed_time(b) / args.steps
    # parity stage by stage on the oracle's own intermediates (end to end the synthetic raw_fine is indexed by sample
    # rank, so a one-ulp difference in a weight that reorders two depths would swap unrelated colours)
    with torch.no_grad():
        zs_g, zall_g = ops.resample_merge(zc, ref[0][3].to(dev), Ni, det=True)
        fine_g = rh.raw2outputs(rfc, ref[2].to(dev), dc)
    same_idx = bool(torch.equal(zall_g.cpu(), ref[2]) and torch.equal(zs_g.cpu(), ref[1]))

    def rel(a, b):
        return ((a.cpu() - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()
    err = max(rel(out[0][0], ref[0][0]), rel(out[0][3], ref[0][3]), rel(fine_g[0], ref[3][0]), rel(fine_g[3], ref[3][3]),
              rel(fine_g[4], ref[3][4]))
    print(json.dumps({"metric": "rays/sec render-only chain (raw2outputs 64 -> sample_pdf det 128 -> merge -> raw2outputs 192)",
                      "value": R / (ms * 1e-3), "unit": "rays/s", "n_gpus": 1, "steps": args.steps, "ms_per_step": ms,
                      "config": {"workload": "configs[0]: 4096 rays x 64 coarse + 128 fine, synthetic raw"},
                      "resample_bit_exact_on_oracle_weights": same_idx, "max_rel_err_composite": err,
                      "cpu_baseline": {"value": R / cpu_s, "unit": "rays/s", "cores": os.cpu_count(), "kind": "port",
                                       "sample": f"the same chain x{reps}, oracle/nerf_oracle.py"}}), flush=True)


def run_inference_cfg(args, which, rank, world, local):
    """BASELINE configs[1] (--cfg2: 800x800 coarse+fine render, row blocks per rank) and configs[3] (--cfg4: 8 views at
    1024x1024 x 192 samples, one view per rank) under torchrun: device time of the sharded render (max over ranks) and
    of the gather to rank 0, plus a bit-equality check of a gathered map against the same render done by rank 0."""
    import torch.distributed as dist
    from ctxnerf.dist import render_image_sharded, render_views_sharded
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import multiview_cameras, orbit_camera
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    K, c2w = orbit_camera()
    tr = NerfTrainer(800, 800, K, c2w, near=2.0, far=6.0, perturb=0.0, white_bkgd=True, device=dev, seed=0)
    cams, sphere = multiview_cameras(8, 1024)
    if which == "cfg2":
        work = lambda gather: render_image_sharded(tr, gather=gather)
        n_rays, evals = 800 * 800, EVALS_PER_RAY
    else:
        work = lambda gather: render_views_sharded(tr, cams, 1024, 1024, 192, sphere, gather=gather)
        n_rays, evals = 8 * 1024 * 1024, 192

    def timed(gather):
        for _ in range(max(args.warmup, 1)):
            work(gather)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            out = work(gather)
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b) / args.steps], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), out
    ms_render, _ = timed(False)
    ms_total, out = timed(True)
    same = None
    if rank == 0:
        if which == "cfg2":
            ref = tr.render(None)["rgb_map"].reshape(800, 800, 3)
            same = bool(torch.equal(out["rgb_map"], ref))
        else:
            v = min(world, 8) - 1          # a view another rank rendered (the last one of the first round)
            ref = tr.render_view(1024, 1024, cams[v][0], cams[v][1], n_samples=192, sphere=sphere)["rgb_map"]
            same = bool(torch.equal(out[v]["rgb_map"], ref))
        pk = peaks()
        tf = 2.0 * MACS_PER_EVAL * n_rays * evals / (ms_render * 1e-3) / 1e12
        print(json.dumps({
            "metric": "rays/sec inference render", "value": n_rays / (ms_total * 1e-3), "unit": "rays/s", "n_gpus": world,
            "steps": args.steps, "ms_render": ms_render, "ms_with_gather": ms_total, "scaling": "strong",
            "config": {"workload": ("configs[1]: 800x800 single view, coarse 64 + fine 128, image row blocks per rank"
                                    if which == "cfg2" else
                                    "configs[3]: 8 views 1024x1024 x 192 samples of the napoleon.obj bounding sphere, "
                                    "one view per rank (round-robin)"), "gather": "maps gathered to rank 0 (NCCL gather)"},
            "tensor_tflops_all_gpus": tf, "tensor_frac_per_gpu": tf / world / pk["tf_sustained"],
            "gathered_equals_single_gpu_render": same, "dtype": "bf16", "data": "synthetic"}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sustained", action="store_true", help="skip the extra 200-step (power-capped) pass")
    ap.add_argument("--ref-rays", type=int, default=0,
                    help="rays per step of the CPU legs (--impl reference / cpu_baseline); default: the full 4096-ray batch")
    ap.add_argument("--cfg1", action="store_true",
                    help="BASELINE configs[0] instead of the training step: raw2outputs(64) -> sample_pdf(det, 128) -> "
                         "merge -> raw2outputs(192) on 4096 rays, GPU chain beside the CPU oracle (parity-test sized)")
    ap.add_argument("--cfg2", action="store_true", help="BASELINE configs[1]: 800x800 inference render, rows sharded over the ranks")
    ap.add_argument("--cfg4", action="store_true", help="BASELINE configs[3]: 8 views 1024^2 x 192 samples, views sharded over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="training step only: after the timed steps, rank 0 writes what the last of them computed as "
                         "DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.cfg1 or args.cfg2 or args.cfg4):
        ap.error("--dump-outputs applies to the training-step benchmark only")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.cfg1:
        if rank == 0:
            run_cfg1(args)
        return
    if args.cfg2 or args.cfg4:
        run_inference_cfg(args, "cfg2" if args.cfg2 else "cfg4", rank, world, local)
        return

    import torch.distributed as dist
    from ctxnerf import _lib
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: ctxnerf has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    warm = max(args.warmup, 3)
    K, c2w = orbit_camera()
    # NerfTrainer draws the Philox seed of the jitter and importance uniforms from torch's global generator, whose
    # start-up seed differs from process to process (torch 2.11): seed it (0 + rank, like the ray selection) so
    # that every run draws the same samples
    torch.manual_seed(rank)
    tr = NerfTrainer(800, 800, K, c2w, near=2.0, far=6.0, N_samples=N_SAMPLES, N_importance=N_IMPORTANCE,
                     perturb=1.0, white_bkgd=True, device=dev, seed=0)
    # per-rank synthetic batches (seed 0 + rank), resident on the device and mirrored in pinned host memory
    from ctxnerf.dist import rank_generator
    g = rank_generator(0, rank)              # SURVEY.md 8e: the seed + rank stream of this rank's ray selection
    NB = 8
    idx_h = [torch.randint(0, 800 * 800, (RAYS_PER_GPU,), generator=g).pin_memory() for _ in range(NB)]
    tgt_h = [torch.rand(RAYS_PER_GPU, 3, generator=g).pin_memory() for _ in range(NB)]
    idx_d = [t.to(dev) for t in idx_h]
    tgt_d = [t.to(dev) for t in tgt_h]
    loss_h = torch.zeros(1).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()

    def timed(step_fn, steps, with_timers, after=None):
        cs = ClockSampler(local)
        cs.start()
        for i in range(warm):
            step_fn(i)
        if after is not None:
            after()
        torch.cuda.synchronize()
        t_idle = time.time()
        cs.wait_first_sample()
        # A fixed pause between the warm-up and the timed region.  The wait for the clock sampler's first line used to
        # make this pause random (0 - 1 s), and under the board's power limiter that moved the 20-step figure by 4 %
        # (tools/first_pass_probe.py: a pass that starts right behind other work runs 4.3 - 4.6 ms per step, one that
        # starts after >= 0.5 s of idle 4.15 - 4.26 ms).  The figure with the limiter engaged is reported as `sustained`.
        time.sleep(max(0.0, SETTLE_S - (time.time() - t_idle)))
        barrier()
        tr.timers = {} if with_timers else None
        l0 = _lib.launch_count
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        cs.mark()
        a.record()
        for i in range(steps):
            step_fn(warm + i)
        if after is not None:
            after()          # the last step's loss is read inside the timed region too
        b.record()
        torch.cuda.synchronize()
        clocks = cs.stop()
        barrier()
        ms = a.elapsed_time(b)
        launches = _lib.launch_count - l0
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        timers, tr.timers = tr.timers, None
        return t.item(), clocks, launches, timers

    # ---- device-resident inputs ("value"): the captured step, no per-kernel timers ----
    ms, clocks, launches, _ = timed(lambda i: tr.step(idx_d[i % NB], tgt_d[i % NB]), args.steps, False)
    if args.dump_outputs and rank == 0:       # before the passes below train the networks further
        dump_step_outputs(args.dump_outputs, tr)
    value = RAYS_PER_GPU * world * args.steps / (ms * 1e-3)
    # ---- end to end through the public API with host buffers ----
    # Every step copies its ray ids + targets from pinned host memory and its loss is read on the host; the host
    # reads the loss of step i after it has submitted step i+1 (two pinned loss slots), as a training loop that logs
    # the loss does, so the submission of the next step is not exposed between steps.
    loss_slots = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]
    pending = []
    host_losses = []

    def e2e_step(i):
        ev = tr.step_from_host(idx_h[i % NB], tgt_h[i % NB], loss_slots[i & 1])
        if pending:
            pev, slot = pending.pop()
            pev.synchronize()
            host_losses.append(float(slot.item()))
        pending.append((ev, loss_slots[i & 1]))

    def e2e_drain():
        while pending:
            pev, slot = pending.pop()
            pev.synchronize()
            host_losses.append(float(slot.item()))

    ms_e2e, _, _, _ = timed(e2e_step, args.steps, False, after=e2e_drain)
    e2e = RAYS_PER_GPU * world * args.steps / (ms_e2e * 1e-3)
    final_loss = host_losses[-1]
    loss_h.fill_(final_loss)

    # ---- per-kernel device times -> roofline (two short extra passes, eager launches with event pairs) ----
    # (1) the schedule of the timed region, with CUDA events around each MLP kernel and around the concurrent backward
    # group; (2) overlap off: every kernel alone on the whole GPU ("kernels").
    pk = peaks()
    n_extra = min(args.steps, 6)
    _, _, _, timers_live = timed(lambda i: tr.step(idx_d[i % NB], tgt_d[i % NB]), n_extra, True)
    group_ms = None
    if timers_live and "bwd_overlap_group" in timers_live:
        evs = timers_live["bwd_overlap_group"]
        group_ms = sum(x.elapsed_time(y) for x, y in evs) / len(evs)
    overlap_was = tr.overlap_backward
    tr.overlap_backward = False
    _, _, _, timers_iso = timed(lambda i: tr.step(idx_d[i % NB], tgt_d[i % NB]), n_extra, True)
    tr.overlap_backward = overlap_was
    kern = {}
    for name, evs in (timers_iso or {}).items():
        kern[name] = sum(x.elapsed_time(y) for x, y in evs) / len(evs)
    pts = {"coarse": RAYS_PER_GPU * N_SAMPLES, "fine": RAYS_PER_GPU * (N_SAMPLES + N_IMPORTANCE)}
    # HBM traffic the design generates per evaluated point (DESIGN.md section 3) -- NOT algorithmic bytes: bf16
    # activation records of the 8 pts layers and the views layer (the linear feature layer keeps none), 1-bit ReLU
    # masks, the two encodings; dgrad writes the dZ records of the same layers + g_out and reads the masks back; wgrad
    # streams sum over its 12 jobs of (A + B channels) x 2 B.
    REC_BYTES_PER_POINT = {"fwd": 2176 * 2 + 272 + 128 + 64 + 16 + 4, "dgrad": 2192 * 2 + 272 + 16,
                           "wgrad": 9856.0}
    # algorithmic I/O of one MLP pass per point (SURVEY.md 8d): z in, raw out (+ g_raw in for the backward kernels);
    # the 2 x 1.2 MB weight streams / 2 x 2.4 MB gradients per launch are added per launch below
    ALG_BYTES_PER_POINT = {"fwd": 4 + 16, "dgrad": 16, "wgrad": 0}
    ALG_BYTES_PER_LAUNCH = {"fwd": 1.2e6, "dgrad": 1.2e6, "wgrad": 2.4e6}
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            traffic = json.load(fh)
    except Exception:
        pass
    kernels = {}
    for name, t_ms in kern.items():
        _, kind, net = name.split("_")
        n = pts[net]
        # SURVEY.md 8d: the MLP is the only dense contraction -> tensor roofline with the algorithmic FLOPs
        # (593 408 MAC per point per pass; fwd, dgrad and wgrad are one pass each of the 3x rule)
        tf = 2.0 * MACS_PER_EVAL * n / (t_ms * 1e-3) / 1e12
        gb = REC_BYTES_PER_POINT[kind] * n / (t_ms * 1e-3) / 1e9
        alg = ALG_BYTES_PER_POINT[kind] * n + ALG_BYTES_PER_LAUNCH[kind]
        kernels[name] = {"bound": "tensor", "achieved": tf, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                         "frac": tf / pk["tf_sustained"], "ms_per_launch": t_ms,
                         "traffic": traffic.get(name), "design_traffic_bytes": REC_BYTES_PER_POINT[kind] * n,
                         "algorithmic_bytes": alg, "traffic_over_algorithmic": REC_BYTES_PER_POINT[kind] * n / alg,
                         "hbm_gbs": gb, "hbm_frac": gb / pk["hbm_gbs"]}
    roofline = None
    dom = max(kern, key=kern.get) if kern else None
    if dom:
        roofline = dict(kernels[dom], kernel=dom + " (timed alone, overlap off; the dominant kernel of the step)",
                        peak_source=pk["source"] + " cuBLAS bf16, sustained")
        if group_ms is not None:
            gbytes = (REC_BYTES_PER_POINT["wgrad"] * pts["fine"]
                      + (REC_BYTES_PER_POINT["dgrad"] + REC_BYTES_PER_POINT["wgrad"]) * pts["coarse"])
            gflops = 2.0 * MACS_PER_EVAL * (pts["fine"] + 2 * pts["coarse"])
            roofline["concurrent_group"] = {
                "what": "mlp_wgrad_fine || (mlp_dgrad_coarse -> mlp_wgrad_coarse), disjoint SM budgets, one span on the "
                        "main stream, measured live in the schedule of the timed region",
                "ms": group_ms, "tensor_tflops": gflops / (group_ms * 1e-3) / 1e12,
                "tensor_frac": gflops / (group_ms * 1e-3) / 1e12 / pk["tf_sustained"],
                "hbm_gbs": gbytes / (group_ms * 1e-3) / 1e9, "hbm_frac": gbytes / (group_ms * 1e-3) / 1e9 / pk["hbm_gbs"]}
    # (last: it heats the board)
    # ---- the same loop held for 200 steps: the step draws ~1 kW, so after ~50 steps the board's power cap pulls the SM
    # clock from 1.96 to ~1.6 GHz (profiles/README.md r02); reported beside the 20-step figure, not instead of it ----
    sustained = None
    if not args.no_sustained:
        ms_s, clocks_s, _, _ = timed(lambda i: tr.step(idx_d[i % NB], tgt_d[i % NB]), 200, False)
        sustained = {"steps": 200, "ms_per_step": ms_s / 200, "value": RAYS_PER_GPU * world * 200 / (ms_s * 1e-3),
                     "unit": "rays/s", "clocks": clocks_s}
    step_flops = 3 * 2.0 * MACS_PER_EVAL * RAYS_PER_GPU * EVALS_PER_RAY
    line = {"metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": CONFIG, "clocks": clocks,
            "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": RAYS_PER_GPU * (8 + 12),
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                    "host_loop": "NerfTrainer.step_from_host per step (pinned ray ids + targets in, loss out); the host "
                                 "reads step i's loss after submitting step i+1, the last one inside the timed region"},
            "gpu_launches": launches, "roofline": roofline,
            "step_tensor_frac": step_flops / (ms / args.steps * 1e-3) / 1e12 / pk["tf_sustained"],
            "step_hbm_frac": (REC_BYTES_PER_POINT["fwd"] + REC_BYTES_PER_POINT["dgrad"] + REC_BYTES_PER_POINT["wgrad"])
            * RAYS_PER_GPU * EVALS_PER_RAY / (ms / args.steps * 1e-3) / 1e9 / pk["hbm_gbs"],
            "kernels": kernels, "final_loss": final_loss, "sustained": sustained}
    if world > 1:
        line["allreduce"] = {"route": ("ctx_allreduce (libctxnerf NCCL binding, inside the step graph"
                                       + (", fine half beside the coarse backward chain)" if tr.split_reduce else ")"))
                             if tr.comm is not None
                             else "torch.distributed between two graphs",
                             "nccl_version": tr.comm.version if tr.comm is not None else None,
                             "bytes": 4 * tr.bucket.numel}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            n = args.ref_rays or RAYS_PER_GPU
            times = cpu_step_sample(n, threads, 3, 1)
            line["cpu_baseline"] = {"value": n * len(times) / sum(times), "unit": "rays/s", "cores": threads,
                                    "kind": "port",
                                    "sample": f"{n}-ray coarse+fine fwd+bwd step x{len(times)}, oracle/nerf_oracle.py "
                                              "(torch CPU fp32, all host threads)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
