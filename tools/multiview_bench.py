"""Cost of multi-view training in NerfTrainer, measured with CUDA events.

    python tools/multiview_bench.py [--steps 20] [--reps 6] [--rays 4096]

1. Two upstream recipes at 4096 rays, each timed as three variants in alternating passes of `steps` captured steps
   (median pass reported):
   * Blender-like: 100 views of 800 x 800, 64+128 samples, no_batching=True with a centre crop (precrop_iters 500).
   * LLFF-like: 20 views of 378 x 504, ndc + raw_noise_std=1 + lrate_decay=250, 64+64 samples, no_batching=False.
   Variants: `one_pose_step` (a trainer of the first pose alone, step() on a fixed device batch of pixel ids: the step
   before multi-view training existed), `stack_step` (the multi-view trainer, step() on a fixed device batch of global
   ids: ctx_raygen_views with a per-lane pose load), `step_random` (the same trainer drawing its batch and gathering
   its targets inside the step: ctx_draw_rays + the stack step).
2. ctx_draw_rays alone with targets from the 100 x 800 x 800 image stack: mode 0 at 4096 rays, mode 1 at 4096 and
   2^20 rays, alternating passes of CUDA graphs of 200 launches each.

The GPU's name and power limit are printed with the numbers: they are part of them.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "contexture-nerf_b200"), os.path.join(ROOT, "tools")]

import torch  # noqa: E402

from forward_facing_bench import event_ms, gpu_info  # noqa: E402


def _poses(recipe, n):
    from ctxnerf.workloads import forward_facing_camera, orbit_camera
    if recipe == "blender":
        cams = [orbit_camera(800, 800, azim_deg=360.0 * v / n) for v in range(n)]
    else:
        cams = [forward_facing_camera(378, 504, 407.0, yaw=0.08 - 0.008 * v, eye=(0.01 * v, -0.03, 0.1))
                for v in range(n)]
    return cams[0][0], torch.stack([c for _, c in cams])


RECIPES = {
    "blender_100x800x800_64+128": dict(recipe="blender", n=100, H=800, W=800,
                                       kw=dict(near=2.0, far=6.0, N_samples=64, N_importance=128, perturb=1.0,
                                               white_bkgd=True, no_batching=True, precrop_iters=500,
                                               precrop_frac=0.5)),
    "llff_20x378x504_64+64": dict(recipe="llff", n=20, H=378, W=504,
                                  kw=dict(near=0.0, far=1.0, N_samples=64, N_importance=64, perturb=1.0,
                                          white_bkgd=False, ndc=True, raw_noise_std=1.0, lrate_decay=250,
                                          no_batching=False)),
}


def bench_recipes(dev, args):
    from ctxnerf.train import NerfTrainer
    res = {}
    for name, rc in RECIPES.items():
        n, H, W, R = rc["n"], rc["H"], rc["W"], args.rays
        K, poses = _poses(rc["recipe"], n)
        g = torch.Generator(device=dev).manual_seed(0)
        images = torch.rand(n, H, W, 3, device=dev, generator=g)
        one_kw = {k: v for k, v in rc["kw"].items() if k not in ("no_batching", "precrop_iters", "precrop_frac")}
        torch.manual_seed(0)
        one = NerfTrainer(H, W, K, poses[0], device=dev, **one_kw)
        torch.manual_seed(0)
        stack = NerfTrainer(H, W, K, poses, images=images, device=dev, **rc["kw"])
        NB = 8
        pix = [torch.randint(0, H * W, (R,), device=dev, generator=g) for _ in range(NB)]
        ids = [torch.randint(0, n * H * W, (R,), device=dev, generator=g) for _ in range(NB)]
        tgt = [torch.rand(R, 3, device=dev, generator=g) for _ in range(NB)]
        it = [0]

        def nxt():
            it[0] += 1
            return it[0] % NB

        fns = {"one_pose_step": lambda: one.step(pix[nxt()], tgt[it[0] % NB]),
               "stack_step": lambda: stack.step(ids[nxt()], tgt[it[0] % NB]),
               "step_random": lambda: stack.step_random(R)}
        for fn in fns.values():                  # eager first step, capture, a few replays
            for _ in range(5):
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in fns}
        for rep in range(args.reps):
            order = list(fns) if rep % 2 == 0 else list(fns)[::-1]
            for k in order:
                times[k].append(event_ms(fns[k], args.steps))
        med = {k: statistics.median(v) for k, v in times.items()}
        res[name] = {"rays": R, "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
                     "ms_per_step_passes": {k: [round(x, 4) for x in v] for k, v in times.items()},
                     "stack_step_over_one_pose": round(med["stack_step"] / med["one_pose_step"], 4),
                     "step_random_over_stack_step": round(med["step_random"] / med["stack_step"], 4)}
        del one, stack, images
        torch.cuda.empty_cache()
    return res


def bench_draw(dev, args):
    from ctxnerf import ops
    n, H, W = 100, 800, 800
    images = torch.rand(n, H, W, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    ctr = torch.tensor([2, 1000], dtype=torch.int64, device=dev)
    cases = {"mode0_4096": (0, 4096), "mode1_4096": (1, 4096), "mode1_2^20": (1, 1 << 20)}
    outs = {k: (torch.empty(R, dtype=torch.int64, device=dev), torch.empty(R, 3, device=dev))
            for k, (_, R) in cases.items()}

    LAUNCHES = 200
    graphs = {}
    for k, (mode, R) in cases.items():          # 200 launches per graph: the host's launch rate stays out of it
        draw = lambda: ops.draw_rays(n, H, W, R, ctr, images=images, mode=mode, seed=12345, out=outs[k])
        draw()
        torch.cuda.synchronize()
        graphs[k] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graphs[k]):
            for _ in range(LAUNCHES):
                draw()
        graphs[k].replay()
    torch.cuda.synchronize()
    times = {k: [] for k in cases}
    for rep in range(args.reps):
        order = list(cases) if rep % 2 == 0 else list(cases)[::-1]
        for k in order:
            times[k].append(event_ms(graphs[k].replay, 5) / LAUNCHES)
    return {k: {"us_per_launch_median": round(1e3 * statistics.median(v), 2),
                "us_per_launch_passes": [round(1e3 * x, 2) for x in v]} for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20, help="captured steps per timed pass")
    ap.add_argument("--reps", type=int, default=6, help="timed passes of each variant (alternating)")
    ap.add_argument("--rays", type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multiview_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = gpu_info(dev)
    result["train_step"] = bench_recipes(dev, args)
    result["ctx_draw_rays"] = bench_draw(dev, args)
    print(json.dumps(result, indent=1), flush=True)


if __name__ == "__main__":
    main()
