"""Cost of upstream's forward-facing (LLFF) recipe in the training step, measured with CUDA events.

    python tools/forward_facing_bench.py [--steps 20] [--reps 6] [--rays 4096]

1. NerfTrainer.step, the default step against the same step with ndc=True, raw_noise_std=1, lrate_decay=250, at
   4096 rays for 64+128 (this project's benchmark) and 64+64 samples (upstream's LLFF config).  Both trainers are
   built once and timed in alternating passes of `steps` captured steps; the median pass is reported.
2. The fused compositing pass alone at 2^20 rays x 192 samples: ctx_composite_train (no noise) against
   ctx_composite_train_noise (noise drawn in-kernel), alternating, as a fraction of the copy bandwidth measured in
   the same run (both move 40 S + 36 bytes per ray, 8 GB per pass: far beyond L2).

The GPU's name and power limit are printed with the numbers: they are part of them.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "contexture-nerf_b200")]

import torch  # noqa: E402


def gpu_info(dev):
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev.index), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(",")]
    except Exception as e:          # the numbers are still printed, marked as lacking the limit
        info["power_limit"] = f"unknown ({e})"
    return info


def event_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def bench_steps(dev, args):
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import forward_facing_camera
    K, c2w = forward_facing_camera()
    H, W = 756, 1008
    g = torch.Generator().manual_seed(0)
    NB = 8
    idx = [torch.randint(0, H * W, (args.rays,), generator=g).to(dev) for _ in range(NB)]
    tgt = [torch.rand(args.rays, 3, generator=g).to(dev) for _ in range(NB)]
    res = {}
    for S, Ni in ((64, 128), (64, 64)):
        torch.manual_seed(0)
        trs = {"default": NerfTrainer(H, W, K, c2w, near=2.0, far=6.0, N_samples=S, N_importance=Ni, perturb=1.0,
                                      white_bkgd=True, device=dev),
               "ndc+noise+decay": NerfTrainer(H, W, K, c2w, near=0.0, far=1.0, N_samples=S, N_importance=Ni,
                                              perturb=1.0, white_bkgd=False, ndc=True, raw_noise_std=1.0,
                                              lrate_decay=250, device=dev)}
        it = {k: 0 for k in trs}

        def run(name):
            tr = trs[name]
            i = it[name]
            it[name] += 1
            tr.step(idx[i % NB], tgt[i % NB])

        for name in trs:                      # eager first step, capture, a few replays
            for _ in range(5):
                run(name)
        torch.cuda.synchronize()
        times = {k: [] for k in trs}
        for rep in range(args.reps):
            order = list(trs) if rep % 2 == 0 else list(trs)[::-1]
            for name in order:
                times[name].append(event_ms(lambda: run(name), args.steps))
        med = {k: statistics.median(v) for k, v in times.items()}
        res[f"{S}+{Ni}"] = {"ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
                            "ms_per_step_passes": {k: [round(x, 4) for x in v] for k, v in times.items()},
                            "options_over_default": round(med["ndc+noise+decay"] / med["default"], 4)}
        del trs
        torch.cuda.empty_cache()
    return res


def bench_composite(dev, args):
    from ctxnerf._lib import call, ptr, stream_ptr
    R, S = 1 << 20, 192
    g = torch.Generator(device=dev).manual_seed(0)
    raw = torch.randn(R * S, 4, device=dev, generator=g)
    z = torch.sort(torch.rand(R, S, device=dev, generator=g) * 4 + 2, -1)[0]
    d = torch.randn(R, 3, device=dev, generator=g)
    tgt = torch.rand(R, 3, device=dev, generator=g)
    loss, g_raw = torch.zeros(1, device=dev), torch.empty(R * S, 4, device=dev)
    w, rgb = torch.empty(R, S, device=dev), torch.empty(R, 3, device=dev)
    ctr = torch.zeros(2, dtype=torch.int64, device=dev)
    st = stream_ptr(dev)

    def plain():
        call("ctx_composite_train", ptr(raw), ptr(z), ptr(d), None, R, S, 0, ptr(tgt), 1.0 / (3 * R), ptr(loss),
             ptr(g_raw), ptr(w), ptr(rgb), st)

    def noisy():
        call("ctx_composite_train_noise", ptr(raw), ptr(z), ptr(d), R, S, 0, ptr(tgt), 1.0 / (3 * R), ptr(loss),
             ptr(g_raw), ptr(w), ptr(rgb), 1.0, 12345, ptr(ctr), 2, st)

    src = torch.empty(1 << 29, device=dev)            # 2 GiB copied -> 4 GiB moved per pass
    dst = torch.empty_like(src)
    copy = lambda: dst.copy_(src)
    fns = {"copy": copy, "ctx_composite_train": plain, "ctx_composite_train_noise": noisy}
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for rep in range(args.reps):
        order = list(fns) if rep % 2 == 0 else list(fns)[::-1]
        for k in order:
            times[k].append(event_ms(fns[k], 10))
    med = {k: statistics.median(v) for k, v in times.items()}
    copy_bw = 2 * src.numel() * 4 / (med["copy"] * 1e-3)
    bytes_ = R * (40 * S + 36)
    out = {"rays": R, "samples": S, "copy_GBps": round(copy_bw / 1e9, 1)}
    for k in ("ctx_composite_train", "ctx_composite_train_noise"):
        out[k] = {"ms_median": round(med[k], 4), "ms_passes": [round(x, 4) for x in times[k]],
                  "fraction_of_copy_bw": round(bytes_ / (med[k] * 1e-3) / copy_bw, 3)}
    out["noise_over_plain"] = round(med["ctx_composite_train_noise"] / med["ctx_composite_train"], 4)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20, help="captured steps per timed pass")
    ap.add_argument("--reps", type=int, default=6, help="timed passes of each variant (alternating)")
    ap.add_argument("--rays", type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("forward_facing_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = gpu_info(dev)
    result["train_step"] = bench_steps(dev, args)
    result["composite_2^20x192"] = bench_composite(dev, args)
    print(json.dumps(result, indent=1), flush=True)


if __name__ == "__main__":
    main()
