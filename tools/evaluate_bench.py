"""Cost of NerfTrainer.evaluate and of its metric kernel, measured on the GPU.

    python tools/evaluate_bench.py [--reps 6] [--launches 10]

1. A Blender-sized trainer (800 x 800, 64+128 samples, random weights) and 25 test poses on the orbit, upstream's
   Blender test split at testskip=8, with random fp32 targets on the device: `evaluate` per view against a bare
   `render(c2w=)` per view, in alternating passes over the 25 poses (host clock around work that ends in a device
   synchronise; median pass reported).
2. ctx_image_metrics alone (MSE and SSIM) on 200 x 800 x 800 images with fp32 and with uint8 targets, CUDA events over
   `launches` calls, as a fraction of the copy bandwidth measured in the same run (a 2 GiB device-to-device copy).
   The inputs (1.5 GB of predictions and 1.5 GB / 384 MB of targets) are larger than the L2, so they come from HBM.

The GPU's name and power limit are printed with the numbers: they are part of them.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "contexture-nerf_b200"), os.path.join(ROOT, "tools")]

import torch  # noqa: E402

from forward_facing_bench import event_ms, gpu_info  # noqa: E402


def bench_evaluate(dev, args):
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera
    H = W = 800
    N = 25
    cams = [orbit_camera(H, W, azim_deg=360.0 * v / N) for v in range(N)]
    poses = torch.stack([c for _, c in cams]).to(dev)
    images = torch.rand(N, H, W, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    torch.manual_seed(0)
    tr = NerfTrainer(H, W, cams[0][0], poses[0], near=2.0, far=6.0, N_samples=64, N_importance=128, device=dev)

    def render_all():
        for v in range(N):
            tr.render(c2w=poses[v])

    fns = {"evaluate": lambda: tr.evaluate(poses, images), "render": render_all}
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for rep in range(args.reps):
        order = list(fns) if rep % 2 == 0 else list(fns)[::-1]
        for k in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fns[k]()
            torch.cuda.synchronize()
            times[k].append(1e3 * (time.perf_counter() - t0) / N)
    med = {k: statistics.median(v) for k, v in times.items()}
    res = tr.evaluate(poses, images)
    return {"views": N, "H": H, "W": W, "samples": "64+128",
            "ms_per_view_median": {k: round(v, 3) for k, v in med.items()},
            "ms_per_view_passes": {k: [round(x, 3) for x in v] for k, v in times.items()},
            "evaluate_over_render": round(med["evaluate"] / med["render"], 4),
            "psnr_mean_random_targets": round(float(res["psnr"].mean()), 3)}


def bench_kernel(dev, args):
    from ctxnerf import _lib
    from ctxnerf._lib import call, ptr, stream_ptr
    B, H, W = 200, 800, 800
    g = torch.Generator(device=dev).manual_seed(1)
    pred = torch.rand(B, H, W, 3, device=dev, generator=g)
    t32 = torch.rand(B, H, W, 3, device=dev, generator=g)
    t8 = torch.randint(0, 256, (B, H, W, 3), device=dev, dtype=torch.uint8, generator=g)
    mse, ssim = (torch.empty(B, device=dev, dtype=torch.float64) for _ in range(2))
    part = torch.empty(int(_lib.lib().ctx_image_metrics_partials(B, H, W)), device=dev, dtype=torch.float64)
    st = stream_ptr(dev)

    def metrics(t, u8):
        return lambda: call("ctx_image_metrics", ptr(pred), ptr(t), u8, B, H, W, ptr(mse), ptr(ssim), ptr(part), st)

    src = torch.empty(1 << 29, device=dev)            # 2 GiB copied -> 4 GiB moved per pass
    dst = torch.empty_like(src)
    fns = {"copy": lambda: dst.copy_(src), "fp32_target": metrics(t32, 0), "uint8_target": metrics(t8, 1)}
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for rep in range(args.reps):
        order = list(fns) if rep % 2 == 0 else list(fns)[::-1]
        for k in order:
            times[k].append(event_ms(fns[k], args.launches))
    med = {k: statistics.median(v) for k, v in times.items()}
    copy_bw = 2 * src.numel() * 4 / (med["copy"] * 1e-3)
    out = {"images": B, "H": H, "W": W, "copy_GBps": round(copy_bw / 1e9, 1)}
    for k, tb in (("fp32_target", 4), ("uint8_target", 1)):
        bytes_ = B * H * W * 3 * (4 + tb)
        out[k] = {"ms_median": round(med[k], 4), "ms_passes": [round(x, 4) for x in times[k]],
                  "us_per_image": round(1e3 * med[k] / B, 2), "GBps": round(bytes_ / (med[k] * 1e-3) / 1e9, 1),
                  "fraction_of_copy_bw": round(bytes_ / (med[k] * 1e-3) / copy_bw, 3)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=6, help="timed passes of each variant (alternating)")
    ap.add_argument("--launches", type=int, default=10, help="ctx_image_metrics calls per timed pass")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("evaluate_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = gpu_info(dev)
    result["evaluate"] = bench_evaluate(dev, args)
    torch.cuda.empty_cache()
    result["ctx_image_metrics"] = bench_kernel(dev, args)
    print(json.dumps(result, indent=1), flush=True)


if __name__ == "__main__":
    main()
