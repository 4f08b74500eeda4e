"""Cost of mesh extraction, measured on the GPU.

    python tools/mesh_bench.py [--reps 4]

1. `density_grid` (the fine network's relu(sigma) on the lattice, zero view directions) at 256^3 and 512^3 cells over
   [-1.2, 1.2]^3, against the measured sustained tensor roof of DESIGN §4 (1412.2 TFLOP/s) with 593 408 MAC per point
   (the whole view-direction network: the view head is computed and discarded).  In the same alternating passes,
   `render(c2w=)` of an 800^2 view with 64+128 samples, so that the two MLP efficiencies compare directly.
2. ctx_marching_cubes alone (pass 0 + pass 1, outputs preallocated) on a 512^3-cell field (0.54 GB of sigma: more than
   the L2) holding a rippled sphere, CUDA events over `launches` calls, against the copy bandwidth measured in the same
   run (a 2 GiB device-to-device copy).  The bytes counted are the least the job needs: sigma read once and the mesh
   (vertices, normals, faces) written once.
3. `extract_mesh` end to end at 256^3 (lattice, marching cubes with its one host synchronisation, vertex colours).

Random weights: the density of an untrained network is small, so the end-to-end mesh uses a threshold at the median
positive density instead of upstream's 50.  The GPU's name and power limit are printed with the numbers.
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

MAC_PER_POINT = 593408
ROOF = 1412.2e12          # measured sustained bf16 tensor rate, DESIGN §4


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def alternate(fns, reps):
    for fn in fns.values():
        fn()
    times = {k: [] for k in fns}
    for rep in range(reps):
        for k in (list(fns) if rep % 2 == 0 else list(fns)[::-1]):
            times[k].append(host_ms(fns[k]))
    return times


def bench_lattice(dev, args):
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera
    K, c2w = orbit_camera(800, 800)
    torch.manual_seed(0)
    tr = NerfTrainer(800, 800, K, c2w, N_samples=64, N_importance=128, device=dev)
    fns = {"density_grid_256": lambda: tr.density_grid(256), "density_grid_512": lambda: tr.density_grid(512),
           "render_800": lambda: tr.render(c2w=c2w)}
    times = alternate(fns, args.reps)
    out = {}
    for k, v in times.items():
        med = statistics.median(v)
        if k.startswith("density"):
            n = int(k.rsplit("_", 1)[1]) + 1
            flop = 2.0 * MAC_PER_POINT * n ** 3
        else:
            flop = 2.0 * MAC_PER_POINT * 800 * 800 * (64 + 192)
        out[k] = {"ms_median": round(med, 3), "ms_passes": [round(x, 3) for x in v],
                  "TFLOPs": round(flop / (med * 1e-3) / 1e12, 1), "fraction_of_tensor_roof": round(
                      flop / (med * 1e-3) / ROOF, 3)}
    sigma = tr.density_grid(256)
    pos = sigma[sigma > 0]
    thr = float(pos.median()) if pos.numel() else 1.0
    m = tr.extract_mesh(256, threshold=thr)
    e2e = [host_ms(lambda: tr.extract_mesh(256, threshold=thr)) for _ in range(args.reps)]
    out["extract_mesh_256"] = {"threshold": round(thr, 4), "vertices": int(m["vertices"].shape[0]),
                               "faces": int(m["faces"].shape[0]), "ms_median": round(statistics.median(e2e), 3),
                               "ms_passes": [round(x, 3) for x in e2e]}
    return out


def bench_mcubes(dev, args):
    from ctxnerf import _lib, mesh
    from ctxnerf._lib import call, ptr, stream_ptr
    n, B = 512, mesh.DEFAULT_BOUNDS
    ax = torch.linspace(-1.2, 1.2, n + 1, device=dev)
    X, Y, Z = ax[:, None, None], ax[None, :, None], ax[None, None, :]
    sigma = (1.0 - torch.sqrt(X * X + Y * Y + Z * Z) + 0.05 * torch.sin(12 * X) * torch.sin(12 * Y)
             * torch.sin(12 * Z)).contiguous()
    ref = mesh.marching_cubes(sigma, 0.0, B)
    V, F = ref["vertices"].shape[0], ref["faces"].shape[0]
    o, h = mesh.lattice(B, (n, n, n))
    need = int(_lib.lib().ctx_marching_cubes_workspace(n, n, n))
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    counts = torch.zeros(2, dtype=torch.int64, device=dev)
    v, nr, f = (torch.empty_like(ref[k]) for k in ("vertices", "normals", "faces"))
    st = stream_ptr(dev)
    args_ = (ptr(sigma), n, n, n, *o, *h, 0.0, ptr(ws), need, ptr(counts))

    def both():
        call("ctx_marching_cubes", *args_, None, None, None, 0, st)
        call("ctx_marching_cubes", *args_, ptr(v), ptr(nr), ptr(f), 1, st)

    src = torch.empty(1 << 29, device=dev)
    dst = torch.empty_like(src)
    fns = {"copy": lambda: dst.copy_(src), "marching_cubes": both}
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    assert torch.equal(v, ref["vertices"]) and torch.equal(f, ref["faces"])
    times = {k: [] for k in fns}
    for rep in range(args.reps):
        for k in (list(fns) if rep % 2 == 0 else list(fns)[::-1]):
            times[k].append(event_ms(fns[k], args.launches))
    med = {k: statistics.median(x) for k, x in times.items()}
    copy_bw = 2 * src.numel() * 4 / (med["copy"] * 1e-3)
    bytes_ = sigma.numel() * 4 + V * 24 + F * 12
    return {"cells": n, "vertices": V, "faces": F, "workspace_MB": round(need / 1e6, 1),
            "copy_GBps": round(copy_bw / 1e9, 1), "ms_median": round(med["marching_cubes"], 4),
            "ms_passes": [round(x, 4) for x in times["marching_cubes"]],
            "fraction_of_copy_bw": round(bytes_ / (med["marching_cubes"] * 1e-3) / copy_bw, 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=4, help="timed passes of each variant (alternating)")
    ap.add_argument("--launches", type=int, default=10, help="marching-cubes calls per timed pass")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mesh_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = gpu_info(dev)
    result["lattice"] = bench_lattice(dev, args)
    torch.cuda.empty_cache()
    result["ctx_marching_cubes"] = bench_mcubes(dev, args)
    print(json.dumps(result, indent=1), flush=True)


if __name__ == "__main__":
    main()
