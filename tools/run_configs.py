"""BASELINE.json configs 2, 4 and 5 on one GPU (config 3 is bench.py, config 1 is the CPU leg).
Writes gpurun_out/configs_r02.json."""
import json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "contexture-nerf_b200")]
import torch
from ctxnerf import ops
from ctxnerf.train import NerfTrainer
from ctxnerf.workloads import orbit_camera, multiview_cameras

dev = torch.device("cuda", 0)
HBM, TF = 6540.2e9, 1412.2e12
MAC = 593408


def timeit(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2]


out = {}
K, c2w = orbit_camera()
tr = NerfTrainer(800, 800, K, c2w, perturb=0.0, white_bkgd=True, device=dev, seed=0)
# ---- config 2: single-view inference 800x800, coarse 64 + fine 128 ----
t = timeit(lambda: tr.render(None), iters=3, warm=1)
fl = 2.0 * MAC * 640000 * 256
out["cfg2_inference_800x800"] = {"ms": t * 1e3, "rays_per_s": 640000 / t, "tflops": fl / t / 1e12,
                                 "frac_tensor_sustained": fl / t / TF}
img = tr.render(None)["rgb_map"]
out["cfg2_inference_800x800"]["finite"] = bool(torch.isfinite(img).all())
# ---- config 4: 8 views x 1024^2, 192 samples, bounding sphere (views would be sharded one per GPU) ----
cams, sph = multiview_cameras()
Kv, cv = cams[0]
t = timeit(lambda: tr.render_view(1024, 1024, Kv, cv, n_samples=192, sphere=sph), iters=3, warm=1)
fl = 2.0 * MAC * 1024 * 1024 * 192
out["cfg4_view_1024x1024_192"] = {"ms_per_view": t * 1e3, "rays_per_s": 1024 * 1024 / t, "tflops": fl / t / 1e12,
                                  "frac_tensor_sustained": fl / t / TF, "views": 8,
                                  "note": "one view per GPU on 8 GPUs: no communication, wall = one view"}
# ---- config 5: HBM kernels, rays 2^12..2^22 x samples 64..512 ----
sweep = []
for lr in (12, 14, 16, 18, 20, 22):
    R = 1 << lr
    for S in (64, 128, 192, 256, 512):
        if R * S * 4 * 4 > (8 << 30):      # raw tensor over 8 GB: skipped as BASELINE allows
            continue
        raw = torch.randn(R, S, 4, device=dev); raw[..., 3] *= 5
        z = torch.sort(torch.rand(R, S, device=dev) * 4 + 2, -1)[0]
        d = torch.randn(R, 3, device=dev)
        w = torch.rand(R, S, device=dev)
        row = {"rays": R, "samples": S}
        t = timeit(lambda: ops.composite(raw, z, d), iters=3, warm=1)
        row["composite_fwd_gbs"] = R * (24 * S + 36) / t / 1e9
        # fused training form (forward + loss + backward in one pass): reads raw 16S + z 4S + d 12 + target 12, writes
        # g_raw 16S + weights 4S
        tgt = torch.rand(R, 3, device=dev); g_raw = torch.empty_like(raw); wts = torch.empty(R, S, device=dev)
        loss = torch.zeros(1, device=dev)
        rgb = torch.empty(R, 3, device=dev)
        from ctxnerf._lib import call, ptr, stream_ptr
        t = timeit(lambda: call("ctx_composite_train", ptr(raw), ptr(z), ptr(d), None, R, S, 1, ptr(tgt), 1.0 / (3 * R),
                                ptr(loss), ptr(g_raw), ptr(wts), ptr(rgb), stream_ptr(dev)), iters=3, warm=1)
        row["composite_train_gbs"] = R * (40 * S + 24) / t / 1e9
        # separate backward (all five output gradients given): reads raw 16S + z 4S + g_weights 4S + 36, writes g_raw 16S
        g = [torch.randn(R, 3, device=dev), torch.randn(R, device=dev), torch.randn(R, device=dev),
             torch.randn(R, S, device=dev), torch.randn(R, device=dev)]
        t = timeit(lambda: call("ctx_composite_bwd", ptr(raw), ptr(z), ptr(d), None, R, S, 1, ptr(g[0]), ptr(g[1]),
                                ptr(g[2]), ptr(g[3]), ptr(g[4]), ptr(g_raw), stream_ptr(dev)), iters=3, warm=1)
        row["composite_bwd_gbs"] = R * (40 * S + 36) / t / 1e9
        del tgt, g_raw, wts, g
        # get_rays + view directions + stratified depths of a sqrt(R) x sqrt(R) image: 36 + 4S B written per ray
        side = 1 << (lr // 2)
        Kc = [[1111.1, 0, side / 2.0], [0, 1111.1, side / 2.0], [0, 0, 1]]
        c2w_i = torch.eye(4, device=dev)[:3].contiguous()
        ro = (torch.empty(R, 3, device=dev), torch.empty(R, 3, device=dev), torch.empty(R, 3, device=dev), torch.empty(R, S, device=dev))
        for tag, pert in (("raygen_gbs", False), ("raygen_jitter_gbs", True)):
            t = timeit(lambda: ops.raygen(side, side, Kc, c2w_i, n_samples=S, near=2., far=6., perturb=pert, seed=1,
                                          want_viewdirs=True, out=ro), iters=3, warm=1)
            row[tag] = R * (36 + 4 * S) / t / 1e9
        del ro
        N = 2 * S
        if N <= 1024:
            bins_c, w_c = z[:, :S - 1].contiguous(), w[:, :S - 2].contiguous()   # (not part of the timed call)
            with torch.no_grad():   # sample_pdf proper (no index output): 4(B + B-1) B read + 4N B written per ray
                t = timeit(lambda: ops.resample(bins_c, w_c, N, det=True), iters=3, warm=1)
            row["resample_gbs"] = R * (4 * (S - 1) + 4 * (S - 2) + 4 * N) / t / 1e9
        pts = torch.rand(min(R * S, 1 << 25), 3, device=dev) * 4 - 2
        t = timeit(lambda: ops.posenc(pts, 10), iters=3, warm=1)
        row["posenc_gbs"] = pts.shape[0] * 264 / t / 1e9
        for k in list(row):
            if k.endswith("_gbs"):
                row[k.replace("_gbs", "_frac")] = row[k] * 1e9 / HBM
        sweep.append(row)
        bins_c = w_c = None
        del raw, z, d, w, pts
        torch.cuda.empty_cache()
out["cfg5_sweep"] = sweep
os.makedirs("gpurun_out", exist_ok=True)
json.dump(out, open("gpurun_out/configs_r02.json", "w"), indent=1)
for k, v in out.items():
    if k != "cfg5_sweep":
        print(k, v)
for r in sweep:
    print({a: (round(b, 3) if isinstance(b, float) else b) for a, b in r.items() if not a.endswith("_gbs")})
