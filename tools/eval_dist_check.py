"""torchrun --nproc-per-node N tools/eval_dist_check.py OUT_DIR : NerfTrainer.evaluate under N ranks.  Rank r renders
the test views v = r mod N and one all-reduce combines the per-view vectors; every rank must return the same vectors
bit for bit, and each rank writes them to OUT_DIR/rank{r}.npy ([3, N_test] fp64: mse, psnr, ssim) so that a caller
can compare them with a single-process evaluate of the same scene (scene() below)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "contexture-nerf_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402


def scene(dev):
    """A trainer on 64 x 64 orbit views (random weights, seed 0) and 5 held-out poses with uint8 targets: five views
    over two ranks give them unequal shares."""
    from ctxnerf.train import NerfTrainer
    from ctxnerf.workloads import orbit_camera
    H = W = 64
    cams = [orbit_camera(H, W, focal=80.0, azim_deg=72.0 * v + 10.0) for v in range(5)]
    poses = torch.stack([c for _, c in cams])
    images = torch.randint(0, 256, (5, H, W, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    torch.manual_seed(0)
    tr = NerfTrainer(H, W, cams[0][0], poses[0], N_samples=32, N_importance=64, device=dev, seed=0)
    return tr, poses, images


def main():
    import torch.distributed as dist
    out_dir = sys.argv[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    tr, poses, images = scene(dev)
    res = tr.evaluate(poses, images)
    vec = torch.stack([res["mse"], res["psnr"], res["ssim"]])
    mine = vec.to(dev)
    everyone = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(everyone, mine)
    same = all(torch.equal(e, mine) for e in everyone)
    print(f"rank {rank}/{world}: evaluate vectors identical on all ranks: {same}; psnr {vec[1].tolist()}", flush=True)
    np.save(os.path.join(out_dir, f"rank{rank}.npy"), vec.numpy())
    dist.barrier()
    dist.destroy_process_group()
    assert same


if __name__ == "__main__":
    main()
