"""torchrun --nproc-per-node N tools/dist_check.py : the all-reduced gradient bucket of N ranks (each with
its own 4096-ray batch) equals the sum of the per-batch gradients computed by one process (SURVEY.md 8e); then four
optimizer steps (the captured graph from the second on, all-reduce inside it when the library's NCCL binding is in
use) must leave bit-identical parameters on every rank.  CTXNERF_NCCL=0 checks the torch.distributed route."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "contexture-nerf_b200")]
import torch
import torch.distributed as dist
from ctxnerf.train import NerfTrainer
from ctxnerf.workloads import orbit_camera

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
K, c2w = orbit_camera()
tr = NerfTrainer(800, 800, K, c2w, perturb=0.0, device=dev, seed=0)       # perturb=0: deterministic sampling
batches = []
for r in range(world):
    g = torch.Generator().manual_seed(100 + r)
    batches.append((torch.randint(0, 640000, (4096,), generator=g).to(dev), torch.rand(4096, 3, generator=g).to(dev)))
# distributed: my batch, one all-reduce
tr.step(*batches[rank], optimizer_step=False)
reduced = tr.bucket.grad.clone()
# single process reference on this rank: sum of the gradients of every batch
ref = torch.zeros_like(reduced)
for b in batches:
    tr.bucket.zero_grad()
    tr.reduce_gradients = False
    tr.step(*b, optimizer_step=False)
    tr.reduce_gradients = True
    ref += tr.bucket.grad
torch.cuda.synchronize()
err = (reduced - ref).abs().max().item() / ref.abs().max().item()
cos = torch.nn.functional.cosine_similarity(reduced, ref, dim=0).item()
route = f"ctx_allreduce (NCCL {tr.comm.version})" if tr.comm is not None else "torch.distributed"
print(f"rank {rank}/{world}: all-reduced vs single-process sum: max rel err {err:.3e}, cosine {cos:.8f} [{route}]",
      flush=True)
assert err < 1e-3 and cos > 0.999999
# optimizer steps: eager, then captured; every rank must hold the same parameters afterwards
tr.bucket.zero_grad()
for i in range(4):
    loss = tr.step(*batches[(rank + i) % world])
torch.cuda.synchronize()
mine = tr.bucket.flat.clone()
everyone = [torch.empty_like(mine) for _ in range(world)]
dist.all_gather(everyone, mine)
same = all(torch.equal(e, mine) for e in everyone)
graphs = sum(pl.graph is not None for pl in tr._plans.values()), sum(pl.graph_tail is not None for pl in tr._plans.values())
print(f"rank {rank}/{world}: parameters after 4 steps identical on all ranks: {same}; loss {loss.item():.5f}; "
      f"graphs head/tail {graphs}", flush=True)
assert same and torch.isfinite(loss).all()
dist.barrier()
dist.destroy_process_group()
