"""Per-role cycle counters of mlp_dgrad_kernel, from the diagnostics build (libctxnerf_diag.so, include/ctxnerf_diag.h)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "contexture-nerf_b200")]
import torch
from ctxnerf import _lib as _l0; lib = _l0.use_diag_lib()   # diagnostics build (include/ctxnerf_diag.h)
from ctxnerf import run_nerf_helpers as rh
from ctxnerf.mlp import forward_raw
from ctxnerf.mlp_bwd import mlp_dgrad
dev = torch.device("cuda", 0)
torch.manual_seed(0)
net = rh.NeRF().to(dev)
R, S = 4096, 192
o = torch.randn(R, 3, device=dev); d = torch.randn(R, 3, device=dev); d = d / d.norm(dim=-1, keepdim=True)
z = torch.sort(torch.rand(R, S, device=dev) * 4 + 2, -1)[0]
out, acts, P, packed = forward_raw(net, rays=(o, d, d, z), save_acts=True)
g = torch.randn(P, 4, device=dev) / P
prof = torch.zeros(148 * 16, dtype=torch.int64, device=dev)
for _ in range(2):
    mlp_dgrad(net, packed, acts, P, g)
torch.cuda.synchronize()
lib.ctx_dgrad_set_prof(prof.data_ptr())
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(); mlp_dgrad(net, packed, acts, P, g); b.record()
torch.cuda.synchronize()
lib.ctx_dgrad_set_prof(None)
print(f"dgrad {a.elapsed_time(b):.3f} ms   (TMA stores: {os.environ.get('CTXNERF_DGRAD_TMA', '1')})")
p = prof.cpu().reshape(148, 16).double()
names = {0: "issuerA.wait_act", 1: "issuerA.wait_full", 2: "issuerA.total", 3: "issuerB.wait_act", 4: "issuerB.wait_full",
         5: "issuerB.total", 6: "store.wait_ready", 7: "store.issue+read", 8: "epi4.wait_acc", 9: "epi4.wait_free",
         10: "epi4.body", 11: "epi4.total", 12: "epi11.wait_acc", 13: "epi11.wait_free", 14: "epi11.body", 15: "epi11.head_init"}
nph = 21 * 9 * 2
for i, n in names.items():
    for par, tag in ((0, "leader"), (1, "peer")):
        col = p[par::2, i]
        nz = col[col > 0]
        if len(nz):
            print(f"   {n:18s} {tag:6s} mean {nz.mean().item():10.0f}  (per phase slot {nz.mean().item() / nph:7.0f})")
