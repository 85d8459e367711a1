"""Per-phase clock64 timeline of CTA 0 of the MLP forward (tuning aid)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import ops, _lib  # noqa: E402
from fsnerf_b200.engine import HotPath  # noqa: E402

dev = torch.device("cuda:0")
hp = HotPath(device=dev)
R = int(os.environ.get("R", "16384"))
g = torch.Generator().manual_seed(0)
o = (torch.tensor([0.0, 0, 4.0]) + 0.05 * torch.randn(R, 3, generator=g)).to(dev)
d = torch.nn.functional.normalize(torch.tensor([0.0, 0, -1.0]) + 0.3 * torch.randn(R, 3, generator=g), dim=-1).to(dev)
TRAIN = os.environ.get("TRAIN", "0") == "1"  # TRAIN=1: the training forward (stash + masks written)


def run():
    if not TRAIN:
        return hp.render(o, d)
    S = 192
    ts, te = ops.sample_stratified(R, S, 2.0, 6.0, None, device=dev)
    hp._pack()
    stash = torch.empty(ops.mlp_stash_bytes(hp.cfg, R * S), dtype=torch.uint8, device=dev)
    return ops.mlp_forward(hp.cfg, hp.net_params(1), hp.packed[1], rays_o=o, rays_d=d, t_starts=ts, t_ends=te, stash=stash)


run()
torch.cuda.synchronize()
trace = torch.zeros(2048, dtype=torch.int64, device=dev)
_lib.load().fsnerf_debug_set_trace(_lib.ptr(trace))
run()
torch.cuda.synchronize()
_lib.load().fsnerf_debug_set_trace(None)
t = trace.cpu()[:512].view(4, 16, 8)
t0 = int(t[t > 0].min())
print("columns: mma_wait_start mma_start mma_committed | epi_wait_start epi_start epi_end   (cycles since first event; fine pass overwrites coarse)")
for it in range(3):
    print(f"tile iter {it}:")
    for g_ in range(10):
        r = [int(x) - t0 if x > 0 else -1 for x in t[it, g_, :6]]
        print(f"  L{g_}: mma wait {r[1]-r[0]:6d} issue {r[2]-r[1]:6d} | epi wait(acc) {r[4]-r[3]:6d} epi {r[5]-r[4]:6d} | abs {r}")
