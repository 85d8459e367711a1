"""Per-phase clock64 timeline of CTA 0 of the MLP dgrad kernel (tuning aid)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import ops, _lib  # noqa: E402
from fsnerf_b200.engine import HotPath  # noqa: E402

dev = torch.device("cuda:0")
hp = HotPath(device=dev)
R = 4096
g = torch.Generator().manual_seed(0)
o = (torch.tensor([0.0, 0, 4.0]) + 0.05 * torch.randn(R, 3, generator=g)).to(dev)
d = torch.nn.functional.normalize(torch.tensor([0.0, 0, -1.0]) + 0.3 * torch.randn(R, 3, generator=g), dim=-1).to(dev)
gt = torch.rand(R, 3, generator=g).to(dev)
hp.train_step(o, d, gt)
torch.cuda.synchronize()
trace = torch.zeros(2048, dtype=torch.int64, device=dev)
_lib.load().fsnerf_debug_set_trace(_lib.ptr(trace))
hp.train_step(o, d, gt)
torch.cuda.synchronize()
_lib.load().fsnerf_debug_set_trace(None)
t = trace.cpu()[:512].view(4, 16, 8)
t0 = int(t[t > 0].min())
print("dgrad (fine pass; forward entries of steps >= 9 are stale): mma_wait_start mma_start mma_committed | epi_wait_start epi_start epi_end")
for it in range(1, 3):
    for s in range(9):
        r = [int(x) - t0 if x > 0 else -1 for x in t[it, s, :6]]
        print(f"  tile {it} step {s}: mma wait {r[1]-r[0]:6d} issue {r[2]-r[1]:6d} | epi wait(acc) {r[4]-r[3]:6d} epi {r[5]-r[4]:6d} | abs {r}")
