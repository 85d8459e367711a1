"""MLP forward throughput (render-style, no stash) — tuning aid."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import ops
from fsnerf_b200.engine import HotPath
dev = torch.device("cuda:0")
hp = HotPath(device=dev)
R, S = 65536, 192
g = torch.Generator().manual_seed(0)
o = (torch.tensor([0.0, 0, 4.0]) + 0.05 * torch.randn(R, 3, generator=g)).to(dev)
d = torch.nn.functional.normalize(torch.tensor([0.0, 0, -1.0]) + 0.3 * torch.randn(R, 3, generator=g), dim=-1).to(dev)
ts, te = ops.sample_stratified(R, S, 2.0, 6.0, None, device=dev)
hp._pack()
for _ in range(2):
    ops.mlp_forward(hp.cfg, hp.net_params(0), hp.packed[0], rays_o=o, rays_d=d, t_starts=ts, t_ends=te)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
n = 5
for _ in range(n):
    ops.mlp_forward(hp.cfg, hp.net_params(0), hp.packed[0], rays_o=o, rays_d=d, t_starts=ts, t_ends=te)
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / n
tf = R * S * 1186816 / (ms * 1e-3) / 1e12
print(f"{ms:.3f} ms, {tf:.0f} TFLOP/s, {tf/1408.5:.3f} of sustained peak")
