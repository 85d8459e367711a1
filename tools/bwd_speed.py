"""Per-kernel times of one training step (tuning aid)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import ops
from fsnerf_b200.engine import HotPath
dev = torch.device("cuda:0")
hp = HotPath(device=dev, n_coarse=int(os.environ.get("N_COARSE", "64")), n_fine=int(os.environ.get("N_FINE", "128")))
R = 4096
g = torch.Generator().manual_seed(0)
o = (torch.tensor([0.0, 0, 4.0]) + 0.05 * torch.randn(R, 3, generator=g)).to(dev)
d = torch.nn.functional.normalize(torch.tensor([0.0, 0, -1.0]) + 0.3 * torch.randn(R, 3, generator=g), dim=-1).to(dev)
gt = torch.rand(R, 3, generator=g).to(dev)
for _ in range(3):
    hp.train_step(o, d, gt)
torch.cuda.synchronize()
import threading, time
clk = []
stop = False
def _sample():
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(0)
        while not stop:
            clk.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetPowerUsage(h) / 1e3))
            time.sleep(0.005)
    except Exception as e:
        clk.append((-1, -1))
th = threading.Thread(target=_sample, daemon=True)
th.start()
n = int(os.environ.get("N_STEPS", "40"))
t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
t0.record()
for _ in range(n):
    hp.train_step(o, d, gt)
t1.record()
torch.cuda.synchronize()
stop = True
print(f"step {t0.elapsed_time(t1) / n:.3f} ms; SM MHz median {sorted(c[0] for c in clk)[len(clk) // 2]} min {min(c[0] for c in clk)}; W max {max(c[1] for c in clk):.0f}", end=" ")
ops.profile_enable(True)
n = 5
for _ in range(n):
    hp.train_step(o, d, gt)
prof = ops.profile_read()
ops.profile_enable(False)
print({k: v[1] // n for k, v in prof.items() if k.startswith("mlp")}, end=" ")
print({k: round(v[0] / n, 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])[:5]})
