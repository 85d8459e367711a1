"""Where the CTAs of the fused MLP backward wait (tuning aid): per-role cycle counters that the
kernel accumulates when a trace buffer is set (csrc/mlp_bwd2.cu: kStatBase)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import _lib, ops  # noqa: E402
from fsnerf_b200.engine import HotPath  # noqa: E402

dev = torch.device("cuda:0")
hp = HotPath(device=dev, n_coarse=int(os.environ.get("N_COARSE", "64")), n_fine=int(os.environ.get("N_FINE", "128")))
R = 4096
g = torch.Generator().manual_seed(0)
o = (torch.tensor([0.0, 0, 4.0]) + 0.05 * torch.randn(R, 3, generator=g)).to(dev)
d = torch.nn.functional.normalize(torch.tensor([0.0, 0, -1.0]) + 0.3 * torch.randn(R, 3, generator=g), dim=-1).to(dev)
gt = torch.rand(R, 3, generator=g).to(dev)
for _ in range(2):
    hp.train_step(o, d, gt)
torch.cuda.synchronize()
trace = torch.zeros(8192, dtype=torch.int64, device=dev)
_lib.load().fsnerf_debug_set_trace(_lib.ptr(trace))
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
ops.profile_enable(True)
hp.train_step(o, d, gt)   # the fine pass (last) overwrites the coarse pass's counters
torch.cuda.synchronize()
print("event times of this step:", {k: round(v[0], 3) for k, v in ops.profile_read().items() if k.startswith("mlp")})
ops.profile_enable(False)
_lib.load().fsnerf_debug_set_trace(None)
s = trace.cpu()[1024:1024 + 148 * 8].view(148, 8).double() / 1e3
g_ = trace.cpu()[6144:6144 + 2 * 148].view(148, 2).double()
g_ = g_[g_[:, 0] > 0]
print(f"last launch on the global timer: first CTA start -> last CTA end {(g_[:, 1].max() - g_[:, 0].min()) / 1e6:.3f} ms; "
      f"start spread {(g_[:, 0].max() - g_[:, 0].min()) / 1e3:.1f} us; end spread {(g_[:, 1].max() - g_[:, 1].min()) / 1e3:.1f} us")
n_w = 58  # kWgradCtas in csrc/mlp_bwd2.cu
n_d = 148 - n_w
dg, wg = s[:n_d], s[n_d:]
print(f"dgrad CTAs ({n_d}), kcycles mean [min..max]:")
for k, name in [(0, "total"), (1, "store warp: ring slot (cons) wait"), (2, "store warp: staged slab wait"),
                (5, "store warp: publish (barrier + fence)"), (3, "epilogue: staging buffer wait"),
                (4, "epilogue: accumulator wait")]:
    c = dg[:, k]
    print(f"  {name:40s} {c.mean():9.1f} [{c.min():9.1f} .. {c.max():9.1f}]")
print(f"wgrad CTAs ({n_w}), per job: CTAs, tiles/CTA, total kcyc, producer ready-wait, producer empty-wait, MMA full-wait, cycles issue->landed per stage")
for j in sorted(set(int(x) for x in (wg[:, 6] * 1e3).round().tolist())):
    m = (wg[:, 6] * 1e3).round() == j
    r = wg[m]
    print(f"  job {j:2d}: {int(m.sum()):3d} {r[:, 4].mean() * 1e3:7.0f} {r[:, 0].mean():9.1f} {r[:, 1].mean():9.1f} "
          f"{r[:, 2].mean():9.1f} {r[:, 3].mean():9.1f} {(r[:, 5] / (2 * r[:, 4])).mean():9.0f}")

# life of the first images of dgrad CTA 0 (global timer, us relative to the first event)
e = trace.cpu()[4096:4096 + 7 * 256].view(7, 256).double()
t0 = e[e > 0].min()
names = ["slot_wait", "slot_ok", "done", "published", "scouted", "issued", "released"]
print("image q (tile iter * 10 + image): " + " ".join(f"{n:>10s}" for n in names) + "   (us; images with two readers have no issue/release stamps)")
for q in list(range(0, 40)) + list(range(100, 120)):
    print(f"  q={q:3d} " + " ".join(f"{(e[k, q] - t0) / 1e3:10.1f}" if e[k, q] > 0 else "         -" for k in range(7)))

# dgrad CTA 0, per tile iteration and step: cycles relative to the tile's first stamp
tl = trace.cpu()[:4 * 16 * 8].view(4, 16, 8).double()
print("dgrad CTA 0 timeline (cycles from the tile's first stamp): issuer reached layer, first MMA issued, layer committed | "
      "epilogue starts waiting, accumulator full, epilogue done")
for it in range(1, 4):
    base = tl[it][tl[it] > 0].min() if (tl[it] > 0).any() else 0
    for s_ in range(12):
        if (tl[it, s_] > 0).any():
            print(f"  tile {it} step/layer {s_:2d}: " + " ".join(f"{(tl[it, s_, k] - base):9.0f}" if tl[it, s_, k] > 0 else "        -" for k in range(6)))

# placement: which SM each CTA of the last launch ran on, and what its TPC sibling (smid ^ 1) did
smid = trace.cpu()[6500:6500 + 148].tolist()
role = {int(sm): ("d" if b < n_d else "w") for b, sm in enumerate(smid)}
print("blockIdx -> smid:", " ".join(f"{b}:{int(sm)}" for b, sm in enumerate(smid)))
import collections
pairs = collections.Counter("".join(sorted(role.get(sm, "-") + role.get(sm ^ 1, "-"))) for sm in role if sm % 2 == 0 or (sm ^ 1) not in role)
print("TPC role pairs:", dict(pairs))
for sib in ("w", "d"):
    m = torch.tensor([role.get(int(smid[n_d + i]) ^ 1, "-") == sib for i in range(n_w)])
    if m.any():
        r = wg[m]
        print(f"wgrad CTAs whose TPC sibling is {sib}: n={int(m.sum())} MMA full-wait {r[:, 3].mean():8.1f} kcyc, issue->landed {(r[:, 5] / (2 * r[:, 4])).mean():6.0f} cyc, ready-wait {r[:, 1].mean():8.1f}")
for sib in ("w", "d"):
    m = torch.tensor([role.get(int(smid[i]) ^ 1, "-") == sib for i in range(n_d)])
    if m.any():
        r = dg[m]
        print(f"dgrad CTAs whose TPC sibling is {sib}: n={int(m.sum())} cons wait {r[:, 1].mean():8.1f} staging wait {r[:, 3].mean():8.1f} acc wait {r[:, 4].mean():8.1f}")

print("wgrad CTAs: id job smid total ready-wait empty-wait full-wait issue->landed")
for i in range(n_w):
    r = wg[i]
    print(f"  {i:3d} {int(round(float(r[6]) * 1e3)):3d} {int(smid[n_d + i]):4d} {r[0]:8.1f} {r[1]:8.1f} {r[2]:8.1f} {r[3]:8.1f} {float(r[5] / (2 * r[4])):7.0f}")
