"""Occupancy-grid sampler: fused engine (HotPath(sampler="occgrid")) against the drop-in loop
(examples/train_dropin.py --sampler occgrid: render_rays + F.mse_loss + backward + torch.optim.Adam
+ update_every_n_steps) from the same trained state, in the reference's configuration
(render_step_size 5e-3, one 128^3 grid).

Setup: the engine trains the synthetic Blender scene (synthetic.make_views, 8 views of 100x100) for
--train-steps steps at 1024 rays, which populates the grid; the drop-in model and estimator then
receive its weights and grid.  Timing: at 1024 and 4096 rays, blocks of --steps steps alternate
between the two (--reps blocks each), each block ending in a device synchronise; both include the
grid update every 16th step.  A separate profiled run gives the engine's per-kernel times.
    python tools/occgrid_speed.py [--train-steps 500 --steps 50 --reps 3]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import ops, synthetic as syn  # noqa: E402
from fsnerf_b200.core.models import NeRF  # noqa: E402
from fsnerf_b200.engine import HotPath  # noqa: E402
from fsnerf_b200.render.rendering import OccGridEstimator, render_rays  # noqa: E402

AABB = [-1.5] * 3 + [1.5] * 3
STEP = 5e-3
KW = {"pos_fn": {"n_freqs": 10, "log_space": True}, "dir_fn": {"n_freqs": 4, "log_space": True}}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        q = ""
    return q or torch.cuda.get_device_name(0) + ", power limit not read"


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--train-steps", type=int, default=500)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args(argv)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(0)
    poses, imgs, focal = syn.make_views(8, 100, 100, seed=42)
    o = np.concatenate([syn.camera_rays(p, 100, 100, focal)[0].reshape(-1, 3) for p in poses])
    d = np.concatenate([syn.camera_rays(p, 100, 100, focal)[1].reshape(-1, 3) for p in poses])
    O, D = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    GT = torch.from_numpy(imgs.reshape(-1, 3).astype(np.float32)).to(dev)
    n = O.shape[0]
    gen = torch.Generator(device=dev).manual_seed(0)

    def batch(R):
        ids = torch.randint(n, (R,), device=dev, generator=gen)
        return O[ids].contiguous(), D[ids].contiguous(), GT[ids].contiguous()

    hp = HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=128, render_step_size=STEP, device=dev)
    for _ in range(args.train_steps):
        ls = hp.train_step(*batch(1024))
    psnr = HotPath.psnr(ls[0].item(), 1024)
    model = NeRF(3, 3, 8, 256, [4], **KW).to(dev)
    model.load_state_dict(hp.state_dict(0))
    est = OccGridEstimator(AABB, resolution=128, levels=1).to(dev)
    est.load_state_dict(hp.estimator.state_dict())
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    model.train(); est.train()
    k_dropin = [hp.k]
    print(f"card: {card()}")
    print(f"setup: {args.train_steps} engine steps at 1024 rays, train PSNR {psnr:.2f} dB, "
          f"{int(hp.estimator.binaries.sum())} of 128^3 cells occupied")

    def engine_step(b):
        hp.train_step(*b)

    def dropin_step(b):
        ro, rd, gt = b
        (rgb, *_, extras), _, _ = render_rays(ro, rd, est, model, train=True, white_bkgd=True,
                                              render_step_size=STEP, device=dev)
        if extras is not None:
            F.mse_loss(rgb, gt).backward()
            opt.step()
            opt.zero_grad()
        est.update_every_n_steps(step=k_dropin[0], occ_eval_fn=lambda x: model(x) * STEP, occ_thre=1e-2)
        k_dropin[0] += 1

    rows = []
    for R in (1024, 4096):
        batches = [batch(R) for _ in range(args.steps)]
        times = {"engine": [], "drop-in": []}
        counts = []
        for name, fn in (("engine", engine_step), ("drop-in", dropin_step)):  # warm-up of every shape
            for b in batches[:5]:
                fn(b)
        for _ in range(args.reps):
            for name, fn in (("engine", engine_step), ("drop-in", dropin_step)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for b in batches:
                    fn(b)
                    if name == "engine":
                        counts.append(hp.last_counts)
                torch.cuda.synchronize()
                times[name].append((time.perf_counter() - t0) / len(batches))
        cand = np.mean([c[0] for c in counts]) / R
        surv = np.mean([c[1] for c in counts]) / R
        for name in ("engine", "drop-in"):
            ms = [1e3 * t for t in times[name]]
            rows.append((R, name, min(ms), max(ms), R / (min(ms) * 1e-3), cand, surv))
    print("| rays | path | ms/step (min-max of reps) | rays/s (best) | candidates/ray | survivors/ray |")
    print("|---|---|---|---|---|---|")
    for R, name, lo, hi, rps, cand, surv in rows:
        print(f"| {R} | {name} | {lo:.2f}-{hi:.2f} | {rps / 1e3:.0f} k | {cand:.1f} | {surv:.1f} |")

    # per-kernel times of the engine (separate, profiled run: the scopes time every launch)
    for R in (1024, 4096):
        batches = [batch(R) for _ in range(args.steps)]
        torch.cuda.synchronize()
        ops.profile_enable(True)
        for b in batches:
            engine_step(b)
        torch.cuda.synchronize()
        prof = ops.profile_read()
        ops.profile_enable(False)
        print(f"\nengine kernels at {R} rays, ms per step over {len(batches)} steps:")
        for k, (ms, cnt) in sorted(prof.items(), key=lambda kv: -kv[1][0]):
            print(f"  {k:28s} {ms / len(batches):8.3f} ms  ({cnt / len(batches):.2f} launches)")


if __name__ == "__main__":
    main()
