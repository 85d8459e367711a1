"""Cost of the deterministic mode: HotPath(deterministic=True) against the default engine on the same
state and rays.

Workloads: the C2 hierarchical step (4096 rays, 64 + 128 samples per ray) and the occupancy-grid step
at 1024 rays (render_step_size 5e-3, one 128^3 grid populated by --train-steps default-mode steps,
then copied into both engines).  Timing: blocks of --steps steps alternate between the two modes
(--reps blocks each), each block ending in a device synchronise.  A separate profiled run per mode
gives the MLP backward's kernels per launch (fsnerf_profile_* scopes).
    python tools/det_speed.py [--train-steps 300 --steps 30 --reps 3]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import ops, synthetic as syn  # noqa: E402
from fsnerf_b200.engine import HotPath  # noqa: E402

AABB = [-1.5] * 3 + [1.5] * 3
STEP = 5e-3
KERNELS = ("mlp_bwd_fused", "mlp_heads_wgrad", "mlp_bwd_det_reduce", "adam")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        q = ""
    return q or torch.cuda.get_device_name(0) + ", power limit not read"


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--train-steps", type=int, default=300)
    ap.add_argument("--steps", type=int, default=30)
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

    print(f"card: {card()}")
    # C2: hierarchical, 4096 rays; occgrid: 1024 rays on a trained grid
    hier = {det: HotPath(device=dev, deterministic=det) for det in (False, True)}
    occ = {det: HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=128, render_step_size=STEP, device=dev,
                        deterministic=det) for det in (False, True)}
    for _ in range(args.train_steps):
        occ[False].train_step(*batch(1024))
    occ[True].params.copy_(occ[False].params)
    occ[True].load_state_dict(0, occ[False].state_dict(0))
    occ[True].estimator.load_state_dict(occ[False].estimator.state_dict())
    occ[True].k = occ[False].k
    print(f"occgrid setup: {args.train_steps} default steps at 1024 rays, "
          f"{int(occ[False].estimator.binaries.sum())} of 128^3 cells occupied")

    rows, prof_rows = [], []
    for wl, engines, R in (("C2 hierarchical", hier, 4096), ("occgrid", occ, 1024)):
        batches = [batch(R) for _ in range(args.steps)]
        for det in (False, True):  # warm-up of every shape
            for b in batches[:5]:
                engines[det].train_step(*b)
        times = {False: [], True: []}
        for _ in range(args.reps):
            for det in (False, True):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for b in batches:
                    engines[det].train_step(*b)
                torch.cuda.synchronize()
                times[det].append(1e3 * (time.perf_counter() - t0) / len(batches))
        for det in (False, True):
            rows.append((wl, R, "deterministic" if det else "default", min(times[det]), max(times[det])))
        for det in (False, True):  # profiled runs, separate from the timed ones
            torch.cuda.synchronize()
            ops.profile_enable(True)
            for b in batches:
                engines[det].train_step(*b)
            torch.cuda.synchronize()
            prof = ops.profile_read()
            ops.profile_enable(False)
            per = {k: (prof[k][0] / prof[k][1] if k in prof and prof[k][1] else None) for k in KERNELS}
            prof_rows.append((wl, "deterministic" if det else "default", per))

    print("| workload | rays | mode | ms/step (min-max of reps) |")
    print("|---|---|---|---|")
    for wl, R, mode, lo, hi in rows:
        print(f"| {wl} | {R} | {mode} | {lo:.2f}-{hi:.2f} |")
    print("\n| workload | mode | " + " | ".join(f"{k} ms/launch" for k in KERNELS) + " |")
    print("|---|---|" + "---|" * len(KERNELS))
    for wl, mode, per in prof_rows:
        print(f"| {wl} | {mode} | " + " | ".join("-" if per[k] is None else f"{per[k]:.3f}" for k in KERNELS) + " |")


if __name__ == "__main__":
    main()
