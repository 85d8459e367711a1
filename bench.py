#!/usr/bin/env python
"""bench.py — train rays/s (fwd+bwd+Adam) of the fs-nerf ray-march hot path on N B200s,
with render Mrays/s, the live roofline of the dominant kernel and the CPU baseline.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs bench_out   # + the last timed step's arrays
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference --steps 3 --warmup 1        # CPU arm

Workload (BASELINE.json configs[1]): synthetic Blender-format scene, 8 views at
400x400, coarse+fine NeRF 8x256 (64 + 128 samples, hierarchical sample_pdf),
4096-ray batches per GPU (weak scaling: global batch 4096*N; N=8 is configs[4]'s
32768-ray global batch; `--scaling strong` keeps the global batch at 32768 rays for every N).
One "step" = one optimisation step: ray generation from pixel ids, stratified + sample_pdf
sampling, coarse+fine MLP forward, compositing, MSE, full backward, [NCCL all-reduce of the flat
gradient], Adam.  Prints ONE JSON line (rank 0) on stdout:

  value     engine.HotPath.train_step with the pixel ids, poses and images resident in HBM
  e2e       the reference's own loop on the drop-in modules — render_rays (autograd) +
            F.mse_loss + loss.backward() + torch.optim.Adam (src/run-nerf.py:232-285) — fed from
            pinned HOST batches, with the loss read back every step
  roofline  the dominant MLP kernel against the bf16 tensor roof (SURVEY.md §8d FLOPs / its
            CUDA-event time, measured in a separate pass AFTER the timed region)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 400
N_VIEWS = 8
R_PER_GPU = 4096
STRONG_GLOBAL = 32768  # configs[4]
N_COARSE, N_FINE = 64, 128
NEAR, FAR = 2.0, 6.0
F_FWD = 1_186_816      # FLOP per sample evaluation, forward (SURVEY.md §8d)
F_TRAIN = 3_489_024    # forward + backward
F_DENSITY = 982_528    # density-only forward (the coarse pass of a hierarchical RENDER skips the view branch)
METRIC = "train_rays_per_s"
CPU_SAMPLE_RAYS = 512  # rays per step of the CPU arm (a bounded sample of the 4096-ray step)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled (NVML) every ~10 ms during the timed region"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.power = []

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            while not self.stop_flag:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1e3)
                except Exception:
                    pass
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                time.sleep(0.01)
        except Exception as e:  # NVML unavailable: fall back to one nvidia-smi sample
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                a, b = out.stdout.strip().split(",")
                self.sm.append(float(a))
                self.max_mhz = float(b)
            except Exception:
                self.reasons.add(f"unavailable: {e}")

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w_max": max(self.power) if self.power else None}


def make_scene():
    from fsnerf_b200 import synthetic as syn
    return syn.make_views(N_VIEWS, H, W, seed=42)


def host_ray_table(poses, imgs, focal):
    """the reference's dataset precomputes one ray per pixel of every view on the host, ONCE
    (src/nerfdata/datasets/llff.py:59-90): [V*H*W,3] x 3"""
    from fsnerf_b200 import synthetic as syn
    ro, rd = [], []
    for v in range(N_VIEWS):
        o_, d_ = syn.camera_rays(poses[v], H, W, focal)
        ro.append(o_.reshape(-1, 3))
        rd.append(d_.reshape(-1, 3))
    return np.concatenate(ro), np.concatenate(rd), imgs.reshape(-1, 3)


# ----------------------------------------------------------------------------- CPU arm
def cpu_step_fn(sample_rays):
    """One optimisation step of the ORACLE PORT (reference's Python NeRF math restated,
    oracle/render.py) on `sample_rays` rays of the same workload; returns a closure.  The ray
    table is built once, outside the timed steps, like the reference's dataset does."""
    import torch
    from oracle import mlp as omlp, render as orender
    poses, imgs, focal = make_scene()
    tab_o, tab_d, tab_rgb = host_ray_table(poses, imgs, focal)
    torch.set_num_threads(os.cpu_count())
    rng = np.random.default_rng(0)
    sdc, sdf = omlp.init_state_dict(seed=42), omlp.init_state_dict(seed=43)
    st = dict(step=0, m={}, v={})

    def step():
        ids = rng.integers(0, tab_o.shape[0], size=sample_rays)  # the DataLoader's shuffled batch
        us = rng.random((sample_rays, N_COARSE), dtype=np.float32)
        up = rng.random((sample_rays, N_FINE), dtype=np.float32)
        orender.train_step(sdc, sdf, st, tab_o[ids], tab_d[ids], tab_rgb[ids], NEAR, FAR, N_COARSE, N_FINE,
                           us, up, 5e-4, True)
    return step


def cpu_baseline(sample_rays=CPU_SAMPLE_RAYS, steps=16, warmup=1):
    step = cpu_step_fn(sample_rays)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": sample_rays / dt, "unit": "rays/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"{steps} optimisation steps of {sample_rays} rays x ({N_COARSE}+{N_COARSE + N_FINE}) "
                      f"sample evaluations of the same workload (oracle/render.py train_step, fp32 torch-CPU, "
                      f"{os.cpu_count()} threads, host ray table built once outside the timed steps); {dt:.2f} s/step"}, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base, dt = cpu_baseline(CPU_SAMPLE_RAYS, steps=max(1, args.steps), warmup=max(1, args.warmup))
    cfg = workload_config(args.gpus, args.scaling)
    cfg["cpu_rays_per_step"] = CPU_SAMPLE_RAYS
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "rays/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference arm = the reference's PyTorch NeRF math on the host CPU (oracle port: the "
                    "reference itself cannot run here, its sampler/compositor nerfacc 0.5.3 is not installable); "
                    f"each step is a bounded {CPU_SAMPLE_RAYS}-ray sample of the workload's {R_PER_GPU}-ray step "
                    "(config.cpu_rays_per_step), rays/s = sample rays / step time"}
    print(json.dumps(line))


def rays_per_gpu(world, scaling):
    return R_PER_GPU if scaling == "weak" else STRONG_GLOBAL // world


def workload_config(n, scaling="weak"):
    r = rays_per_gpu(n, scaling)
    return {"workload": f"C2: synthetic Blender-format scene {N_VIEWS} views {H}x{W}, coarse+fine NeRF 8x256, "
                        f"{N_COARSE}+{N_FINE} samples/ray (hierarchical sample_pdf), {r}-ray batch per GPU"
                        + ("" if scaling == "weak" else f" (C5: {STRONG_GLOBAL}-ray global batch, strong scaling)"),
            "rays_per_gpu": r, "global_rays": r * n, "n_coarse": N_COARSE, "n_fine": N_FINE,
            "parallelism": f"dp{n} (ray-sharded, one NCCL all-reduce of the flat fp32 gradient)" if n > 1 else "single GPU",
            "l2": "per-step working set (>5 GB of activation stash) exceeds the 126 MB L2; no explicit flush"}


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` (mean over the launches
    of one step) from the newest committed `ncu --set full` capture (profiles/*_traffic.json,
    written by tools/ncu_table.py); None when there is no capture of that kernel."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return None, None
    d = json.load(open(files[-1]))
    # (the forward's template arguments: <train> in older captures, <train, pair> since r02c)
    key = {"mlp_fwd_train": "mlp_fwd2_kernel<1", "mlp_fwd": "mlp_fwd2_kernel<0"}.get(kernel, kernel)
    rows = [r for k, v in d.items() if k.startswith(key) for r in v]
    if not rows:
        return None, None
    return (sum(r["dram_read_bytes"] + r["dram_write_bytes"] for r in rows) / len(rows),
            os.path.relpath(files[-1], ROOT) + f" ({len(rows)} launches)")


def nccl_summary(path, world):
    """rank lines of the NCCL INFO log (NCCL_DEBUG_FILE), echoed to stderr so that the launcher's
    log shows every rank's communicator without touching the one JSON line on stdout"""
    import glob
    import re
    lines, ranks = [], set()
    for f in sorted(glob.glob(path.replace("%h", "*").replace("%p", "*"))):
        try:
            for ln in open(f, errors="replace"):
                m = re.search(r"rank (\d+) nranks (\d+)", ln)
                if m and "Init COMPLETE" in ln:
                    ranks.add(int(m.group(1)))
                    lines.append(ln.rstrip())
        except OSError:
            pass
    for ln in lines:
        print(ln, file=sys.stderr)
    return {"nranks_seen": len(ranks), "nranks_expected": world, "init_lines": len(lines)}


# ----------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 4096 rays per GPU; strong: configs[4]'s 32768-ray global batch split over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-render", action="store_true")
    ap.add_argument("--no-engine-e2e", action="store_true", help="skip the fused-engine host-batch leg")
    ap.add_argument("--no-micro", action="store_true", help="skip the render-scale compositing / sampling rooflines")
    ap.add_argument("--no-sustain", action="store_true", help="skip the >= 2 s sustained leg")
    ap.add_argument("--no-c4", action="store_true", help="skip the C4 render_path leg")
    ap.add_argument("--c4-frames", type=int, default=8, help="800x800 poses of the C4 leg (whole job, split over the GPUs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed train step computed to DIR/<name>.npy (float32): loss_sums "
                         "(the step's return value), params and grads (the flat buffers of both networks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    nccl_file = None
    if world > 1:
        # NCCL's INFO log goes to a file (one per process), never to stdout: the banner would break the
        # ONE JSON line.  Rank 0 echoes the communicator lines of every rank to stderr at the end.
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        # The logs go to the temporary directory (the source tree may be read-only).  The launcher's pid,
        # which every local rank shares as its parent, keeps one run's logs apart from an earlier run's.
        nccl_file = os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join(
            tempfile.gettempdir(), f"fsnerf_nccl_{os.getppid()}_n{world}.%h.%p.log"))

    import torch
    import torch.distributed as dist
    import torch.nn.functional as Fnn
    from fsnerf_b200 import ops, synthetic as syn
    from fsnerf_b200.engine import HotPath
    from fsnerf_b200.core.models import NeRF
    from fsnerf_b200.parallel import allreduce_module_gradients
    from fsnerf_b200.render.rendering import HierarchicalEstimator, render_path, render_rays

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ops.require_device(local)
    W_ = max(3, args.warmup)
    K = args.steps
    Rg = rays_per_gpu(world, args.scaling)
    G = Rg * world

    poses, imgs, focal = make_scene()
    poses_d = torch.from_numpy(poses).to(dev)
    imgs_d = torch.from_numpy(imgs).to(dev)
    hp = HotPath(n_coarse=N_COARSE, n_fine=N_FINE, near=NEAR, far=FAR, white_bkgd=True, device=dev, lr=5e-4)
    g = torch.Generator().manual_seed(1234)
    n_pix = N_VIEWS * H * W
    total_steps = W_ + K
    # seeded pixel permutation, sliced per step and per rank (SURVEY.md §8e)
    perm = torch.stack([torch.randperm(n_pix, generator=g)[:G] for _ in range(total_steps)])  # [steps, G]
    ids_all = perm[:, rank * Rg:(rank + 1) * Rg].contiguous()
    ids_dev = ids_all.to(dev)

    def step_resident(i):
        ro, rd, gt = ops.gen_rays(poses_d, H, W, focal, pixel_ids=ids_dev[i % total_steps], images=imgs_d)
        hp.launches += 1
        return hp.train_step(ro, rd, gt, global_rays=G)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms_):
        t = torch.tensor([ms_], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- value: inputs resident in HBM (no per-kernel events inside this region)
    for i in range(W_):
        step_resident(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = hp.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(K):
        ls = step_resident(W_ + i)
    ev1.record()
    barrier()
    sampler.stop_flag = True
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = hp.launches - l0
    value = G * K / (ms / 1e3)
    final_loss = (ls[0].item() + ls[1].item()) / (3 * Rg)
    if args.dump_outputs and rank == 0:
        # Saved before the passes below train the same HotPath further.  The inputs are seeded, so two
        # builds run with the same arguments can be compared array by array (~9.5 MB in all), within a
        # tolerance: the loss and gradient sums are float atomics, and Adam turns their order noise in
        # near-zero gradients into lr-sized steps.  Two runs of one build at --steps 20 --warmup 3 (NVIDIA
        # B200, 1000 W limit) differed by 7e-6 relative in loss_sums, 1e-3 absolute in params, 2e-5 in grads.
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (("loss_sums", ls), ("params", hp.params), ("grads", hp.grads)):
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), t.detach().float().cpu().numpy())

    # ---- per-kernel times: a separate pass after the timed region (cudaEvent pairs around every launch)
    ops.profile_enable(True)
    for i in range(K):
        step_resident(W_ + i)
    torch.cuda.synchronize()
    prof = ops.profile_read()
    ops.profile_enable(False)
    prof_ms = sum(v[0] for v in prof.values())

    # ---- sustained leg: >= 2 s of back-to-back steps with the clocks sampled, so that the choice
    #      between the burst and the sustained bf16 peak is evidenced by this run's own clocks
    sustain = None
    if not args.no_sustain:
        n_sus = max(K, int(2200.0 / (ms / K)) + 1)
        s2 = ClockSampler(local)
        barrier()
        if rank == 0:
            s2.start()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for i in range(n_sus):
            step_resident(i)
        a1.record()
        barrier()
        s2.stop_flag = True
        ms_s = max_over_ranks(a0.elapsed_time(a1))
        sustain = {"steps": n_sus, "seconds": ms_s / 1e3, "value": G * n_sus / (ms_s / 1e3), "unit": "rays/s",
                   "ms_per_step": ms_s / n_sus, "clocks": s2.summary() if rank == 0 else None}

    # ---- host batches (pinned), the reference's DataLoader output: [B,3] x 3 fp32 per step
    tab_o, tab_d, tab_rgb = host_ray_table(poses, imgs, focal)
    host_batches = []
    for i in range(W_ + K):
        idx = ids_all[i % total_steps].numpy()
        host_batches.append(tuple(torch.from_numpy(np.ascontiguousarray(a[idx])).pin_memory()
                                  for a in (tab_o, tab_d, tab_rgb)))
    h2d = 3 * Rg * 3 * 4

    # ---- e2e: the reference's own train loop (src/run-nerf.py:232-285) on the drop-in modules
    kw = {"pos_fn": {"n_freqs": 10, "log_space": True}, "dir_fn": {"n_freqs": 4, "log_space": True}}
    torch.manual_seed(42)
    coarse, fine = NeRF(3, 3, 8, 256, [4], **kw).to(dev), NeRF(3, 3, 8, 256, [4], **kw).to(dev)
    est = HierarchicalEstimator(near=NEAR, far=FAR, n_coarse=N_COARSE, n_fine=N_FINE, proposal_model=coarse)
    opt = torch.optim.Adam(list(fine.parameters()) + list(coarse.parameters()), lr=5e-4)
    fine.train(); coarse.train(); est.train()
    loss_host = torch.zeros(1).pin_memory()
    mse_scale = float(Rg) / float(G)  # F.mse_loss over the LOCAL shard -> mean over the global batch after the SUM

    def step_dropin(i):
        ro, rd, gt = (b.to(dev, non_blocking=True) for b in host_batches[i])
        (rgb, *_, extras), _, _ = render_rays(ro, rd, est, fine, train=True, white_bkgd=True, device=dev)
        loss = Fnn.mse_loss(rgb, gt) + Fnn.mse_loss(extras["rgb_coarse"], gt)
        if world > 1:
            loss = loss * mse_scale
        loss.backward()
        if world > 1:
            allreduce_module_gradients([fine, coarse])
        opt.step()
        opt.zero_grad()
        loss_host.copy_(loss.detach().reshape(1), non_blocking=False)  # D2H read of the step's loss (synchronises)
        return loss_host

    for i in range(W_):
        step_dropin(i)
    barrier()
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    for i in range(K):
        step_dropin(W_ + i)
    d1.record()
    barrier()
    ms_d = max_over_ranks(d0.elapsed_time(d1))
    e2e_value = G * K / (ms_d / 1e3)
    del opt

    # ---- the fused engine fed from the same host batches (extra; the kernels' own host driver)
    engine_e2e = None
    if not args.no_engine_e2e:
        ls_host = torch.zeros(2).pin_memory()

        def step_host(i):
            ro, rd, gt = (b.to(dev, non_blocking=True) for b in host_batches[i])
            ls_ = hp.train_step(ro, rd, gt, global_rays=G)
            ls_host.copy_(ls_, non_blocking=False)
        for i in range(W_):
            step_host(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            step_host(W_ + i)
        e1.record()
        barrier()
        ms_e = max_over_ranks(e0.elapsed_time(e1))
        engine_e2e = {"value": G * K / (ms_e / 1e3), "unit": "rays/s", "ms_per_step": ms_e / K,
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                      "what": "engine.HotPath.train_step on pinned host batches, loss read back every step"}

    # ---- render Mrays/s (rank-local pixel slice of one 800x800 frame; no collective)
    render = None
    pk = peaks()
    if not args.no_render:
        RH = RW = 800
        chunk = 65536
        n_chunks = 4
        rfocal = syn.focal_from_fov(RW)
        pose_r = torch.from_numpy(syn.orbit_poses(8)[rank % 8]).to(dev)[None].contiguous()

        def render_chunk(c):
            ro, rd, _ = ops.gen_rays(pose_r, RH, RW, rfocal, first_id=(c * chunk) % (RH * RW - chunk), n_rays=chunk)
            return hp.render(ro, rd)
        render_chunk(0)
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for c in range(n_chunks):
            render_chunk(c + 1)
        r1.record()
        barrier()
        ms_r = max_over_ranks(r0.elapsed_time(r1))
        ops.profile_enable(True)
        for c in range(n_chunks):
            render_chunk(c + 1)
        torch.cuda.synchronize()
        rprof = ops.profile_read()
        ops.profile_enable(False)
        fwd_ms, _ = rprof.get("mlp_fwd", (0.0, 1))
        fl = n_chunks * chunk * (N_COARSE * F_DENSITY + (N_COARSE + N_FINE) * F_FWD)
        render = {"value": world * n_chunks * chunk / (ms_r / 1e3) / 1e6, "unit": "Mrays/s",
                  "chunk_rays": chunk, "chunks": n_chunks, "frame": f"{RH}x{RW}",
                  "mlp_fwd_tflops": fl / (fwd_ms / 1e3) / 1e12 if fwd_ms > 0 else None,
                  "mlp_fwd_frac_of_bf16_sustained": fl / (fwd_ms / 1e3) / 1e12 / pk["tf_sus"] if fwd_ms > 0 else None,
                  "mlp_fwd_frac_of_bf16_burst": fl / (fwd_ms / 1e3) / 1e12 / pk["tf_burst"] if fwd_ms > 0 else None,
                  "flops_per_ray": N_COARSE * F_DENSITY + (N_COARSE + N_FINE) * F_FWD}

    # ---- C4 (configs[3]) through the drop-in render_path: 800x800 poses, the flattened pixel range
    #      partitioned over the ranks with no collective, frames copied to the host like the reference
    c4 = None
    if not args.no_c4 and args.c4_frames > 0:
        Fc = args.c4_frames
        hwf = (800, 800, syn.focal_from_fov(800))
        c4_poses = torch.from_numpy(syn.orbit_poses(max(Fc, 2))[:Fc])
        fine.eval(); coarse.eval(); est.eval()
        render_path(c4_poses[:1], hwf, NEAR, FAR, 65536, fine, est, white_bkgd=True, device=dev)  # warm-up
        barrier()
        t0 = time.perf_counter()
        out = render_path(c4_poses, hwf, NEAR, FAR, 65536, fine, est, white_bkgd=True, device=dev,
                          rank=rank, world_size=world)
        torch.cuda.synchronize()
        sec = max_over_ranks((time.perf_counter() - t0) * 1e3) / 1e3
        n_local = out[0].reshape(-1, 3).shape[0]
        c4 = {"config": f"C4 sample: {Fc} of the 200 poses at 800x800 through render_path (chunk 65536), pixels "
                        f"partitioned over {world} GPU(s), frames returned as host numpy arrays",
              "rays": Fc * 800 * 800, "rays_this_rank": n_local, "seconds": sec,
              "value": Fc * 800 * 800 / sec / 1e6, "unit": "Mrays/s",
              "full_c4_seconds_extrapolated": sec * 200.0 / Fc}
    del coarse, fine, est

    # ---- compositing kernel at render scale (HBM roofline of kernel (4); SURVEY.md §7 "hard parts":
    #      at training sizes it is launch-latency bound and L2 resident)
    comp = None
    if rank == 0 and not args.no_micro:
        Rc, Sc_ = 262144, N_COARSE + N_FINE
        gcomp = torch.Generator(device=dev).manual_seed(0)
        raw = torch.rand(Rc, Sc_, 4, device=dev, generator=gcomp)
        e_ = torch.sort(2 + 4 * torch.rand(Rc, Sc_ + 1, device=dev, generator=gcomp), -1).values
        ts_, te_ = e_[:, :-1].contiguous(), e_[:, 1:].contiguous()
        d_rgb_ = torch.rand(Rc, 3, device=dev, generator=gcomp)
        bk_ = torch.ones(3, device=dev)
        for _ in range(3):
            ops.composite_forward(raw, ts_, te_, bkgd=bk_)
            ops.composite_backward(raw, ts_, te_, d_rgb_, bkgd=bk_)
        torch.cuda.synchronize()
        ops.profile_enable(True)
        for _ in range(10):
            ops.composite_forward(raw, ts_, te_, bkgd=bk_)   # 1.4 GB in + out per launch >> L2
            ops.composite_backward(raw, ts_, te_, d_rgb_, bkgd=bk_)
        cprof = ops.profile_read()
        ops.profile_enable(False)
        f_ms, b_ms = cprof["composite_fwd"][0] / 10, cprof["composite_bwd"][0] / 10
        f_bytes, b_bytes = Rc * (28 * Sc_ + 20), Rc * (40 * Sc_ + 40)  # bwd recomputes weights: 24 B in + 16 B out / sample
        comp = {"rays": Rc, "samples_per_ray": Sc_, "bound": "hbm", "peak": pk["hbm"], "unit": "GB/s",
                "fwd": {"ms": f_ms, "achieved": f_bytes / f_ms / 1e6, "frac": f_bytes / f_ms / 1e6 / pk["hbm"]},
                "bwd": {"ms": b_ms, "achieved": b_bytes / b_ms / 1e6, "frac": b_bytes / b_ms / 1e6 / pk["hbm"]}}
        del raw, e_, ts_, te_
        # sampling kernels (1) at the same scale, against the same HBM roof (algorithmic bytes of SURVEY §8d)
        us_ = torch.rand(Rc, N_COARSE, device=dev, generator=gcomp)
        up_ = torch.rand(Rc, N_FINE, device=dev, generator=gcomp)
        w_ = torch.rand(Rc, N_COARSE, device=dev, generator=gcomp) ** 4
        for _ in range(2):
            tsc_, _ = ops.sample_stratified(Rc, N_COARSE, NEAR, FAR, us_)
            ops.sample_pdf(tsc_, w_, N_FINE, FAR, up_, want_aux=False)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        for _ in range(10):
            tsc_, _ = ops.sample_stratified(Rc, N_COARSE, NEAR, FAR, us_)
        ev[1].record()
        for _ in range(10):
            ops.sample_pdf(tsc_, w_, N_FINE, FAR, up_, want_aux=False)       # training: random u
        ev[2].record()
        for _ in range(10):
            ops.sample_pdf(tsc_, w_, N_FINE, FAR, None, want_aux=False)      # rendering: deterministic u
        ev[3].record()
        torch.cuda.synchronize()
        st_b = Rc * (24 + 12 * N_COARSE)
        pdf_b = Rc * (4 * (2 * N_COARSE - 3) + 4 * N_FINE + 8 * (N_COARSE + N_FINE))  # weights, bins, u in; merged intervals out

        def _roof(b, ms_):
            return {"ms": ms_, "achieved": b / ms_ / 1e6, "frac": b / ms_ / 1e6 / pk["hbm"]}
        comp["sampling"] = {"stratified": _roof(st_b, ev[0].elapsed_time(ev[1]) / 10),
                            "sample_pdf_random_u": _roof(pdf_b, ev[1].elapsed_time(ev[2]) / 10),
                            "sample_pdf_deterministic_u": _roof(pdf_b - Rc * 4 * N_FINE, ev[2].elapsed_time(ev[3]) / 10)}
        del us_, up_, w_

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: an MLP kernel against the bf16 TENSOR roof (SURVEY.md §8d).
    #      achieved = algorithmic FLOPs of that kernel per step / its CUDA-event time per step (the
    #      profiled pass above): reproducible by hand from kernel_ms_per_step.
    P_all = Rg * (N_COARSE + N_COARSE + N_FINE)  # sample evaluations per step (both networks)
    # the backward's FLOPs include the degenerate heads (sigma / rgb weight gradients): their kernel's time is added to it
    flops = {"mlp_fwd_train": P_all * F_FWD, "mlp_bwd_fused": P_all * (F_TRAIN - F_FWD)}
    kms = {k: v[0] / K for k, v in prof.items()}
    dom = max((k for k in flops if k in kms), key=lambda k: kms[k])
    per_kernel = {}
    for k in flops:
        if k not in kms:
            continue
        t = kms[k] + (kms.get("mlp_heads_wgrad", 0.0) if k == "mlp_bwd_fused" else 0.0)
        tf = flops[k] / (t / 1e3) / 1e12
        tb, tsrc = ncu_traffic("mlp_bwd_fused_kernel" if k == "mlp_bwd_fused" else k)
        n_launch = prof[k][1] / K
        per_kernel[k] = {"ms_per_step": t, "flops_per_step": flops[k], "achieved_tflops": tf,
                         "frac_of_bf16_sustained": tf / pk["tf_sus"], "frac_of_bf16_burst": tf / pk["tf_burst"],
                         "dram_bytes_per_step_ncu": None if tb is None else tb * n_launch, "traffic_source": tsrc}
    D = per_kernel[dom]
    traffic, traffic_src = ncu_traffic("mlp_bwd_fused_kernel" if dom == "mlp_bwd_fused" else dom)
    # compulsory HBM bytes of the MLP part of a step: rays + intervals in, raw out, d_raw in (fp32)
    compulsory = P_all * (8 + 16 + 16) + Rg * 24 * 2
    mlp_dram = sum(v["dram_bytes_per_step_ncu"] for v in per_kernel.values() if v["dram_bytes_per_step_ncu"])
    mlp_ms = sum(kms.get(k, 0.0) for k in ("mlp_fwd_train", "mlp_bwd_fused", "mlp_heads_wgrad"))
    roofline = {"kernel": dom, "bound": "tensor", "achieved": D["achieved_tflops"], "peak": pk["tf_sus"],
                "unit": "TFLOP/s", "frac": D["frac_of_bf16_sustained"],
                "frac_of_burst_peak": D["frac_of_bf16_burst"],
                "peak_source": pk["src"] + " MEASURED_PEAKS.json: sustained bf16 (burst given beside it; the sustained "
                               "leg's clocks say which applies)",
                "traffic": traffic, "traffic_source": traffic_src,
                "mlp_dram_bytes_per_step_ncu": mlp_dram or None, "mlp_compulsory_bytes_per_step": compulsory,
                "wasted_traffic_ratio": (mlp_dram / compulsory) if mlp_dram else None,
                "launches_per_step": prof[dom][1] / K, "ms_per_step": D["ms_per_step"],
                "per_kernel": per_kernel,
                "kernel_ms_per_step": {k: v for k, v in sorted(kms.items(), key=lambda kv: -kv[1])},
                "kernel_share_of_step": {k: round(v / (prof_ms / K), 4) for k, v in sorted(kms.items(), key=lambda kv: -kv[1])},
                "profiled_pass_ms_per_step": prof_ms / K,
                "mlp_all_tflops": P_all * F_TRAIN / (mlp_ms / 1e3) / 1e12 if mlp_ms > 0 else None,
                "mlp_all_frac_of_bf16_sustained": P_all * F_TRAIN / (mlp_ms / 1e3) / 1e12 / pk["tf_sus"] if mlp_ms > 0 else None}

    base = None
    if not args.no_cpu_baseline:
        base, _ = cpu_baseline(CPU_SAMPLE_RAYS, steps=16, warmup=1)  # ~10-15 s of CPU work on the box's host cores

    nccl = nccl_summary(nccl_file, world) if nccl_file else None
    line = {"metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": K, "warmup": W_,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": workload_config(world, args.scaling),
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_d / K,
                    "what": "the reference's loop on the drop-in modules: render_rays (autograd) + F.mse_loss + "
                            "loss.backward() + torch.optim.Adam, pinned host batches, loss read back every step"
                            + (", NCCL all-reduce of the two flat gradient buffers" if world > 1 else "")},
            "e2e_engine": engine_e2e,
            "gpu_launches": launches, "roofline": roofline, "roofline_compositing": comp, "cpu_baseline": base,
            "render": render, "render_path_c4": c4, "sustained": sustain, "nccl": nccl,
            "clocks": sampler.summary(), "final_loss": final_loss,
            "mlp_model_flops_per_ray": (N_COARSE + N_COARSE + N_FINE) * F_TRAIN}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
