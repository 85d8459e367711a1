"""The occupancy-grid sampler on the fused engine (HotPath(sampler="occgrid")) and the kernels it adds:
the visibility filter (fsnerf_occgrid_filter) against a compaction of the compositor's own trans /
alphas and against oracle/occgrid.visibility, the packed sample points (fsnerf_packed_points) against
the drop-in's torch expression, and the engine's step / render / training against the drop-in loop
(examples/train_dropin.py --sampler occgrid) on the same weights, grid and jitter."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import occgrid as oocc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AABB = [-1.5] * 3 + [1.5] * 3
KW = {"pos_fn": {"n_freqs": 10, "log_space": True}, "dir_fn": {"n_freqs": 4, "log_space": True}}


@pytest.fixture(scope="module")
def dev():
    from fsnerf_b200 import ops
    ops.require_device(0)
    return torch.device("cuda:0")


def _candidates(counts, seed, dev, sigma_scale=20.0, sigma_shift=3.0):
    g = torch.Generator().manual_seed(seed)
    counts = torch.tensor(counts)
    ts = torch.cat([torch.sort(2 + 4 * torch.rand(int(c), generator=g)).values for c in counts])
    te = ts + 0.02
    sig = torch.randn(ts.numel(), generator=g) * sigma_scale + sigma_shift  # about 45 % negative
    offsets = torch.zeros(len(counts) + 1, dtype=torch.int64)
    offsets[1:] = torch.cumsum(counts, 0)
    return ts.to(dev), te.to(dev), sig.to(dev), offsets.to(dev)


@pytest.mark.parametrize("alpha_thre", [0.0, 0.05])
def test_filter_matches_compaction_and_oracle(dev, alpha_thre):
    from fsnerf_b200 import ops
    counts = [0, 1, 31, 32, 33, 1500, 0, 64, 2, 1200, 97, 0]
    eps = 1e-4
    ts, te, sig, offsets = _candidates(counts, 0, dev)
    ri, ts_k, te_k, off_k = ops.occgrid_filter(ts, te, offsets, sig, eps, alpha_thre)
    # reference 1: the mask the drop-in built from composite_packed_forward's trans / alphas, compacted
    raw = torch.zeros(ts.numel(), 4, device=dev)
    raw[:, 3] = sig
    *_, trans, alphas = ops.composite_packed_forward(raw, ts, te, offsets)
    mask = (trans >= eps).cpu().numpy()
    if alpha_thre > 0:
        mask &= (alphas >= alpha_thre).cpu().numpy()
    ri_all = np.repeat(np.arange(len(counts)), counts)
    assert 0 < mask.sum() < len(mask)
    np.testing.assert_array_equal(ri.cpu().numpy(), ri_all[mask])
    np.testing.assert_array_equal(ts_k.cpu().numpy(), ts.cpu().numpy()[mask])
    np.testing.assert_array_equal(te_k.cpu().numpy(), te.cpu().numpy()[mask])
    kept_counts = np.bincount(ri_all[mask], minlength=len(counts))
    np.testing.assert_array_equal(off_k.cpu().numpy(), np.concatenate([[0], np.cumsum(kept_counts)]))
    # reference 2: the fp32 torch oracle (different scan order): flips only where T sits at the threshold
    ref = oocc.visibility(sig.cpu().numpy(), ts.cpu().numpy(), te.cpu().numpy(), ri_all, eps, alpha_thre)
    flips = np.flatnonzero(ref != mask)
    assert len(flips) <= 3, len(flips)
    tr = trans.cpu().numpy()
    al = alphas.cpu().numpy()
    for i in flips:
        assert abs(tr[i] / eps - 1) < 1e-3 or (alpha_thre > 0 and abs(al[i] / alpha_thre - 1) < 1e-5), (i, tr[i])


def test_filter_general_compaction_not_prefix(dev):
    """one ray: dense, then negative density raises T back above the threshold"""
    from fsnerf_b200 import ops
    sig = torch.tensor([0.0, 300.0, 300.0, 0.0, -600.0, 0.0, 0.0], device=dev)
    ts = torch.arange(7, dtype=torch.float32, device=dev) * 0.02
    te = ts + 0.02
    offsets = torch.tensor([0, 7], dtype=torch.int64, device=dev)
    ri, ts_k, _, off = ops.occgrid_filter(ts, te, offsets, sig, 1e-4, 0.0)
    # T: 1, 1, e^-6, e^-12 (< 1e-4), e^-12, 1, 1
    np.testing.assert_array_equal(ts_k.cpu().numpy(), ts.cpu().numpy()[[0, 1, 2, 5, 6]])
    assert off.tolist() == [0, 5] and ri.tolist() == [0] * 5


def test_filter_empty_and_canary(dev):
    from fsnerf_b200 import ops, _lib
    from fsnerf_b200._lib import ptr
    ts, te, sig, offsets = _candidates([0, 0, 0], 1, dev)
    ri, a, b, off = ops.occgrid_filter(ts, te, offsets, sig)
    assert ri.numel() == 0 and off.tolist() == [0, 0, 0, 0]
    empty = torch.zeros(1, dtype=torch.int64, device=dev)  # R = 0
    ri, a, b, off = ops.occgrid_filter(ts[:0], te[:0], empty, sig[:0])
    assert ri.numel() == 0 and off.tolist() == [0]
    # fill pass into oversized outputs: nothing past the M survivors is written
    ts, te, sig, offsets = _candidates([40, 7, 300], 2, dev)
    ri, ts_k, te_k, off = ops.occgrid_filter(ts, te, offsets, sig)
    M = ri.numel()
    ri_big = torch.full((M + 64,), -7, dtype=torch.int64, device=dev)
    ts_big = torch.full((M + 64,), 1234.5, device=dev)
    te_big = torch.full((M + 64,), 1234.5, device=dev)
    lib = _lib.load()
    _lib.check(lib.fsnerf_occgrid_filter(3, ptr(offsets), ptr(ts), ptr(te), ptr(sig), 1e-4, 0.0, ptr(off), None,
                                         ptr(ri_big), ptr(ts_big), ptr(te_big), None), "filter")
    torch.cuda.synchronize()
    assert torch.equal(ri_big[:M], ri) and torch.equal(ts_big[:M], ts_k) and torch.equal(te_big[:M], te_k)
    assert bool((ri_big[M:] == -7).all()) and bool((ts_big[M:] == 1234.5).all()) and bool((te_big[M:] == 1234.5).all())
    # argument checks
    assert lib.fsnerf_occgrid_filter(3, None, ptr(ts), ptr(te), ptr(sig), 1e-4, 0.0, None, None, None, None, None,
                                     None) == -1
    assert lib.fsnerf_packed_points(5, None, ptr(ts), ptr(te), ptr(ts), ptr(ts), ptr(ts), None, None) == -1


def test_packed_points_bit_equal(dev):
    from fsnerf_b200 import ops
    g = torch.Generator().manual_seed(3)
    R, N = 500, 40000
    ro = (torch.randn(R, 3, generator=g) * 4).to(dev)
    rd = F.normalize(torch.randn(R, 3, generator=g), dim=-1).to(dev)
    ri = torch.sort(torch.randint(R, (N,), generator=g)).values.to(dev)
    ts = (torch.rand(N, generator=g) * 6).to(dev)
    te = ts + torch.rand(N, generator=g).to(dev) * 0.01
    x, dirs = ops.packed_points(ri, ts, te, ro, rd, want_dirs=True)
    ref = ro[ri] + rd[ri] * (ts + te)[:, None] / 2.0  # src/render/rendering.py:58-84
    assert torch.equal(x, ref) and torch.equal(dirs, rd[ri])
    x2, none = ops.packed_points(ri, ts, te, ro, rd)
    assert torch.equal(x2, ref) and none is None
    x0, _ = ops.packed_points(ri[:0], ts[:0], te[:0], ro, rd)
    assert x0.shape == (0, 3)


# ------------------------------------------------------------------ engine vs drop-in
def _scene(R, seed, H=64, W=64, n_views=6):
    from fsnerf_b200 import synthetic as syn
    poses, imgs, focal = syn.make_views(n_views, H, W, seed=42)
    o = np.concatenate([syn.camera_rays(p, H, W, focal)[0].reshape(-1, 3) for p in poses])
    d = np.concatenate([syn.camera_rays(p, H, W, focal)[1].reshape(-1, 3) for p in poses])
    gt = imgs.reshape(-1, 3)
    rng = np.random.default_rng(seed)
    ids = rng.permutation(len(o))[:R] if R else rng.permutation(len(o))
    return o[ids].astype(np.float32), d[ids].astype(np.float32), gt[ids].astype(np.float32)


def _pair(dev, res=128, step=5e-3, bump=3.0):
    """drop-in model + estimator and an engine with the same weights (seed 42, sigma.bias + bump)"""
    from fsnerf_b200.core.models import NeRF
    from fsnerf_b200.engine import HotPath
    from fsnerf_b200.render.rendering import OccGridEstimator
    torch.manual_seed(42)
    model = NeRF(3, 3, 8, 256, [4], **KW).to(dev)
    with torch.no_grad():
        model.sigma.bias += bump
    est = OccGridEstimator(AABB, resolution=res, levels=1).to(dev)
    hp = HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=res, render_step_size=step, device=dev)
    hp.load_state_dict(0, model.state_dict())
    return model, est, hp


def _check_adam_step(ours, ref, lr, name):
    """as tests/test_gpu_train.py: Adam's first step moves every weight by ~ +-lr; entries with a ~0
    gradient may flip sign (2*lr apart), everything else must agree"""
    diff = (ours - ref).abs()
    assert diff.max().item() <= 2.05 * lr, name
    assert (diff > 0.05 * lr).float().mean().item() < 0.05, name


def test_grid_update_is_the_estimators_and_rank_independent(dev):
    from fsnerf_b200.engine import HotPath, grid_seed
    model, est, hp = _pair(dev, res=64, bump=0.0)  # seed-42 densities: a partly occupied grid
    hp2 = HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=64, device=dev, seed=42)
    hp2.load_state_dict(0, model.state_dict())
    for k in (0, 16):  # warm-up (every cell) and, past warmup_steps=8, the random subset
        est.train()
        gen = torch.Generator(device=dev).manual_seed(grid_seed(42, k))
        est.update_every_n_steps(step=k, occ_eval_fn=lambda x: model(x) * 5e-3, occ_thre=1e-2, warmup_steps=8,
                                 generator=gen)
        for h in (hp, hp2):
            h._grid_gen.manual_seed(grid_seed(42, k))
            h.estimator.update_every_n_steps(step=k, occ_eval_fn=h._occ_eval, occ_thre=1e-2, warmup_steps=8,
                                             generator=h._grid_gen)
        assert torch.equal(hp.estimator.occs, hp2.estimator.occs)
        assert torch.equal(hp.estimator.binaries, hp2.estimator.binaries)
        assert torch.equal(hp.estimator.occs, est.occs) and torch.equal(hp.estimator.binaries, est.binaries)
    assert 0 < int(est.binaries.sum()) < 64 ** 3
    from fsnerf_b200._lib import FsnerfError
    with pytest.raises(FsnerfError, match="occ_reg"):
        o, d, gt = _scene(64, 0)
        cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
        hp.train_step(cu(o), cu(d), cu(gt), occ_reg=(0.5, 2.0, "linear"))
    with pytest.raises(FsnerfError, match="roi_aabb"):
        HotPath(sampler="occgrid", device=dev)


def test_engine_step_matches_dropin_step(dev):
    from fsnerf_b200.render.rendering import render_rays
    R, step = 1024, 5e-3
    model, est, hp = _pair(dev)
    hp.update_grid(0)
    est.occs.copy_(hp.estimator.occs)
    est.binaries.copy_(hp.estimator.binaries)
    o, d, gt = _scene(R, 1)
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    ro, rd, gt = cu(o), cu(d), cu(gt)
    u = torch.rand(R, device=dev)
    model.train(); est.train()

    def sigma_fn(t_starts, t_ends, ray_indices):
        x = ro[ray_indices] + rd[ray_indices] * (t_starts + t_ends)[:, None] / 2.0
        return model(x).squeeze(-1)

    est.set_uniforms(u)
    ri_d, ts_d, te_d = est.sampling(ro, rd, sigma_fn=sigma_fn, render_step_size=step, stratified=True,
                                    near_plane=0.0, far_plane=1e10)
    fo = hp._forward_occgrid(ro, rd, u, train=True)  # the training forward, as the drop-in's under grad
    assert fo["M"] > 1000 and fo["M"] < hp.last_counts[0]
    assert torch.equal(fo["ri"], ri_d) and torch.equal(fo["ts"], ts_d) and torch.equal(fo["te"], te_d)
    est.set_uniforms(u)
    (rgb, op, dp, extras), ri2, tv = render_rays(ro, rd, est, model, train=True, white_bkgd=True,
                                                 render_step_size=step, device=dev)
    assert torch.equal(ri2, ri_d)
    assert torch.equal(fo["rgb"], rgb.detach()) and torch.equal(fo["opacity"], op.detach())
    assert torch.equal(fo["depth"], dp.detach())
    loss = F.mse_loss(rgb, gt)
    loss.backward()
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    opt.step()
    ls = hp.train_step(ro, rd, gt, u_strat=u, lr=5e-4)
    assert abs(ls[0].item() / (3 * R) - loss.item()) <= 1e-6 * loss.item()
    g_ref = model._last_flat_grad
    for (off, n), name in zip(hp.layout, hp.names):
        a, b = hp.grads[off:off + n].double(), g_ref[off:off + n].double()
        assert ((a - b).norm() / b.norm().clamp_min(1e-30)).item() <= 1e-5, name
    assert hp.step == 1
    for (off, n), name in zip(hp.layout, hp.names):
        _check_adam_step(hp.params[off:off + n].cpu(), model.flat_parameters()[off:off + n].detach().cpu(), 5e-4,
                         name)


def test_empty_grid_and_single_survivor(dev):
    from fsnerf_b200.core.models import NeRF
    from fsnerf_b200.engine import HotPath
    from fsnerf_b200.render.rendering import OccGridEstimator, render_rays
    _, _, hp = _pair(dev, res=32)
    o, d, gt = _scene(512, 2)
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    ro, rd, gt = cu(o), cu(d), cu(gt)
    p0 = hp.params.clone()
    ls = hp.train_step(ro, rd, gt)  # k = 0: the grid is still empty
    assert hp.last_counts == (0, 0) and hp.step == 0
    assert torch.equal(hp.params, p0) and not bool(hp.m.any()) and not bool(hp.v.any())
    assert abs(ls[0].item() - float(((1.0 - gt) ** 2).sum())) <= 1e-5 * float(((1.0 - gt) ** 2).sum())
    assert int(hp.estimator.binaries.sum()) > 0  # the step-0 update filled it
    rgb, op, dp = hp.render(ro, rd)
    assert hp.last_counts[1] > 1000 and float(op.max()) > 0
    hp.train_step(ro, rd, gt)
    assert hp.step == 1 and not torch.equal(hp.params, p0)
    # exactly one survivor: render_rays' background fallback (src/render/rendering.py:97-103), no Adam step
    box = [-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]
    hp1 = HotPath(sampler="occgrid", roi_aabb=box, grid_resolution=4, render_step_size=0.5, device=dev)
    hp1.estimator.binaries[0, 2, 2, 0] = True
    o = torch.tensor([[0.25, 0.25, 3.0], [0.9, 0.9, 3.0]], device=dev)
    d = torch.tensor([[0.0, 0.0, -1.0], [0.0, 0.0, -1.0]], device=dev)
    rgb, op, dp = hp1.render(o, d)
    assert hp1.last_counts == (1, 1)
    assert torch.equal(rgb, torch.ones(2, 3, device=dev)) and not bool(dp.any()) and not bool(op.any())
    torch.manual_seed(42)
    model = NeRF(3, 3, 8, 256, [4], **KW).to(dev)
    est = OccGridEstimator(box, resolution=4, levels=1).to(dev)
    est.binaries.copy_(hp1.estimator.binaries)
    est.eval()
    with torch.no_grad():
        (rgb_d, _, dp_d, extras), _, _ = render_rays(o, d, est, model, train=False, white_bkgd=True,
                                                     render_step_size=0.5, device=dev)
    assert extras is None and torch.equal(rgb, rgb_d) and torch.equal(dp, dp_d)
    p1 = hp1.params.clone()
    hp1.train_step(o, d, torch.zeros(2, 3, device=dev), u_strat=torch.zeros(2, device=dev))
    assert hp1.last_counts == (1, 1) and hp1.step == 0 and torch.equal(hp1.params, p1)


def test_render_matches_dropin(dev):
    from fsnerf_b200.render.rendering import render_rays
    model, est, hp = _pair(dev)
    hp.update_grid(0)
    est.occs.copy_(hp.estimator.occs)
    est.binaries.copy_(hp.estimator.binaries)
    o, d, _ = _scene(3000, 3)
    ro, rd = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    model.eval(); est.eval()
    with torch.no_grad():
        (rgb, op, dp, _), _, _ = render_rays(ro, rd, est, model, train=False, white_bkgd=True,
                                             render_step_size=5e-3, device=dev)
    rgb_e, op_e, dp_e = hp.render(ro, rd)
    assert hp.last_counts[1] > 10000
    assert torch.equal(rgb_e, rgb) and torch.equal(op_e, op) and torch.equal(dp_e, dp)


# ------------------------------------------------------------------ training
def train_both(dev, steps=300, batch=1024, seed=0):
    """The drop-in loop (examples/train_dropin.py --sampler occgrid without the regularisers) and the
    engine from the same seed-42 weights and empty grid on the synthetic scene.
    -> (first, last) mean train PSNR over 10 steps for (drop-in, engine)"""
    from fsnerf_b200.core.models import NeRF
    from fsnerf_b200.engine import HotPath
    from fsnerf_b200.render.rendering import OccGridEstimator, render_rays
    o, d, gt = _scene(0, seed)
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    o, d, gt = cu(o), cu(d), cu(gt)
    step = 5e-3
    torch.manual_seed(42)
    model = NeRF(3, 3, 8, 256, [4], **KW).to(dev)
    est = OccGridEstimator(AABB, resolution=128, levels=1).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    hp = HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=128, render_step_size=step, device=dev)
    ps_d, ps_e = [], []
    n = o.shape[0]
    for k in range(steps):
        a = (k * batch) % (n - batch)
        ro, rd, g = o[a:a + batch], d[a:a + batch], gt[a:a + batch]
        model.train(); est.train()
        (rgb, *_, extras), _, _ = render_rays(ro, rd, est, model, train=True, white_bkgd=True,
                                              render_step_size=step, device=dev)
        if extras is not None:
            loss = F.mse_loss(rgb, g)
            ps_d.append(-10.0 * torch.log10(loss.detach()).item())
            loss.backward()
            opt.step()
            opt.zero_grad()
        est.update_every_n_steps(step=k, occ_eval_fn=lambda x: model(x) * step, occ_thre=1e-2)
        ls = hp.train_step(ro, rd, g)
        if hp.last_counts[1] > 1:
            ps_e.append(HotPath.psnr(ls[0].item(), batch))
    return (float(np.mean(ps_d[:10])), float(np.mean(ps_d[-10:]))), (float(np.mean(ps_e[:10])), float(np.mean(ps_e[-10:])))


def test_training_raises_psnr_like_the_dropin_loop(dev):
    """Measured on one B200 (1000 W), train_both(seed=0, 1, 2): drop-in 6.36 -> 22.02, 6.43 -> 22.45,
    6.42 -> 22.06 dB; engine 6.36 -> 22.37, 6.39 -> 21.83, 6.40 -> 21.86 dB; engine - drop-in at
    the end +0.35, -0.63, -0.20 dB.  The two loops draw different jitter, and float atomics in the
    backward make even a repeated engine run land 0.5 dB apart (21.90 and 22.37 dB for seed 0), so
    the bar is a rise of 12 dB for both and 1.0 dB between them."""
    (d0, d1), (e0, e1) = train_both(dev)
    print(f"drop-in {d0:.2f} -> {d1:.2f} dB, engine {e0:.2f} -> {e1:.2f} dB")
    assert e1 > e0 + 12.0 and d1 > d0 + 12.0
    assert abs(e1 - d1) < 1.0


@pytest.mark.parametrize("n", [2, 4, 8])
def test_data_parallel_occgrid(n):
    """ray-sharded engine step on n GPUs: all-reduced gradient == single-GPU gradient of the same global
    batch, and every rank holds the same grid after an update"""
    if not torch.cuda.is_available() or torch.cuda.device_count() < n:
        pytest.skip(f"needs {n} CUDA devices")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
           "--master-addr", "127.0.0.1", "--master-port", str(29700 + n),
           os.path.join(ROOT, "tools", "dp_check_occgrid.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0
    assert f"occgrid dp{n} vs single GPU" in r.stdout
