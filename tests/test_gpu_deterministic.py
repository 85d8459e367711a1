"""Deterministic mode: the MLP backward (fsnerf_mlp_backward_deterministic), the engine built with
HotPath(deterministic=True) and the drop-in under torch.use_deterministic_algorithms(True) repeat
bit for bit on one GPU."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import mlp as omlp

pytestmark = pytest.mark.gpu
AABB = [-1.5] * 3 + [1.5] * 3
KW = {"pos_fn": {"n_freqs": 10, "log_space": True}, "dir_fn": {"n_freqs": 4, "log_space": True}}


@pytest.fixture(scope="module")
def dev():
    from fsnerf_b200 import ops
    ops.require_device(0)
    return torch.device("cuda:0")


def _unflatten(cfg, flat):
    from fsnerf_b200 import ops
    return {n: flat[o:o + k].cpu() for (o, k), n in zip(ops.mlp_param_layout(cfg), ops.state_dict_names(cfg))}


# ------------------------------------------------------------------ kernel level
@pytest.mark.parametrize("P,seed,scale", [(4096 * 192, 11, 1.0), (54321, 12, 1.0), (300, 13, 3.0)])
def test_backward_is_bitwise_reproducible(dev, P, seed, scale):
    """4096 x 192: the fine pass of a C2 step; 54 321: not a multiple of the 128-sample tile; 300: fewer
    tiles than dgrad CTAs.  Ten runs, each on a workspace filled with garbage and after a default-mode
    backward that disturbs L2 and timing.  (Weights and the incoherent d_out as in
    tests/test_gpu_kernels.py::test_mlp_backward_weight_grads.)"""
    from fsnerf_b200 import ops
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict(seed=seed)
    sd["sigma.weight"] = sd["sigma.weight"] * scale
    params = ops.flatten_state_dict(cfg, sd, dev)
    packed = ops.mlp_pack(cfg, params)
    g = torch.Generator().manual_seed(P)
    x = (torch.rand(P, 3, generator=g) * 2 - 1) * 2.5
    d = F.normalize(torch.randn(P, 3, generator=g), dim=-1)
    d_out = torch.randn(P, 4, generator=g).to(dev)
    stash = torch.empty(ops.mlp_stash_bytes(cfg, P), dtype=torch.uint8, device=dev)
    out = ops.mlp_forward(cfg, params, packed, x=x.to(dev), dirs=d.to(dev), stash=stash)
    ws_def = torch.empty(ops.mlp_bwd_workspace_bytes(cfg, P), dtype=torch.uint8, device=dev)
    ws_det = torch.empty(ops.mlp_bwd_workspace_bytes(cfg, P, deterministic=True), dtype=torch.uint8, device=dev)
    assert ws_det.numel() > ws_def.numel()
    runs, defaults = [], []
    for _ in range(10):
        ws_det.random_(0, 256)
        g_def = torch.zeros_like(params)
        ops.mlp_backward(cfg, params, packed, P, stash, out, d_out, g_def, ws_def)
        defaults.append(g_def)
        g_det = torch.zeros_like(params)
        ops.mlp_backward(cfg, params, packed, P, stash, out, d_out, g_det, ws_det, deterministic=True)
        runs.append(g_det)
    torch.cuda.synchronize()
    for r in runs[1:]:
        assert torch.equal(r, runs[0])
    # the same sums in another order: per tensor within 1e-5 of the default, or, where the default's
    # own run-to-run spread is larger (long fp32 accumulations with cancellation), within twice that
    rel = lambda a, b: ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()  # noqa: E731
    ours = _unflatten(cfg, runs[0])
    dflt = [_unflatten(cfg, g) for g in defaults]
    for n in ours:
        spread = max(rel(dd[n], dflt[0][n]) for dd in dflt[1:])
        worst = max(rel(ours[n], dd[n]) for dd in dflt)
        print(f"{n}: deterministic vs default {worst:.2e}, default run to run {spread:.2e}")
        assert worst <= max(1e-5, 2 * spread), (n, worst, spread)
    # accumulated into, once per element: pre-filled grads give g0 + det(zeros) bit for bit
    g0 = torch.randn(params.numel(), generator=g).to(dev)
    pre = g0.clone()
    ops.mlp_backward(cfg, params, packed, P, stash, out, d_out, pre, ws_det, deterministic=True)
    assert torch.equal(pre, g0 + runs[0])
    if P > 60000:
        return  # (the CPU oracle at C2 size takes minutes; the two smaller sizes cover it)
    # the fp32 oracle on bf16 operands, as tests/test_gpu_kernels.py::test_mlp_backward_weight_grads
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref_out = omlp.nerf_forward_bf16emu(sdr, x, d)
    names = list(sdr.keys())
    ref = dict(zip(names, torch.autograd.grad((ref_out * d_out.cpu()).sum(), [sdr[n] for n in names])))
    for n in names:
        rel = ((ours[n].reshape(-1).double() - ref[n].reshape(-1).double()).norm() /
               ref[n].double().norm().clamp_min(1e-12)).item()
        assert rel < 8e-3, (n, rel)


def test_adam_step_reg_deterministic_matches_default(dev):
    from fsnerf_b200 import ops
    cfg = ops.make_cfg()
    params = ops.flatten_state_dict(cfg, omlp.init_state_dict(seed=4), dev)
    grads = torch.randn(params.numel(), generator=torch.Generator().manual_seed(4)).to(dev) * 1e-3
    segs = ops.reg_segments(cfg)
    res = []
    for det in (False, True, True):
        p, m, v = params.clone(), torch.zeros_like(params), torch.zeros_like(params)
        sums = torch.full((len(segs),), 7.0, device=dev)
        ops.adam_step_reg(p, grads, m, v, 5e-4, 1, "l2", 1e-3, segs, sums, deterministic=det)
        res.append((p, m, v, sums))
    assert all(torch.equal(a, b) for a, b in zip(res[1], res[2]))
    assert torch.allclose(res[0][3], res[1][3], rtol=1e-5)
    assert (res[0][0] - res[1][0]).abs().max().item() < 1e-6


# ------------------------------------------------------------------ engine
def _scene(R, seed, H=64, W=64, n_views=6):
    from fsnerf_b200 import synthetic as syn
    poses, imgs, focal = syn.make_views(n_views, H, W, seed=42)
    o = np.concatenate([syn.camera_rays(p, H, W, focal)[0].reshape(-1, 3) for p in poses])
    d = np.concatenate([syn.camera_rays(p, H, W, focal)[1].reshape(-1, 3) for p in poses])
    gt = imgs.reshape(-1, 3)
    rng = np.random.default_rng(seed)
    ids = rng.permutation(len(o))[:R] if R else rng.permutation(len(o))
    return o[ids].astype(np.float32), d[ids].astype(np.float32), gt[ids].astype(np.float32)


def _lockstep(dev, make, steps, batch, train_kw, extra_state=lambda hp: []):
    """two engines from the same seed, stepped alternately on the same rays; every 10 steps the
    parameters, Adam moments, renders (and extra_state) must be bitwise equal.  The loss sums are
    atomics of block partials (only reported, never fed back): compared at 1e-6 relative."""
    o, d, gt = _scene(0, 0)
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    o, d, gt = cu(o), cu(d), cu(gt)
    a, b = make(), make()
    n = o.shape[0]
    ro_eval, rd_eval = o[:2048], d[:2048]
    for k in range(steps):
        s = (k * batch) % (n - batch)
        la = a.train_step(o[s:s + batch], d[s:s + batch], gt[s:s + batch], **train_kw).clone()
        lb = b.train_step(o[s:s + batch], d[s:s + batch], gt[s:s + batch], **train_kw).clone()
        torch.testing.assert_close(la, lb, rtol=1e-6, atol=0)
        if k % 10 == 9:
            assert torch.equal(a.params, b.params), k
            assert torch.equal(a.m, b.m) and torch.equal(a.v, b.v), k
            for x, y in zip(extra_state(a), extra_state(b)):
                assert torch.equal(x, y), k
            for x, y in zip(a.render(ro_eval, rd_eval), b.render(ro_eval, rd_eval)):
                assert torch.equal(x, y), k
    assert a.step > 0 and not torch.equal(a.m, torch.zeros_like(a.m))
    return a


def test_engine_hierarchical_repeats_bit_for_bit(dev):
    from fsnerf_b200.engine import HotPath
    make = lambda: HotPath(device=dev, seed=42, deterministic=True)  # noqa: E731
    _lockstep(dev, make, 100, 1024, dict(occ_reg=(0.5, 2.0, "linear"), weight_reg=("l2", 1e-4)))


def test_engine_occgrid_repeats_bit_for_bit(dev):
    from fsnerf_b200.engine import HotPath
    make = lambda: HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=128, device=dev, seed=42,  # noqa: E731
                           deterministic=True)
    hp = _lockstep(dev, make, 100, 1024, dict(weight_reg=("l2", 1e-4)),
                   extra_state=lambda h: [h.estimator.occs, h.estimator.binaries])
    assert int(hp.estimator.binaries.sum()) > 0 and hp.k == 100  # seven grid updates (every 16th step)


def test_deterministic_engine_trains_like_the_dropin_loop(dev):
    """as tests/test_gpu_occgrid_engine.py::test_training_raises_psnr_like_the_dropin_loop, with the
    engine in deterministic mode: a rise of 12 dB and within 1.0 dB of the drop-in loop"""
    from fsnerf_b200.core.models import NeRF
    from fsnerf_b200.engine import HotPath
    from fsnerf_b200.render.rendering import OccGridEstimator, render_rays
    o, d, gt = _scene(0, 0)
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    o, d, gt = cu(o), cu(d), cu(gt)
    step, batch = 5e-3, 1024
    torch.manual_seed(42)
    model = NeRF(3, 3, 8, 256, [4], **KW).to(dev)
    est = OccGridEstimator(AABB, resolution=128, levels=1).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    hp = HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=128, render_step_size=step, device=dev,
                 deterministic=True)
    ps_d, ps_e = [], []
    n = o.shape[0]
    for k in range(300):
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
    d0, d1, e0, e1 = (float(np.mean(v)) for v in (ps_d[:10], ps_d[-10:], ps_e[:10], ps_e[-10:]))
    print(f"drop-in {d0:.2f} -> {d1:.2f} dB, deterministic engine {e0:.2f} -> {e1:.2f} dB")
    assert e1 > e0 + 12.0 and d1 > d0 + 12.0
    assert abs(e1 - d1) < 1.0


# ------------------------------------------------------------------ drop-in
def _reference_loop(dev, occgrid, steps=30, batch=1024):
    """the reference's loop (render_rays + F.mse_loss + backward + torch.optim.Adam) from
    torch.manual_seed(42) -> every parameter after `steps` steps"""
    from fsnerf_b200.core.models import NeRF
    from fsnerf_b200.render.rendering import HierarchicalEstimator, OccGridEstimator, render_rays
    o, d, gt = _scene(0, 1)
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    o, d, gt = cu(o), cu(d), cu(gt)
    torch.manual_seed(42)
    model = NeRF(3, 3, 8, 256, [4], **KW).to(dev)
    params = list(model.parameters())
    if occgrid:
        est = OccGridEstimator(AABB, resolution=128, levels=1).to(dev)
    else:
        coarse = NeRF(3, 3, 8, 256, [4], **KW).to(dev)
        est = HierarchicalEstimator(near=2.0, far=6.0, n_coarse=64, n_fine=128, proposal_model=coarse)
        params += list(coarse.parameters())
    opt = torch.optim.Adam(params, lr=5e-4)
    n = o.shape[0]
    for k in range(steps):
        a = (k * batch) % (n - batch)
        model.train(); est.train()
        (rgb, *_, extras), _, _ = render_rays(o[a:a + batch], d[a:a + batch], est, model, train=True,
                                              white_bkgd=True, render_step_size=5e-3, device=dev)
        if extras is not None:
            loss = F.mse_loss(rgb, gt[a:a + batch])
            if "rgb_coarse" in extras:
                loss = loss + F.mse_loss(extras["rgb_coarse"], gt[a:a + batch])
            loss.backward()
            opt.step()
            opt.zero_grad()
        est.update_every_n_steps(step=k, occ_eval_fn=lambda x: model(x) * 5e-3, occ_thre=1e-2)
    return [p.detach().clone() for p in params]


@pytest.mark.parametrize("occgrid", [False, True], ids=["hierarchical", "occgrid"])
def test_dropin_under_torch_deterministic_algorithms(dev, occgrid):
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        first = _reference_loop(dev, occgrid)
        second = _reference_loop(dev, occgrid)
    finally:
        torch.use_deterministic_algorithms(was)
    assert len(first) == len(second) > 0
    for p, q in zip(first, second):
        assert torch.equal(p, q)
