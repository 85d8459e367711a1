"""GPU parity tests (run on the B200 box): each CUDA kernel, called through the
C ABI, against the CPU oracle on the same seeded inputs.
Bars (BASELINE.json north_star): integer/index outputs bit-exact; fp32 kernels
to ~1e-5; the bf16 MLP within 1e-3 absolute on per-ray outputs."""
import numpy as np
import pytest
import torch

from oracle import rays as orays, sampling as osamp, compositing as ocomp, mlp as omlp, render as orender

pytestmark = pytest.mark.gpu
f32 = np.float32


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fsnerf_b200 import ops
    ops.require_device(0)
    return torch.device("cuda:0")


def cu(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ----------------------------------------------------------------- rays
def test_gen_rays_bit_exact(dev, golden):
    from fsnerf_b200 import ops
    g = golden("reference_rays.npz")
    H, W, f = int(g["hwf2"][0]), int(g["hwf2"][1]), float(g["hwf2"][2])
    poses = np.stack([g["pose2"], g["pose"]]).astype(f32)
    o, d, _ = ops.gen_rays(cu(poses, dev), H, W, f, first_id=0, n_rays=2 * H * W)
    o_ref = np.concatenate([orays.get_rays(p, (H, W, f))[0].reshape(-1, 3) for p in poses])
    d_ref = np.concatenate([orays.get_rays(p, (H, W, f))[1].reshape(-1, 3) for p in poses])
    np.testing.assert_array_equal(o.cpu().numpy(), o_ref)
    np.testing.assert_array_equal(d.cpu().numpy(), d_ref)  # same op order -> bit-exact
    np.testing.assert_allclose(d.cpu().numpy()[:H * W].reshape(H, W, 3), g["rd2"], atol=1.2e-7)
    # pixel-id bookkeeping + rgb gather + 3x4 poses
    rng = np.random.default_rng(0)
    ids = rng.permutation(2 * H * W)[:301].astype(np.int64)
    imgs = rng.random((2, H, W, 3), dtype=f32)
    o2, d2, rgb = ops.gen_rays(cu(poses[:, :3], dev), H, W, f, pixel_ids=cu(ids, dev), images=cu(imgs, dev))
    np.testing.assert_array_equal(d2.cpu().numpy(), d_ref[ids])
    np.testing.assert_array_equal(o2.cpu().numpy(), o_ref[ids])
    np.testing.assert_array_equal(rgb.cpu().numpy(), imgs.reshape(-1, 3)[ids])
    # NDC (fused and standalone)
    no_ref, nd_ref = orays.to_ndc(o_ref, d_ref, (H, W, f), 1.0)
    o3, d3, _ = ops.gen_rays(cu(poses, dev), H, W, f, first_id=0, n_rays=2 * H * W, ndc=True)
    np.testing.assert_array_equal(o3.cpu().numpy(), no_ref)
    np.testing.assert_array_equal(d3.cpu().numpy(), nd_ref)
    o4, d4 = ops.to_ndc(o, d, H, W, f, 1.0)
    np.testing.assert_array_equal(o4.cpu().numpy(), no_ref)
    np.testing.assert_allclose(o4.cpu().numpy()[:H * W], g["ndc_o2"], rtol=2e-6, atol=2e-6)


def test_stratified_bit_exact(dev):
    from fsnerf_b200 import ops
    rng = np.random.default_rng(1)
    for R, S, near, far in ((257, 64, 2.0, 6.0), (5, 7, 0.0, 1.0), (3, 1, 0.5, 2.5)):
        u = rng.random((R, S), dtype=f32)
        ts, te = ops.sample_stratified(R, S, near, far, cu(u, dev))
        z = osamp.stratified(R, S, near, far, u)
        ts_ref, te_ref = osamp.intervals_from_points(z, far)
        np.testing.assert_array_equal(ts.cpu().numpy(), ts_ref)
        np.testing.assert_array_equal(te.cpu().numpy(), te_ref)
        ts, te = ops.sample_stratified(R, S, near, far, None, device=dev)
        np.testing.assert_array_equal(ts.cpu().numpy(), osamp.stratified(R, S, near, far))
    ts, te = ops.sample_stratified(0, 8, 0.0, 1.0, None, device=dev)
    assert ts.shape == (0, 8)


@pytest.mark.parametrize("R,Sc,Sf", [(515, 64, 128), (33, 8, 16), (17, 33, 7), (9, 128, 64), (4, 3, 5)])
def test_sample_pdf_bit_exact(dev, R, Sc, Sf):
    from fsnerf_b200 import ops
    rng = np.random.default_rng(2)
    z = osamp.stratified(R, Sc, 2.0, 6.0, rng.random((R, Sc), dtype=f32))
    w = rng.random((R, Sc), dtype=f32) ** 6
    w[0] = 0
    w[3 % R] -= 0.5  # negative weights (raw sigma < 0) are clamped at 0
    if Sc > 8:
        w[1, 1:-1] = 0
        w[1, Sc // 2] = 1
    u = rng.random((R, Sf), dtype=f32)
    u[2 % R, :3] = [0.0, 0.99999994, 0.5]
    for uu in (u, None):
        ref = osamp.sample_pdf(z, w, Sf, 6.0, uu)
        ts, te, smp, inds, perm = ops.sample_pdf(cu(z, dev), cu(w, dev), Sf, 6.0,
                                                 None if uu is None else cu(uu, dev))
        np.testing.assert_array_equal(inds.cpu().numpy(), ref["inds"])      # searchsorted: bit-exact
        np.testing.assert_array_equal(perm.cpu().numpy(), ref["perm"])      # sort permutation: bit-exact
        np.testing.assert_array_equal(smp.cpu().numpy(), ref["samples"])
        np.testing.assert_array_equal(ts.cpu().numpy(), ref["t_starts"])
        np.testing.assert_array_equal(te.cpu().numpy(), ref["t_ends"])


@pytest.mark.parametrize("seed", [0, 1, 42, 0x9E3779B97F4A7C15, (1 << 64) - 1])
def test_seeded_samplers_bit_exact(dev, seed):
    """In-kernel uniforms: the device stream equals oracle.sampling.rng_uniform bit for bit, and
    the seeded samplers equal the explicit-u ones (and the oracle) fed with that stream."""
    from fsnerf_b200 import ops
    R, Sc, Sf = 515, 64, 128
    n = 70000
    np.testing.assert_array_equal(ops.rng_uniform(n, seed, device=dev).cpu().numpy(), osamp.rng_uniform(seed, n))
    us = osamp.rng_uniform(seed, R * Sc).reshape(R, Sc)
    up = osamp.rng_uniform(seed ^ 0x5555, R * Sf).reshape(R, Sf)
    ts, te = ops.sample_stratified(R, Sc, 2.0, 6.0, device=dev, seed=seed)
    z = osamp.stratified(R, Sc, 2.0, 6.0, us)
    np.testing.assert_array_equal(ts.cpu().numpy(), z)
    ts2, te2 = ops.sample_stratified(R, Sc, 2.0, 6.0, cu(us, dev))
    assert torch.equal(ts, ts2) and torch.equal(te, te2)
    w = np.random.default_rng(5).random((R, Sc), dtype=f32) ** 6
    ref = osamp.sample_pdf(z, w, Sf, 6.0, up)
    got = ops.sample_pdf(ts, cu(w, dev), Sf, 6.0, seed=seed ^ 0x5555)
    for g, k in zip(got, ("t_starts", "t_ends", "samples", "inds", "perm")):
        np.testing.assert_array_equal(g.cpu().numpy(), ref[k])
    with pytest.raises(Exception):
        ops.sample_stratified(R, Sc, 2.0, 6.0, cu(us, dev), seed=1)


def test_engine_default_jitter_is_in_kernel_and_reproducible(dev):
    """train_step without explicit uniforms: no generator launch, a fresh stream every step (the
    weights are held fixed, so a different loss means different jitter), the same streams for
    the same construction seed."""
    from fsnerf_b200.engine import HotPath
    g = torch.Generator().manual_seed(3)
    R = 256
    o = torch.rand(R, 3, generator=g).to(dev) * 0.1
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1).to(dev)
    gt = torch.rand(R, 3, generator=g).to(dev)
    runs = []
    for _ in range(2):
        hp = HotPath(n_coarse=16, n_fine=16, near=2.0, far=6.0, device=dev, seed=7)
        state = torch.cuda.get_rng_state(dev)
        losses = [hp.train_step(o, d, gt, apply_update=False).clone() for _ in range(3)]
        assert torch.equal(state, torch.cuda.get_rng_state(dev))  # torch's device generator untouched
        runs.append(torch.stack(losses).cpu())
    # the loss sums are float atomics (order varies run to run): same stream <=> equal to ~1 ulp,
    # while a different stream moves them in the 4th digit
    torch.testing.assert_close(runs[0], runs[1], rtol=2e-6, atol=0)
    assert (runs[0][0] - runs[0][1]).abs().max() > 1e-4 * runs[0][0].abs().max()


# ----------------------------------------------------------- compositing
def _comp_inputs(R, S, seed, neg_sigma=True):
    g = torch.Generator().manual_seed(seed)
    e = torch.sort(2 + 4 * torch.rand(R, S + 1, generator=g), -1).values
    ts, te = e[:, :-1].contiguous(), e[:, 1:].contiguous()
    raw = torch.rand(R, S, 4, generator=g)
    raw[..., 3] = torch.randn(R, S, generator=g) * 6 + (0 if neg_sigma else 4)
    return raw, ts, te


@pytest.mark.parametrize("R,S", [(1000, 192), (77, 64), (13, 1), (9, 33), (5, 300), (3, 256)])
@pytest.mark.parametrize("flags", [0, 1, 2, 4, 7])
def test_composite_forward_backward(dev, R, S, flags):
    from fsnerf_b200 import ops
    raw, ts, te = _comp_inputs(R, S, seed=R + S)
    if flags & 4:
        raw[..., 3] = raw[..., 3].abs()  # product form: keep 1-alpha positive
    g = torch.Generator().manual_seed(7)
    bk = torch.tensor([1.0, 0.5, 0.25])
    ds = 1 + torch.rand(R, generator=g)
    kw = dict(sigma_relu=bool(flags & 1), normalize_depth=not (flags & 2), product_trans=bool(flags & 4))
    raw_r = raw.clone().requires_grad_(True)
    bk_r = bk.clone().requires_grad_(True)
    rgb, op, dp, w, al, tr = ocomp.composite_dense(raw_r, ts, te, bk_r, delta_scale=ds, **kw)
    out = ops.composite_forward(cu(raw.numpy(), dev), cu(ts.numpy(), dev), cu(te.numpy(), dev),
                                bkgd=bk.to(dev), delta_scale=ds.to(dev), flags=flags, extras=True)
    names = ["rgb", "opacity", "depth", "weights", "alphas", "trans"]
    for n, a, b in zip(names, out, (rgb, op, dp, w, al, tr)):
        tol = 2e-5 * max(1.0, float(b.detach().abs().max()))
        assert (a.cpu() - b.detach()).abs().max().item() <= tol, n
    if S > 512:
        return
    d_rgb = torch.randn(R, 3, generator=g)
    d_op = torch.randn(R, 1, generator=g)
    d_dp = torch.randn(R, 1, generator=g) * (0.0 if not (flags & 2) and op.detach().abs().min() < 1e-3 else 1.0)
    d_w = torch.randn(R, S, generator=g)
    loss = (rgb * d_rgb).sum() + (op * d_op).sum() + (dp * d_dp).sum() + (w * d_w).sum()
    g_raw, g_bk = torch.autograd.grad(loss, [raw_r, bk_r])
    d_raw, d_bk = ops.composite_backward(cu(raw.numpy(), dev), cu(ts.numpy(), dev), cu(te.numpy(), dev),
                                         d_rgb.to(dev), d_op.to(dev), d_dp.to(dev), d_w.to(dev),
                                         bkgd=bk.to(dev), delta_scale=ds.to(dev), flags=flags,
                                         want_d_bkgd=True)
    scale = max(1.0, g_raw.abs().max().item())
    assert (d_raw.cpu() - g_raw).abs().max().item() <= 1e-4 * scale
    assert (d_bk.cpu() - g_bk).abs().max().item() <= 1e-4 * max(1.0, g_bk.abs().max().item())


def test_composite_matches_reference_fixture(dev, golden):
    """sigmas/rgbs of the reference-generated render fixture -> our compositor."""
    from fsnerf_b200 import ops
    g = golden("reference_render.npz")
    ts, te = g["t_starts"], g["t_ends"]
    sd = omlp.init_state_dict()
    sd["sigma.weight"] = sd["sigma.weight"] * float(g["sigma_w_scale"])
    sd["sigma.bias"] = sd["sigma.bias"] + float(g["sigma_b_add"])
    raw = orender.query_mlp(sd, torch.from_numpy(g["rays_o"]), torch.from_numpy(g["rays_d"]),
                            torch.from_numpy(ts), torch.from_numpy(te))
    for tag, bk in (("b", None), ("w", torch.ones(3, device=dev))):
        rgb, op, dp, w, _, _ = ops.composite_forward(raw.to(dev), cu(ts, dev), cu(te, dev), bkgd=bk)
        np.testing.assert_allclose(rgb.cpu().numpy(), g[f"rgb_{tag}"], atol=5e-6)
        np.testing.assert_allclose(op.cpu().numpy(), g[f"opacity_{tag}"], atol=5e-6)
        np.testing.assert_allclose(dp.cpu().numpy(), g[f"depth_{tag}"], rtol=2e-5, atol=1e-5)
        np.testing.assert_allclose(w.cpu().numpy().reshape(-1), g[f"weights_{tag}"], atol=5e-6)


# ------------------------------------------------------------------- MLP
def _flat_params(sd, dev):
    from fsnerf_b200 import ops
    return ops.flatten_state_dict(ops.make_cfg(), sd, dev)


def test_mlp_forward_points(dev, golden):
    """model(x, dirs) and model(x) against the reference outputs (golden) —
    bf16 operands / fp32 accumulate vs the fp32 reference."""
    from fsnerf_b200 import ops
    g = golden("reference_mlp.npz")
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict()
    params = _flat_params(sd, dev)
    packed = ops.mlp_pack(cfg, params)
    out = ops.mlp_forward(cfg, params, packed, x=cu(g["x"], dev), dirs=cu(g["d"], dev))
    torch.cuda.synchronize()
    err = np.abs(out.cpu().numpy() - g["out"])
    print("mlp fwd max err rgb/sigma:", err[:, :3].max(), err[:, 3].max())
    assert err[:, :3].max() < 2e-3 and err[:, 3].max() < 4e-3
    sig = ops.mlp_forward(cfg, params, packed, x=cu(g["x"], dev), density_only=True)
    assert np.abs(sig.cpu().numpy() - g["sigma_only"][:, 0]).max() < 4e-3


@pytest.mark.parametrize("P", [1, 127, 128, 129, 5000, 128 * 300 + 17])
def test_mlp_forward_sizes(dev, P):
    """ragged tile counts; bf16-emulated oracle bound (tight) + fp32 oracle bound."""
    from fsnerf_b200 import ops
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict(seed=5)
    params = _flat_params(sd, dev)
    packed = ops.mlp_pack(cfg, params)
    g = torch.Generator().manual_seed(P)
    x = (torch.rand(P, 3, generator=g) * 2 - 1) * 3
    d = torch.nn.functional.normalize(torch.randn(P, 3, generator=g), dim=-1)
    mp = torch.rand(63, generator=g)
    md = torch.rand(27, generator=g)
    out = ops.mlp_forward(cfg, params, packed, x=x.to(dev), dirs=d.to(dev), mask_pos=mp.to(dev),
                          mask_dir=md.to(dev))
    ref = omlp.nerf_forward(sd, x, d, mask_pos=mp, mask_dir=md)
    err = (out.cpu() - ref).abs()
    assert err[:, :3].max() < 2e-3 and err[:, 3].max() < 4e-3, (err[:, :3].max(), err[:, 3].max())


def test_mlp_forward_rays_and_stash(dev):
    from fsnerf_b200 import ops
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict(seed=6)
    params = _flat_params(sd, dev)
    packed = ops.mlp_pack(cfg, params)
    R, S = 37, 48
    g = torch.Generator().manual_seed(0)
    o = torch.tensor([0.0, 0, 4]) + 0.1 * torch.randn(R, 3, generator=g)
    d = torch.nn.functional.normalize(torch.tensor([0.0, 0, -1]) + 0.2 * torch.randn(R, 3, generator=g), dim=-1)
    e = torch.sort(2 + 4 * torch.rand(R, S + 1, generator=g), -1).values
    ts, te = e[:, :-1].contiguous(), e[:, 1:].contiguous()
    ref = orender.query_mlp(sd, o, d, ts, te).reshape(-1, 4)
    out = ops.mlp_forward(cfg, params, packed, rays_o=o.to(dev), rays_d=d.to(dev),
                          t_starts=ts.to(dev), t_ends=te.to(dev))
    err = (out.cpu() - ref).abs()
    assert err[:, :3].max() < 2e-3 and err[:, 3].max() < 4e-3
    stash = torch.zeros(ops.mlp_stash_bytes(cfg, R * S), dtype=torch.uint8, device=dev)
    out2 = ops.mlp_forward(cfg, params, packed, rays_o=o.to(dev), rays_d=d.to(dev),
                           t_starts=ts.to(dev), t_ends=te.to(dev), stash=stash)
    torch.cuda.synchronize()
    assert torch.equal(out, out2)
    assert stash.view(torch.int16).count_nonzero().item() > 0.5 * stash.numel() / 2 * 0.4


def test_train_step_arithmetic(dev):
    from fsnerf_b200 import ops
    g = torch.Generator().manual_seed(0)
    n = 100003
    p = torch.randn(n, generator=g)
    ref = torch.nn.Parameter(p.clone())
    opt = torch.optim.Adam([ref], lr=5e-4)
    pc, m, v = p.to(dev), torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    for step in range(1, 4):
        gr = torch.randn(n, generator=g)
        ref.grad = gr.clone()
        opt.step()
        ops.adam_step(pc, gr.to(dev), m, v, 5e-4, step)
        assert (pc.cpu() - ref.detach()).abs().max().item() < 5e-7
    rgb, gt = torch.rand(4096, 3, generator=g), torch.rand(4096, 3, generator=g)
    loss_sum = torch.zeros(1, device=dev)
    d = ops.mse_loss_grad(rgb.to(dev), gt.to(dev), 1.0 / rgb.numel(), loss_sum)
    ref_loss = torch.nn.functional.mse_loss(rgb, gt)
    assert abs(loss_sum.item() / rgb.numel() - ref_loss.item()) < 1e-6
    np.testing.assert_allclose(d.cpu().numpy(), (2 * (rgb - gt) / rgb.numel()).numpy(), atol=1e-9)


def _unflatten(cfg, flat):
    from fsnerf_b200 import ops
    return {n: flat[o:o + k].cpu() for (o, k), n in zip(ops.mlp_param_layout(cfg), ops.state_dict_names(cfg))}


@pytest.mark.parametrize("P,seed,scale", [(5000, 11, 1.0), (128 * 311 + 17, 12, 1.0), (300, 13, 3.0)])
def test_mlp_backward_weight_grads(dev, P, seed, scale):
    """Kernel correctness of the backward: per-tensor ||g - g_ref|| / ||g_ref|| against
    the bf16-operand emulation of the same math (oracle.mlp.nerf_forward_bf16emu), with
    an adversarial *incoherent* d_out (independent random per sample).  The fp32-reference
    bar (1e-2, BASELINE.json north_star) is checked on the real rendering loss in
    tests/test_gpu_train.py: with incoherent d_out every ReLU-mask flip caused by bf16
    forward noise shows up undamped (relative error ~ sqrt(flipped fraction))."""
    from fsnerf_b200 import ops
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict(seed=seed)
    sd["sigma.weight"] = sd["sigma.weight"] * scale
    params = ops.flatten_state_dict(cfg, sd, dev)
    packed = ops.mlp_pack(cfg, params)
    g = torch.Generator().manual_seed(P)
    x = (torch.rand(P, 3, generator=g) * 2 - 1) * 2.5
    d = torch.nn.functional.normalize(torch.randn(P, 3, generator=g), dim=-1)
    d_out = torch.randn(P, 4, generator=g)
    stash = torch.empty(ops.mlp_stash_bytes(cfg, P), dtype=torch.uint8, device=dev)
    out = ops.mlp_forward(cfg, params, packed, x=x.to(dev), dirs=d.to(dev), stash=stash)
    grads = torch.zeros_like(params)
    ws = torch.empty(ops.mlp_bwd_workspace_bytes(cfg, P), dtype=torch.uint8, device=dev)
    ops.mlp_backward(cfg, params, packed, P, stash, out, d_out.to(dev), grads, ws)
    torch.cuda.synchronize()
    ours = _unflatten(cfg, grads)
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref_out = omlp.nerf_forward_bf16emu(sdr, x, d)
    assert (ref_out.detach() - out.cpu()).abs().max().item() < 3e-4  # forward vs emulation: tight
    names = list(sdr.keys())
    ref = dict(zip(names, torch.autograd.grad((ref_out * d_out).sum(), [sdr[n] for n in names])))
    rels = {}
    for n in names:
        rels[n] = ((ours[n].reshape(-1).double() - ref[n].reshape(-1).double()).norm() /
                   ref[n].double().norm().clamp_min(1e-12)).item()
    print("relative weight-grad errors:", {k: round(v, 5) for k, v in rels.items()})
    for n in names:
        assert rels[n] < 8e-3, (n, rels[n])
    # calling it twice accumulates (grads are added into)
    ops.mlp_backward(cfg, params, packed, P, stash, out, d_out.to(dev), grads, ws)
    twice = _unflatten(cfg, grads)
    n0 = "layers.3.weight"
    assert ((twice[n0] - 2 * ours[n0]).norm() / (2 * ours[n0]).norm()).item() < 1e-3


# ------------------------------------------------------------------ in-step regularisers (f2)
@pytest.mark.gpu
@pytest.mark.parametrize("R,S,flags,func", [(300, 192, 0, "linear"), (77, 64, 1, "exp"), (9, 33, 4, "linear"),
                                            (5, 300, 2, "exp")])
def test_composite_backward_with_occlusion_reg(dev, R, S, flags, func):
    """occlusion regulariser (src/core/loss.py:26-60) fused into the compositing backward:
    d_raw and the loss value vs autograd of oracle compositing + oracle.regularizers."""
    from fsnerf_b200 import ops
    from oracle import regularizers as oreg
    raw, ts, te = _comp_inputs(R, S, seed=3 * R + S)
    if flags & 4:
        raw[..., 3] = raw[..., 3].abs()
    a, b = (0.5, 2.0) if func == "linear" else (1.5, 0.7)
    kw = dict(sigma_relu=bool(flags & 1), normalize_depth=not (flags & 2), product_trans=bool(flags & 4))
    g = torch.Generator().manual_seed(3)
    d_rgb = torch.randn(R, 3, generator=g)
    raw_r = raw.clone().requires_grad_(True)
    rgb, *_ = ocomp.composite_dense(raw_r, ts, te, None, **kw)
    G = 4 * R  # this launch is one shard of a 4x larger global batch
    occ = oreg.occlusion_reg_dense(raw_r[..., 3], ts, te, a, b, func) * (R / G)
    (g_raw,) = torch.autograd.grad((rgb * d_rgb).sum() + occ, raw_r)
    occ_sum = torch.zeros(1, device=dev)
    d_raw, _ = ops.composite_backward(cu(raw.numpy(), dev), cu(ts.numpy(), dev), cu(te.numpy(), dev),
                                      d_rgb.to(dev), flags=flags, occ=(a, b, func, 1.0 / G, occ_sum))
    assert (d_raw.cpu() - g_raw).abs().max().item() <= 1e-4 * max(1.0, g_raw.abs().max().item())
    assert abs(occ_sum.item() / G - occ.item()) <= 1e-5 * max(1.0, abs(occ.item()))
    with pytest.raises(ValueError):
        ops.composite_backward(cu(raw.numpy(), dev), cu(ts.numpy(), dev), cu(te.numpy(), dev), d_rgb.to(dev),
                               occ=(a, b, "cubic", 1.0, occ_sum))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["l1", "l2"])
def test_adam_with_weight_penalty(dev, mode):
    """weight-norm penalty (src/run-nerf.py:266-279) fused into Adam vs torch.optim.Adam on
    grad + alpha * d(penalty), on the reference's parameter set (golden-pinned coverage)."""
    from fsnerf_b200 import ops
    from oracle import regularizers as oreg
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict(seed=42)
    segs = ops.reg_segments(cfg, 1)
    names = oreg.regularised_names([(k, tuple(v.shape)) for k, v in sd.items()])
    lay = dict(zip(ops.state_dict_names(cfg), ops.mlp_param_layout(cfg)))
    assert segs == [(lay[n][0], lay[n][0] + lay[n][1]) for n in names]
    alpha = 1e-3
    p = ops.flatten_state_dict(cfg, sd, dev)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    sums = torch.zeros(len(segs), device=dev)
    ref = {k: torch.nn.Parameter(t.clone()) for k, t in sd.items()}
    opt = torch.optim.Adam(list(ref.values()), lr=5e-4)
    g = torch.Generator().manual_seed(1)
    for step in range(1, 4):
        grads = {k: 1e-3 * torch.randn(t.shape, generator=g) for k, t in sd.items()}
        pen = oreg.weight_reg(ref, mode)
        pg = torch.autograd.grad(alpha * pen, [ref[n] for n in names])
        for k in ref:
            ref[k].grad = grads[k].clone()
        for n, gg in zip(names, pg):
            ref[n].grad += gg
        flat_g = ops.flatten_state_dict(cfg, grads, dev)
        ops.adam_step_reg(p, flat_g, m, v, 5e-4, step, mode, alpha, segs, sums)
        val = sums.sum().item() if mode == "l1" else sums.sqrt().sum().item()
        assert abs(val - pen.item()) <= 1e-5 * pen.item()
        opt.step()
        ours = _unflatten(cfg, p)
        for k in ref:
            assert (ours[k] - ref[k].detach().reshape(-1)).abs().max().item() < 2e-6, (k, step)


@pytest.mark.gpu
def test_standalone_positional_encoder(dev, golden):
    """M.PositionalEncoder.forward as a standalone kernel vs the reference's own outputs"""
    from fsnerf_b200.core.models import PositionalEncoder
    g = golden("reference_mlp.npz")
    x, d = torch.from_numpy(g["x"]).to(dev), torch.from_numpy(g["d"]).to(dev)
    pe = PositionalEncoder(3, 10, True)
    assert pe.d_output == 63
    np.testing.assert_allclose(pe(x).cpu().numpy(), g["pe_pos"], atol=2e-6 * 512)  # |arg| up to 2^9: few-ulp sincos
    np.testing.assert_allclose(PositionalEncoder(3, 4, True)(d).cpu().numpy(), g["pe_dir"], atol=4e-6)
    np.testing.assert_allclose(PositionalEncoder(3, 4, False)(d).cpu().numpy(), g["pe_lin"], atol=4e-6)
    pin = torch.tensor([[0.1, -0.2, 0.3]], device=dev)
    np.testing.assert_allclose(pe(pin).cpu().numpy(), g["pe_pin"], atol=2e-5)
    from oracle import encoding as oenc
    m = torch.from_numpy(oenc.freq_mask(63, 300, 900)).to(dev)
    np.testing.assert_allclose(pe(x, m).cpu().numpy(), g["pe_pos"] * m.cpu().numpy(), atol=2e-6 * 512)
    assert pe(x[:0]).shape == (0, 63) and pe(x.reshape(2, -1, 3)).shape[:2] == (2, x.shape[0] // 2)


@pytest.mark.gpu
@pytest.mark.parametrize("log_space", [True, False])
@pytest.mark.parametrize("L", [0, 1, 6])
def test_standalone_positional_encoder_widths(dev, L, log_space):
    """the encoder at the widths and spacings the non-default networks use, against the oracle"""
    from fsnerf_b200.core.models import PositionalEncoder
    from oracle import encoding as oenc
    g = torch.Generator().manual_seed(L)
    x = (torch.rand(1000, 3, generator=g) * 2 - 1) * 3
    pe = PositionalEncoder(3, L, log_space)
    assert pe.d_output == 3 * (1 + 2 * L)
    ref = oenc.positional_encoding(x, L, log_space)
    assert ref.shape == (1000, pe.d_output)
    np.testing.assert_allclose(pe(x.to(dev)).cpu().numpy(), ref.numpy(), rtol=0, atol=1e-6)  # same fp32 arguments
    m = torch.rand(pe.d_output, generator=g)
    np.testing.assert_allclose(pe(x.to(dev), m.to(dev)).cpu().numpy(), (ref * m).numpy(), rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_mlp_forward_sigma_slot_and_render_coarse_skip(dev):
    """density_only=2 writes exactly the sigma of the full forward into raw[:,3]; a hierarchical
    render whose coarse pass skips the view branch gives bit-identical fine samples and image."""
    from fsnerf_b200 import ops
    from fsnerf_b200.engine import HotPath
    cfg = ops.make_cfg()
    params = ops.flatten_state_dict(cfg, omlp.init_state_dict(seed=3), dev)
    packed = ops.mlp_pack(cfg, params)
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(1000, 3, generator=g) * 2 - 1).to(dev)
    d = torch.nn.functional.normalize(torch.randn(1000, 3, generator=g), dim=-1).to(dev)
    full = ops.mlp_forward(cfg, params, packed, x=x, dirs=d)
    sig = ops.mlp_forward(cfg, params, packed, x=x, density_only=True)
    slot = ops.mlp_forward(cfg, params, packed, x=x, density_only=2)
    assert torch.equal(sig, full[:, 3]) and torch.equal(slot[:, 3], full[:, 3]) and float(slot[:, :3].abs().max()) == 0
    hp = HotPath(n_coarse=32, n_fine=64, device=dev)
    o = torch.tensor([0.0, 0.0, 4.0], device=dev).expand(500, 3).contiguous()
    dd = torch.nn.functional.normalize(torch.tensor([0.0, 0.0, -1.0], device=dev) + 0.2 * torch.randn(500, 3, device=dev), dim=-1)
    a = hp._forward(o, dd, None, None, train=False)           # coarse pass: sigma only
    hp.hier_skip = None
    ts_c, te_c = ops.sample_stratified(500, 32, hp.near, hp.far, None, device=dev)
    raw_c = ops.mlp_forward(cfg, hp.net_params(0), hp.packed[0], rays_o=o, rays_d=dd, t_starts=ts_c, t_ends=te_c)
    w_c = ops.composite_forward(raw_c.view(500, 32, 4), ts_c, te_c, bkgd=hp.bkgd)[3]
    assert torch.equal(a["w_c"], w_c)                          # same weights -> same fine samples
    ts_f, te_f, *_ = ops.sample_pdf(ts_c, w_c, 64, hp.far, None, want_aux=False)
    assert torch.equal(a["ts_f"], ts_f)
    raw_f = ops.mlp_forward(cfg, hp.net_params(1), hp.packed[1], rays_o=o, rays_d=dd, t_starts=ts_f, t_ends=te_f)
    assert torch.equal(a["rgb"], ops.composite_forward(raw_f.view(500, 96, 4), ts_f, te_f, bkgd=hp.bkgd)[0])
