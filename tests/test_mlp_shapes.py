"""The fused MLP on every network shape it accepts, against the oracle (oracle/mlp.py, oracle/render.py).

The forward issue table, the backward's image ring, its dgrad parities, the release of the position
encoding buffer, the width of the encoding K chunk and the weight-gradient job plan all depend on
the shape (n_layers, skip, frequencies, spacing).  The reference 8x256 net reaches one side of each;
NETS below reaches the others, and each entry says which edge it covers.  The CPU tests check the
host-side layout and size queries of every entry; the GPU tests check the kernels' numbers.

The weights are the default nn.Linear init with every ReLU layer's weights scaled by GAIN, so that
activations keep their size through a 10-layer net and every ReLU mask is mixed (asserted): with
the plain init a deep net's activations shrink toward zero and its outputs hardly depend on them."""
import os
import sys
from dataclasses import dataclass

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import encoding as oenc, mlp as omlp, render as orender  # noqa: E402
from test_gpu_stash import _check_masks, _layout  # noqa: E402


@dataclass(frozen=True)
class Net:
    id: str
    n_layers: int
    skip: tuple
    fp: int           # frequencies of the position encoding
    fd: int           # ... of the direction encoding
    log_space: bool
    n_gemm: int       # counts derived by hand from build_program / build_wgrad_plan
    blocks: int       # forward + dgrad 16 KB operand blocks of the packed image
    jobs: int         # weight-gradient jobs of the backward
    masked: bool      # run with random FreeNeRF masks
    covers: str

    def cfg(self):
        from fsnerf_b200 import ops
        return ops.make_cfg(self.n_layers, 256, self.skip, self.fp, self.fd, self.log_space)

    def kw(self):  # oracle architecture arguments
        return dict(n_layers=self.n_layers, skip=self.skip, n_freqs=self.fp, n_freqs_dir=self.fd,
                    log_space=self.log_space)

    @property
    def d_pe(self):
        return 3 * (1 + 2 * self.fp)

    @property
    def d_de(self):
        return 3 * (1 + 2 * self.fd)


NETS = [
    Net("ref", 8, (4,), 10, 4, True, 10, 141, 12, False, "the reference net: calibrates the bars"),
    Net("min", 2, (), 10, 4, True, 4, 43, 5, False, "ring depth 2; last_pos_user = 0"),
    Net("min_skip0", 2, (0,), 0, 0, True, 4, 45, 6, True, "skip into the sigma layer; 3-channel encodings"),
    Net("odd_lin", 7, (2, 5), 6, 2, False, 9, 127, 12, True,
        "even n_cons; rotating ring slots; linspace encoder in the MLP"),
    Net("skip_last", 5, (3,), 1, 10, False, 7, 93, 9, True,
        "skip into the last hidden layer; L = 1 linspace; 63-channel directions"),
    Net("odd_all_skips", 9, tuple(range(8)), 3, 0, True, 11, 171, 20, False, "odd n_gemm with kMaxJobs jobs"),
    Net("deepest", 10, tuple(range(7)), 10, 10, True, 12, 185, 20, True,
        "n_gemm = 12 and 20 jobs, both at their limits"),
]
BY_ID = {n.id: n for n in NETS}
# 21 weight-gradient jobs: the forward runs, the backward refuses
TOO_MANY_JOBS = Net("too_many_jobs", 10, tuple(range(8)), 10, 4, True, 12, 187, 21, False,
                    "one wgrad job past the limit")

P_BIG = 128 * (148 * 3 + 5) + 37   # every forward CTA runs >= 3 tiles, every dgrad CTA wraps its ring
GAIN = 6 ** 0.5                    # U(-1/sqrt(fan_in), ..) * sqrt(6): the ReLU-preserving variance 2 / fan_in
CHUNK = 128 * 128                  # one [128 rows x 64 channels] bf16 SW128 image

# Bars, calibrated on the reference net ("ref") with these weights and inputs, about twice its
# largest error measured on a B200: forward vs the bf16 emulation, max 9.3e-3 and rms 1.6e-4 over
# all samples; vs fp32, max 5.8e-3 rgb and 1.7e-2 sigma; weight gradients vs the emulation, 1.4e-2
# per tensor.  (The bars of tests/test_gpu_kernels.py hold for the plain init, whose small
# activations make every error small.)  Every other entry meets the same bars.
EMU_BAR = 2e-2
EMU_RMS_BAR = 4e-4
RGB_BAR, SIGMA_BAR = 1.5e-2, 3.5e-2
GRAD_BAR = 3e-2
# one engine step of 512 rays against the fp32 oracle: measured 2.1e-4 loss, 2.5e-2 per tensor
ENGINE_LOSS_BAR, ENGINE_GRAD_BAR = 1e-3, 5e-2


@pytest.fixture(scope="module")
def lib():
    from fsnerf_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fsnerf_b200 import ops
    ops.require_device(0)
    return torch.device("cuda:0")


def _ids(nets):
    return [n.id for n in nets]


# ------------------------------------------------------------------------ CPU: host-side layout
@pytest.mark.parametrize("net", NETS + [TOO_MANY_JOBS], ids=_ids(NETS + [TOO_MANY_JOBS]))
def test_param_layout_matches_the_oracle_and_the_drop_in(lib, net):
    from fsnerf_b200 import ops
    from fsnerf_b200.core.models import NeRF
    from fsnerf_b200.engine import NeRF_shapes
    cfg = net.cfg()
    sd = omlp.init_state_dict(net.n_layers, 256, net.skip, net.fp, net.fd, seed=42)
    names = ops.state_dict_names(cfg)
    assert list(sd) == names
    layout = ops.mlp_param_layout(cfg)
    assert [n for _, n in layout] == [sd[k].numel() for k in names]
    shapes = NeRF_shapes(cfg)
    assert [shapes[k] for k in names] == [tuple(sd[k].shape) for k in names]
    kw = {"pos_fn": {"n_freqs": net.fp, "log_space": net.log_space},
          "dir_fn": {"n_freqs": net.fd, "log_space": net.log_space}}
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(42)
        model = NeRF(3, 3, net.n_layers, 256, list(net.skip), **kw)
    msd = model.state_dict()
    assert list(msd) == names
    for k in names:
        assert msd[k].shape == sd[k].shape, k
        assert torch.equal(msd[k], sd[k]), k   # same seed-42 init, bit for bit
    # the GEMM layers (every Linear but the sigma / rgb heads) and their weight-gradient jobs: one per
    # input part, activations (in_features >= 256) and an encoding (in_features != 256)
    gemm_in = [sd[k].shape[1] for k in names if k.endswith(".weight") and k not in ("sigma.weight", "rgb.weight")]
    assert len(gemm_in) == net.n_gemm == net.n_layers + 2
    assert sum((i >= 256) + (i != 256) for i in gemm_in) == net.jobs


@pytest.mark.parametrize("net", NETS + [TOO_MANY_JOBS], ids=_ids(NETS + [TOO_MANY_JOBS]))
def test_packed_stash_and_workspace_sizes(lib, net):
    from fsnerf_b200 import ops
    from fsnerf_b200._lib import FsnerfError
    cfg = net.cfg()
    assert ops.mlp_packed_bytes(cfg) == net.blocks * 16384 + 4864 * 4
    rec = _layout(cfg)[1]
    for n in (1, 128, 129, 5000, P_BIG):
        assert ops.mlp_stash_bytes(cfg, n) == rec * ((n + 127) // 128), n
    for n in (1, 300, P_BIG):
        default = ops.mlp_bwd_workspace_bytes(cfg, n)
        assert default > 0
        if net.jobs <= 20:
            assert ops.mlp_bwd_workspace_bytes(cfg, n, deterministic=True) > default, n
        else:  # the deterministic workspace query builds the job plan, and refuses it
            with pytest.raises(FsnerfError, match="too many wgrad jobs"):
                ops.mlp_bwd_workspace_bytes(cfg, n, deterministic=True)


@pytest.mark.parametrize("n_layers,skip,fp,fd,match", [
    (11, (4,), 10, 4, "n_layers must be in"),      # n_gemm 13: no forward can run it
    (14, (), 10, 4, "n_layers must be in"),
    (1, (), 10, 4, "n_layers must be in"),
    (8, (7,), 10, 4, "skip on or after the last hidden layer"),
    (2, (1,), 10, 4, "skip on or after the last hidden layer"),
    (8, (4,), 11, 4, "n_freqs_pos"),
    (8, (4,), 10, 11, "n_freqs_dir"),
    (8, (4,), -1, 4, "n_freqs_pos"),
])
def test_unsupported_networks_are_refused_by_every_query(lib, n_layers, skip, fp, fd, match):
    from fsnerf_b200 import ops
    from fsnerf_b200._lib import FsnerfError
    from fsnerf_b200.core.models import NeRF
    cfg = ops.make_cfg(n_layers, 256, skip, fp, fd)
    for query in (ops.mlp_param_count, ops.mlp_param_layout, ops.mlp_packed_bytes,
                  lambda c: ops.mlp_stash_bytes(c, 128), lambda c: ops.mlp_bwd_workspace_bytes(c, 128),
                  lambda c: ops.mlp_bwd_workspace_bytes(c, 128, deterministic=True)):
        with pytest.raises(FsnerfError, match=match):
            query(cfg)
    if fp >= 0:  # (a negative width fails in nn.Linear before the library is asked)
        kw = {"pos_fn": {"n_freqs": fp, "log_space": True}, "dir_fn": {"n_freqs": fd, "log_space": True}}
        with pytest.raises(FsnerfError, match=match):
            NeRF(3, 3, n_layers, 256, list(skip), **kw)


# ------------------------------------------------------------------------ GPU helpers
def _state_dict(net, seed):
    sd = omlp.init_state_dict(net.n_layers, 256, net.skip, net.fp, net.fd, seed=seed)
    for k in sd:
        if k.endswith(".weight") and (k.startswith("layers.") or k in ("connection.weight", "branch.weight")):
            sd[k] = sd[k] * GAIN
    return sd


def _points(net, P, seed):
    """-> x [P,3], dirs [P,3], mask_pos, mask_dir (None unless net.masked)"""
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(P, 3, generator=g) * 2 - 1) * 2.5
    d = F.normalize(torch.randn(P, 3, generator=g), dim=-1)
    mp = torch.rand(net.d_pe, generator=g) if net.masked else None
    md = torch.rand(net.d_de, generator=g) if net.masked else None
    return x, d, mp, md


def _cu(t, dev):
    return None if t is None else t.to(dev)


def _relu_fractions(sd, net, x, d, mp, md):
    """fraction of positive outputs of every ReLU layer (hidden layers, branch) in fp32"""
    enc = oenc.positional_encoding(x, net.fp, net.log_space)
    if mp is not None:
        enc = enc * mp
    h, fr = enc, []
    for i in range(net.n_layers):
        h = F.relu(F.linear(h, sd[f"layers.{i}.weight"], sd[f"layers.{i}.bias"]))
        fr.append((h > 0).float().mean().item())
        if i in net.skip:
            h = torch.cat([h, enc], -1)
    c = F.linear(h, sd["connection.weight"], sd["connection.bias"])
    de = oenc.positional_encoding(d, net.fd, net.log_space)
    if md is not None:
        de = de * md
    hb = F.relu(F.linear(torch.cat([c, de], -1), sd["branch.weight"], sd["branch.bias"]))
    fr.append((hb > 0).float().mean().item())
    return fr


def _setup(net, seed, dev):
    from fsnerf_b200 import ops
    cfg = net.cfg()
    sd = _state_dict(net, seed)
    params = ops.flatten_state_dict(cfg, sd, dev)
    return cfg, sd, params, ops.mlp_pack(cfg, params)


def _out_errors(out, ref):
    e = (out.cpu() - ref).abs()
    return e[:, :3].max().item(), e[:, 3].max().item()


def _check_forward(tag, net, out, emu, ref32):
    emu_e = max(_out_errors(out, emu))
    emu_rms = (out.cpu() - emu).square().mean().sqrt().item()
    rgb_e, sig_e = _out_errors(out, ref32)
    print(f"{tag}: vs bf16emu max {emu_e:.2e} rms {emu_rms:.2e}; vs fp32 max rgb {rgb_e:.2e} sigma {sig_e:.2e}")
    assert emu_e < EMU_BAR and emu_rms < EMU_RMS_BAR, (tag, emu_e, emu_rms)
    assert rgb_e < RGB_BAR and sig_e < SIGMA_BAR, (tag, rgb_e, sig_e)


def _density_only_is_the_full_sigma(cfg, params, packed, full, **inputs):
    from fsnerf_b200 import ops
    sig = ops.mlp_forward(cfg, params, packed, density_only=1, **inputs)
    slot = ops.mlp_forward(cfg, params, packed, density_only=2, **inputs)
    torch.cuda.synchronize()
    assert torch.equal(sig, full[:, 3])
    assert torch.equal(slot[:, 3], full[:, 3]) and not slot[:, :3].any()


def _unflatten(cfg, flat):
    from fsnerf_b200 import ops
    return {n: flat[o:o + k].cpu() for (o, k), n in zip(ops.mlp_param_layout(cfg), ops.state_dict_names(cfg))}


def _rel(a, b):
    a, b = a.reshape(-1).double(), b.reshape(-1).double()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


# ------------------------------------------------------------------------ GPU: forward
@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 129, P_BIG])
@pytest.mark.parametrize("net", NETS, ids=_ids(NETS))
def test_forward_points_match_the_oracles(dev, net, P):
    from fsnerf_b200 import ops
    cfg, sd, params, packed = _setup(net, 5, dev)
    x, d, mp, md = _points(net, P, seed=P)
    inputs = dict(x=x.to(dev), mask_pos=_cu(mp, dev), mask_dir=_cu(md, dev))
    out = ops.mlp_forward(cfg, params, packed, dirs=d.to(dev), **inputs)
    with torch.no_grad():
        emu = omlp.nerf_forward_bf16emu(sd, x, d, mask_pos=mp, mask_dir=md, **net.kw())
        ref32 = omlp.nerf_forward(sd, x, d, mask_pos=mp, mask_dir=md, **net.kw())
    if P == P_BIG:
        fr = _relu_fractions(sd, net, x, d, mp, md)
        print(f"{net.id}: ReLU ones per layer", [round(f, 3) for f in fr])
        assert all(0.1 <= f <= 0.9 for f in fr), fr
    _check_forward(f"{net.id} P={P} points", net, out, emu, ref32)
    _density_only_is_the_full_sigma(cfg, params, packed, out, **inputs)


@pytest.mark.gpu
@pytest.mark.parametrize("net", NETS, ids=_ids(NETS))
def test_forward_rays_match_the_oracles(dev, net):
    """ray input (x = o + d (t0 + t1) / 2 in the kernel), S not a multiple of 128"""
    from fsnerf_b200 import ops
    cfg, sd, params, packed = _setup(net, 6, dev)
    R, S = 300, 97
    g = torch.Generator().manual_seed(11)
    o = torch.tensor([0.0, 0.0, 4.0]) + 0.3 * torch.randn(R, 3, generator=g)
    rd = F.normalize(torch.tensor([0.0, 0.0, -1.0]) + 0.3 * torch.randn(R, 3, generator=g), dim=-1)
    e = torch.sort(2 + 4 * torch.rand(R, S + 1, generator=g), -1).values
    ts, te = e[:, :-1].contiguous(), e[:, 1:].contiguous()
    _, _, mp, md = _points(net, 1, seed=12)
    inputs = dict(rays_o=o.to(dev), rays_d=rd.to(dev), t_starts=ts.to(dev), t_ends=te.to(dev),
                  mask_pos=_cu(mp, dev), mask_dir=_cu(md, dev))
    out = ops.mlp_forward(cfg, params, packed, **inputs)
    # the kernel evaluates o + d * tm as one fused multiply-add: the same point, rounded once
    tm = (ts + te) / 2.0
    x = (o[:, None, :].double() + rd[:, None, :].double() * tm[..., None].double()).float().reshape(-1, 3)
    dirs = rd[:, None, :].expand(R, S, 3).reshape(-1, 3)
    with torch.no_grad():
        emu = omlp.nerf_forward_bf16emu(sd, x, dirs, mask_pos=mp, mask_dir=md, **net.kw())
        ref32 = orender.query_mlp(sd, o, rd, ts, te, mp, md, **net.kw()).reshape(-1, 4)
    _check_forward(f"{net.id} rays {R}x{S}", net, out, emu, ref32)
    _density_only_is_the_full_sigma(cfg, params, packed, out, **inputs)


# ------------------------------------------------------------------------ GPU: stash
def _unswizzle(img, n_tiles):
    """[n_tiles, CHUNK] bytes of SW128 images -> [n_tiles, 128, 64] bf16 bit patterns (uint16)"""
    rows = np.arange(128)
    c = img.reshape(n_tiles, 128, 8, 16)
    units = c[:, rows[:, None], (np.arange(8)[None, :] ^ (rows[:, None] & 7))]  # unit u of row r is at u ^ (r & 7)
    return np.ascontiguousarray(units).reshape(n_tiles, 128, 128).view(np.uint16)


def _ordered(bits):
    """bf16 bit patterns -> integers in value order (adjacent bf16 values differ by 1, -0 == +0)"""
    b = bits.astype(np.int32)
    return np.where(b & 0x8000, -(b & 0x7FFF), b)


def _check_encoding_image(tag, img, n_tiles, P, v, L, log_space, mask):
    enc = oenc.positional_encoding(v, L, log_space)
    if mask is not None:
        enc = enc * mask
    want = enc.bfloat16().view(torch.int16).numpy().view(np.uint16)
    w = enc.shape[1]
    got = _unswizzle(img, n_tiles).reshape(-1, 64)[:P]
    assert not got[:, w:].any(), f"{tag}: channels past {w} must be 0"
    diff = np.abs(_ordered(got[:, :w]) - _ordered(want))
    exact = float((diff == 0).mean())
    print(f"{tag}: {w} channels, max {int(diff.max())} bf16 ulp, {100 * exact:.3f} % exact")
    assert diff.max() <= 1, (tag, np.argwhere(diff > 1)[:4])
    assert exact >= 0.999, (tag, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("net", NETS, ids=_ids(NETS))
def test_stash_masks_and_encoding_images(dev, net):
    from fsnerf_b200 import ops
    cfg, sd, params, packed = _setup(net, 7, dev)
    P = 128 * 5 + 77
    x, d, mp, md = _points(net, P, seed=13)
    n_tiles = (P + 127) // 128
    stash = torch.full((ops.mlp_stash_bytes(cfg, P),), 0xA5, dtype=torch.uint8, device=dev)
    ops.mlp_forward(cfg, params, packed, x=x.to(dev), dirs=d.to(dev), mask_pos=_cu(mp, dev),
                    mask_dir=_cu(md, dev), stash=stash)
    torch.cuda.synchronize()
    _check_masks(cfg, stash, n_tiles)
    layers, rec = _layout(cfg)
    s = stash.view(n_tiles, rec).cpu().numpy()
    dir_off = layers[-1][0] - CHUNK  # the direction image sits right before the branch output
    _check_encoding_image(f"{net.id} position", s[:, :CHUNK], n_tiles, P, x, net.fp, net.log_space, mp)
    _check_encoding_image(f"{net.id} direction", s[:, dir_off:dir_off + CHUNK], n_tiles, P, d, net.fd,
                          net.log_space, md)


# ------------------------------------------------------------------------ GPU: backward
def _forward_backward(net, dev, P, seed):
    from fsnerf_b200 import ops
    cfg, sd, params, packed = _setup(net, seed, dev)
    x, d, mp, md = _points(net, P, seed=100 + seed)
    d_out = torch.randn(P, 4, generator=torch.Generator().manual_seed(200 + seed))
    stash = torch.empty(ops.mlp_stash_bytes(cfg, P), dtype=torch.uint8, device=dev)
    out = ops.mlp_forward(cfg, params, packed, x=x.to(dev), dirs=d.to(dev), mask_pos=_cu(mp, dev),
                          mask_dir=_cu(md, dev), stash=stash)
    return cfg, sd, params, packed, (x, d, mp, md), d_out, stash, out


@pytest.mark.gpu
@pytest.mark.parametrize("net", NETS, ids=_ids(NETS))
def test_backward_matches_the_bf16_emulation(dev, net):
    """every weight and bias (heads included) against autograd of the bf16 emulation, under an
    incoherent d_out (see test_gpu_kernels.test_mlp_backward_weight_grads); a second call adds"""
    from fsnerf_b200 import ops
    P = P_BIG
    cfg, sd, params, packed, (x, d, mp, md), d_out, stash, out = _forward_backward(net, dev, P, 11)
    grads = torch.zeros_like(params)
    ws = torch.empty(ops.mlp_bwd_workspace_bytes(cfg, P), dtype=torch.uint8, device=dev)
    ops.mlp_backward(cfg, params, packed, P, stash, out, d_out.to(dev), grads, ws)
    torch.cuda.synchronize()
    ours = _unflatten(cfg, grads)
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref_out = omlp.nerf_forward_bf16emu(sdr, x, d, mask_pos=mp, mask_dir=md, **net.kw())
    fwd_e = (ref_out.detach() - out.cpu()).abs().max().item()
    names = list(sdr)
    ref = dict(zip(names, torch.autograd.grad((ref_out * d_out).sum(), [sdr[n] for n in names])))
    rels = {n: _rel(ours[n], ref[n]) for n in names}
    print(f"{net.id}: forward vs bf16emu {fwd_e:.2e}; relative gradient errors",
          {k: round(v, 5) for k, v in rels.items()})
    assert fwd_e < EMU_BAR, fwd_e
    for n in names:
        assert rels[n] < GRAD_BAR, (n, rels[n])
    ops.mlp_backward(cfg, params, packed, P, stash, out, d_out.to(dev), grads, ws)
    twice = _unflatten(cfg, grads)
    for n in names:
        assert _rel(twice[n], 2 * ours[n]) < 1e-3, n


@pytest.mark.gpu
@pytest.mark.parametrize("net", [BY_ID["odd_lin"], BY_ID["deepest"]], ids=["odd_lin", "deepest"])
def test_deterministic_backward(dev, net):
    from fsnerf_b200 import ops
    P = P_BIG
    cfg, sd, params, packed, _, d_out, stash, out = _forward_backward(net, dev, P, 21)
    d_out = d_out.to(dev)
    ws = torch.empty(ops.mlp_bwd_workspace_bytes(cfg, P, deterministic=True), dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev).manual_seed(3)

    def det(g0):
        ws.copy_(torch.randint(0, 256, ws.shape, dtype=torch.uint8, device=dev, generator=gen))  # garbage
        g = g0.clone()
        ops.mlp_backward(cfg, params, packed, P, stash, out, d_out, g, ws, deterministic=True)
        torch.cuda.synchronize()
        return g

    zeros = torch.zeros_like(params)
    a, b = det(zeros), det(zeros)
    assert torch.equal(a, b)
    default = torch.zeros_like(params)
    ws_d = torch.empty(ops.mlp_bwd_workspace_bytes(cfg, P), dtype=torch.uint8, device=dev)
    ops.mlp_backward(cfg, params, packed, P, stash, out, d_out, default, ws_d)
    ours, theirs = _unflatten(cfg, a), _unflatten(cfg, default)
    rels = {n: _rel(ours[n], theirs[n]) for n in ours}
    print(f"{net.id}: deterministic vs default, max relative tensor difference {max(rels.values()):.2e}")
    for n, r in rels.items():
        assert r < GRAD_BAR, (n, r)
    g0 = torch.randn(params.shape, generator=torch.Generator().manual_seed(4)).to(dev)
    assert torch.equal(det(g0), g0 + a)


@pytest.mark.gpu
def test_too_many_wgrad_jobs_forward_runs_backward_refuses(dev):
    from fsnerf_b200 import ops
    from fsnerf_b200._lib import FsnerfError
    net = TOO_MANY_JOBS
    P = 1000
    cfg, sd, params, packed, (x, d, mp, md), d_out, stash, out = _forward_backward(net, dev, P, 31)
    with torch.no_grad():
        emu = omlp.nerf_forward_bf16emu(sd, x, d, **net.kw())
        ref32 = omlp.nerf_forward(sd, x, d, **net.kw())
    _check_forward(f"{net.id} P={P} points", net, out, emu, ref32)
    grads = torch.zeros_like(params)
    ws = torch.empty(ops.mlp_bwd_workspace_bytes(cfg, P), dtype=torch.uint8, device=dev)
    with pytest.raises(FsnerfError, match="too many wgrad jobs"):
        ops.mlp_backward(cfg, params, packed, P, stash, out, d_out.to(dev), grads, ws)
    torch.cuda.synchronize()
    assert not grads.any()
    # the context stays usable: a backward of a supported net runs and adds its gradient
    cfg2, _, params2, packed2, _, d_out2, stash2, out2 = _forward_backward(BY_ID["min"], dev, P, 32)
    g2 = torch.zeros_like(params2)
    ws2 = torch.empty(ops.mlp_bwd_workspace_bytes(cfg2, P), dtype=torch.uint8, device=dev)
    ops.mlp_backward(cfg2, params2, packed2, P, stash2, out2, d_out2.to(dev), g2, ws2)
    torch.cuda.synchronize()
    assert g2.abs().sum().item() > 0 and bool(torch.isfinite(g2).all())


# ------------------------------------------------------------------------ GPU: engine
@pytest.mark.gpu
@pytest.mark.parametrize("net,mask_step", [(BY_ID["odd_lin"], 300), (BY_ID["skip_last"], None)],
                         ids=["odd_lin", "skip_last"])
def test_engine_train_step_against_oracle(dev, net, mask_step):
    """one hierarchical HotPath step of a non-default net: loss and every gradient tensor against
    oracle.render.train_step (fp32), as tests/test_gpu_parity_hard.py does for the reference net"""
    from fsnerf_b200.engine import HotPath
    R, Sc, Sf, reg_steps = 512, 32, 64, 1000
    rng = np.random.default_rng(41)
    o = np.tile(np.array([[0.0, 0.0, 4.0]], np.float32), (R, 1)) + 0.2 * rng.standard_normal((R, 3)).astype(np.float32)
    d = np.array([0, 0, -1], np.float32) + 0.3 * rng.standard_normal((R, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    gt = rng.random((R, 3), dtype=np.float32)
    us, up = rng.random((R, Sc), dtype=np.float32), rng.random((R, Sf), dtype=np.float32)
    hp = HotPath(n_coarse=Sc, n_fine=Sf, near=2.0, far=6.0, white_bkgd=True, device=dev, **net.kw())
    sds = []
    for i in range(2):
        sd = _state_dict(net, 50 + i)
        sd["sigma.bias"] = sd["sigma.bias"] + 0.5  # mostly positive densities: the weights matter
        hp.load_state_dict(i, sd)
        sds.append(sd)
    mp = md = None
    if mask_step is not None:
        hp.set_freq_mask(mask_step, reg_steps)
        mp = oenc.freq_mask(net.d_pe, mask_step, reg_steps)
        md = oenc.freq_mask(net.d_de, mask_step, reg_steps)
        assert hp.mask_pos.numel() == net.d_pe and hp.mask_dir.numel() == net.d_de
        assert 0 < mp.sum() < net.d_pe and 0 < md.sum() < net.d_de
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    ls = hp.train_step(cu(o), cu(d), cu(gt), cu(us), cu(up), lr=5e-4, apply_update=False)
    grads = hp.grads.cpu()
    ref_loss, _, ref_g = orender.train_step({k: v.clone() for k, v in sds[0].items()},
                                            {k: v.clone() for k, v in sds[1].items()},
                                            dict(step=0, m={}, v={}), o, d, gt, 2.0, 6.0, Sc, Sf, us, up, 5e-4,
                                            True, mask_pos=mp, mask_dir=md, **net.kw())
    loss = (ls[0].item() + ls[1].item()) / (3 * R)
    rels = {}
    for i, tag in ((0, "c."), (1, "f.")):
        flat = grads[i * hp.n_net:(i + 1) * hp.n_net]
        for (off, n), name in zip(hp.layout, hp.names):
            rels[tag + name] = _rel(flat[off:off + n], ref_g[tag + name])
    print(f"{net.id} engine step: loss {loss:.6f} vs {ref_loss:.6f}; max relative gradient error "
          f"{max(rels.values()):.2e}", {k: round(v, 4) for k, v in rels.items()})
    assert abs(loss - ref_loss) < ENGINE_LOSS_BAR, (loss, ref_loss)
    for k, r in rels.items():
        assert r < ENGINE_GRAD_BAR, (k, r)
