"""Thin torch-tensor wrappers over the C ABI (device memory + stream plumbing
only; all arithmetic happens in libfsnerf_b200.so).  Every function requires
CUDA tensors; there is no CPU path."""
import ctypes as C

import torch

from . import _lib
from ._lib import NetCfg, check, ptr

COMP_SIGMA_RELU = 1
COMP_DEPTH_UNNORM = 2
COMP_PRODUCT_TRANS = 4


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.FsnerfError(f"{name}: expected a CUDA tensor (no CPU fallback)")
    if t.device.index != torch.cuda.current_device():
        # kernels launch on the CURRENT device's stream; function attributes are configured per device
        raise _lib.FsnerfError(f"{name}: tensor on cuda:{t.device.index} but the current device is "
                               f"cuda:{torch.cuda.current_device()} (wrap the call in torch.cuda.device(...))")
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.contiguous().float()
    return t


def require_device(dev=None):
    dev = torch.cuda.current_device() if dev is None else dev
    check(_lib.load().fsnerf_device_ok(int(dev)), "fsnerf_device_ok")


# ------------------------------------------------------------------ rays
def gen_rays(poses, H, W, focal, pixel_ids=None, first_id=0, n_rays=None, ndc=False,
             ndc_near=1.0, images=None):
    """poses [V,3|4,4] f32 cuda; pixel_ids int64 [R] or None (first_id + arange(n_rays)).
    -> rays_o [R,3], rays_d [R,3], rgb_gt [R,3] | None"""
    poses = _f32c(poses, "poses")
    if poses.dim() == 2:
        poses = poses[None]
    V, rows = poses.shape[0], poses.shape[1]
    if pixel_ids is not None:
        pixel_ids = pixel_ids.contiguous().to(torch.int64)
        n_rays = pixel_ids.numel()
    dev = poses.device
    rays_o = torch.empty(n_rays, 3, device=dev)
    rays_d = torch.empty(n_rays, 3, device=dev)
    images = _f32c(images, "images")
    rgb = torch.empty(n_rays, 3, device=dev) if images is not None else None
    sx = -1.0 / (W / (2.0 * focal))
    sy = -1.0 / (H / (2.0 * focal))
    check(_lib.load().fsnerf_gen_rays(ptr(poses), V, rows, H, W, float(focal), ptr(pixel_ids),
                                      int(first_id), int(n_rays), int(ndc), float(ndc_near), sx, sy,
                                      ptr(images), ptr(rays_o), ptr(rays_d), ptr(rgb), _stream()),
          "fsnerf_gen_rays")
    return rays_o, rays_d, rgb


def to_ndc(rays_o, rays_d, H, W, focal, near):
    ro, rd = _f32c(rays_o.reshape(-1, 3), "rays_o"), _f32c(rays_d.reshape(-1, 3), "rays_d")
    no, nd = torch.empty_like(ro), torch.empty_like(rd)
    sx = -1.0 / (W / (2.0 * focal))
    sy = -1.0 / (H / (2.0 * focal))
    check(_lib.load().fsnerf_to_ndc(ptr(ro), ptr(rd), ro.shape[0], float(near), sx, sy, ptr(no),
                                    ptr(nd), _stream()), "fsnerf_to_ndc")
    return no.reshape(rays_o.shape), nd.reshape(rays_d.shape)


def rng_uniform(n, seed, device=None):
    """u(seed, i), i < n: the stream the seeded samplers draw from (oracle/sampling.py:rng_uniform)."""
    out = torch.empty(n, device=device)
    check(_lib.load().fsnerf_rng_uniform(n, int(seed) & _SEED_MASK, ptr(out), _stream()), "fsnerf_rng_uniform")
    return out


_SEED_MASK = (1 << 64) - 1


def sample_stratified(n_rays, n_samples, near, far, u=None, device=None, seed=None):
    """u: explicit uniforms [R,S]; seed: draw them in the kernel (u must be None); neither: the
    deterministic points."""
    u = _f32c(u, "u")
    dev = u.device if u is not None else device
    ts = torch.empty(n_rays, n_samples, device=dev)
    te = torch.empty(n_rays, n_samples, device=dev)
    if seed is not None:
        if u is not None:
            raise _lib.FsnerfError("sample_stratified: pass u or seed, not both")
        check(_lib.load().fsnerf_sample_stratified_seeded(n_rays, n_samples, float(near), float(far),
                                                          int(seed) & _SEED_MASK, ptr(ts), ptr(te), _stream()),
              "fsnerf_sample_stratified_seeded")
        return ts, te
    check(_lib.load().fsnerf_sample_stratified(n_rays, n_samples, float(near), float(far), ptr(u),
                                               ptr(ts), ptr(te), _stream()), "fsnerf_sample_stratified")
    return ts, te


def sample_pdf(z_coarse, w_coarse, n_fine, far, u=None, want_aux=True, seed=None):
    z, w, u = _f32c(z_coarse, "z_coarse"), _f32c(w_coarse, "w_coarse"), _f32c(u, "u")
    R, Sc = z.shape
    dev = z.device
    ts = torch.empty(R, Sc + n_fine, device=dev)
    te = torch.empty(R, Sc + n_fine, device=dev)
    samples = torch.empty(R, n_fine, device=dev) if want_aux else None
    inds = torch.empty(R, n_fine, device=dev, dtype=torch.int32) if want_aux else None
    perm = torch.empty(R, Sc + n_fine, device=dev, dtype=torch.int32) if want_aux else None
    if seed is not None:
        if u is not None:
            raise _lib.FsnerfError("sample_pdf: pass u or seed, not both")
        check(_lib.load().fsnerf_sample_pdf_seeded(R, Sc, n_fine, ptr(z), ptr(w), int(seed) & _SEED_MASK,
                                                   float(far), ptr(samples), ptr(inds), ptr(perm), ptr(ts),
                                                   ptr(te), _stream()), "fsnerf_sample_pdf_seeded")
        return ts, te, samples, inds, perm
    check(_lib.load().fsnerf_sample_pdf(R, Sc, n_fine, ptr(z), ptr(w), ptr(u), float(far),
                                        ptr(samples), ptr(inds), ptr(perm), ptr(ts), ptr(te),
                                        _stream()), "fsnerf_sample_pdf")
    return ts, te, samples, inds, perm


# ------------------------------------------------------------ compositing
def composite_forward(raw, t_starts, t_ends, bkgd=None, delta_scale=None, flags=0, extras=False):
    raw, ts, te = _f32c(raw, "raw"), _f32c(t_starts, "t_starts"), _f32c(t_ends, "t_ends")
    R, S = ts.shape
    dev = raw.device
    rgb = torch.empty(R, 3, device=dev)
    op = torch.empty(R, 1, device=dev)
    dp = torch.empty(R, 1, device=dev)
    w = torch.empty(R, S, device=dev)
    al = torch.empty(R, S, device=dev) if extras else None
    tr = torch.empty(R, S, device=dev) if extras else None
    check(_lib.load().fsnerf_composite_forward(R, S, ptr(raw), ptr(ts), ptr(te),
                                               ptr(_f32c(delta_scale, "delta_scale")),
                                               ptr(_f32c(bkgd, "bkgd")), flags, ptr(rgb), ptr(op),
                                               ptr(dp), ptr(w), ptr(al), ptr(tr), _stream()),
          "fsnerf_composite_forward")
    return rgb, op, dp, w, al, tr


OCC_FUNCS = {"linear": 1, "exp": 2}  # core.loss.OcclusionRegularizer.func (src/core/loss.py:57-62)


def composite_backward(raw, t_starts, t_ends, d_rgb, d_opacity=None, d_depth=None, d_weights=None,
                       bkgd=None, delta_scale=None, flags=0, want_d_bkgd=False, occ=None):
    """occ = None, or (a, b, func, scale, loss_sum): the occlusion regulariser fused in
    (d_raw.sigma += scale*w(t_mid); loss_sum[0] += sum w(t_mid)*sigma, unscaled)."""
    raw, ts, te = _f32c(raw, "raw"), _f32c(t_starts, "t_starts"), _f32c(t_ends, "t_ends")
    R, S = ts.shape
    d_raw = torch.empty(R, S, 4, device=raw.device)
    d_bkgd = torch.zeros(3, device=raw.device) if want_d_bkgd else None
    if occ is not None:
        a, b, func, scale, loss_sum = occ
        if func not in OCC_FUNCS:
            raise ValueError(f"Unknown occlusion regularizer type: {func}")  # loss.py:62
        check(_lib.load().fsnerf_composite_backward_occ(
            R, S, ptr(raw), ptr(ts), ptr(te), ptr(_f32c(delta_scale, "delta_scale")),
            ptr(_f32c(bkgd, "bkgd")), flags, ptr(_f32c(d_rgb, "d_rgb")),
            ptr(_f32c(d_opacity, "d_opacity")), ptr(_f32c(d_depth, "d_depth")),
            ptr(_f32c(d_weights, "d_weights")), ptr(d_raw), ptr(d_bkgd), OCC_FUNCS[func], float(a),
            float(b), float(scale), ptr(loss_sum), _stream()), "fsnerf_composite_backward_occ")
        return d_raw, d_bkgd
    check(_lib.load().fsnerf_composite_backward(
        R, S, ptr(raw), ptr(ts), ptr(te), ptr(_f32c(delta_scale, "delta_scale")),
        ptr(_f32c(bkgd, "bkgd")), flags, ptr(_f32c(d_rgb, "d_rgb")),
        ptr(_f32c(d_opacity, "d_opacity")), ptr(_f32c(d_depth, "d_depth")),
        ptr(_f32c(d_weights, "d_weights")), ptr(d_raw), ptr(d_bkgd), _stream()),
        "fsnerf_composite_backward")
    return d_raw, d_bkgd


def encode(x, freqs, mask=None):
    """standalone positional encoding: x [P,d] -> [P, d*(1+2L)] fp32 (reference channel order)"""
    x = _f32c(x, "x")
    P, d = x.shape
    L = freqs.numel()
    out = torch.empty(P, d * (1 + 2 * L), device=x.device)
    check(_lib.load().fsnerf_encode(P, d, L, ptr(_f32c(freqs, "freqs")), ptr(_f32c(mask, "mask")), ptr(x), ptr(out),
                                    _stream()), "fsnerf_encode")
    return out


# ---------------------------------------------- occupancy grid + packed compositing
def occgrid_march(rays_o, rays_d, binaries, aabbs, step, near=0.0, far=1e10, near_planes=None):
    """-> (ray_indices int64 [N], t_starts [N], t_ends [N], offsets int64 [R+1]); two launches of
    the marching kernel (count, fill) around one exclusive scan of the per-ray counts."""
    rays_o, rays_d = _f32c(rays_o, "rays_o"), _f32c(rays_d, "rays_d")
    aabbs = _f32c(aabbs, "aabbs").reshape(-1, 6)
    levels, res = binaries.shape[0], binaries.shape[1]
    if binaries.dtype != torch.uint8:
        binaries = binaries.to(torch.uint8)
    binaries = binaries.contiguous()
    R, dev = rays_o.shape[0], rays_o.device
    counts = torch.zeros(R, dtype=torch.int32, device=dev)
    lib = _lib.load()
    args = (R, ptr(rays_o), ptr(rays_d), ptr(_f32c(near_planes, "near_planes")), float(near), float(far),
            float(step), ptr(aabbs), int(levels), int(res), ptr(binaries))
    check(lib.fsnerf_occgrid_march(*args, None, ptr(counts), None, None, None, _stream()), "fsnerf_occgrid_march")
    offsets = torch.zeros(R + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=offsets[1:])
    N = int(offsets[-1].item())  # packed size: the one host read of the sampler, as in nerfacc
    ri = torch.empty(N, dtype=torch.int64, device=dev)
    ts, te = torch.empty(N, device=dev), torch.empty(N, device=dev)
    if N > 0:
        check(lib.fsnerf_occgrid_march(*args, ptr(offsets), None, ptr(ri), ptr(ts), ptr(te), _stream()),
              "fsnerf_occgrid_march")
    return ri, ts, te, offsets


def occgrid_filter(t_starts, t_ends, offsets, sigmas, early_stop_eps=1e-4, alpha_thre=0.0):
    """Transmittance visibility filter of OccGridEstimator.sampling on packed candidates (ray r owns
    [offsets[r], offsets[r+1])).  -> survivors' (ray_indices int64 [M], t_starts [M], t_ends [M],
    offsets int64 [R+1]); two launches (count, fill) around one exclusive scan, one host read of M."""
    ts, te, sig = _f32c(t_starts, "t_starts"), _f32c(t_ends, "t_ends"), _f32c(sigmas, "sigmas").reshape(-1)
    if offsets.dtype != torch.int64 or offsets.dim() != 1 or offsets.numel() < 1:
        raise _lib.FsnerfError("occgrid_filter: offsets must be int64 [R+1]")
    R, N, dev = offsets.numel() - 1, ts.numel(), ts.device
    if te.numel() != N or sig.numel() != N:
        raise _lib.FsnerfError(f"occgrid_filter: t_starts / t_ends / sigmas sizes {N} / {te.numel()} / {sig.numel()}")
    offsets = offsets.contiguous()
    out_offsets = torch.zeros(R + 1, dtype=torch.int64, device=dev)
    if N == 0 or R == 0:
        return torch.empty(0, dtype=torch.int64, device=dev), ts.new_empty(0), ts.new_empty(0), out_offsets
    counts = torch.empty(R, dtype=torch.int32, device=dev)
    lib = _lib.load()
    args = (R, ptr(offsets), ptr(ts), ptr(te), ptr(sig), float(early_stop_eps), float(alpha_thre))
    check(lib.fsnerf_occgrid_filter(*args, None, ptr(counts), None, None, None, _stream()), "fsnerf_occgrid_filter")
    torch.cumsum(counts, 0, out=out_offsets[1:])
    M = int(out_offsets[-1].item())  # survivor count: the filter's one host read
    ri = torch.empty(M, dtype=torch.int64, device=dev)
    ts_o, te_o = torch.empty(M, device=dev), torch.empty(M, device=dev)
    if M > 0:
        check(lib.fsnerf_occgrid_filter(*args, ptr(out_offsets), None, ptr(ri), ptr(ts_o), ptr(te_o), _stream()),
              "fsnerf_occgrid_filter")
    return ri, ts_o, te_o, out_offsets


def packed_points(ray_indices, t_starts, t_ends, rays_o, rays_d, want_dirs=False):
    """-> x [N,3] = rays_o[ri] + rays_d[ri] * (t_starts + t_ends)[:, None] / 2 (bit-identical to that torch
    expression) and, with want_dirs, dirs [N,3] = rays_d[ri] (else None)."""
    ts, te = _f32c(t_starts, "t_starts"), _f32c(t_ends, "t_ends")
    rays_o, rays_d = _f32c(rays_o, "rays_o"), _f32c(rays_d, "rays_d")
    N, dev = ts.numel(), ts.device
    if ray_indices.dtype != torch.int64 or ray_indices.numel() != N or te.numel() != N:
        raise _lib.FsnerfError("packed_points: ray_indices must be int64 with one entry per interval")
    if rays_o.shape != rays_d.shape or rays_o.dim() != 2 or rays_o.shape[1] != 3:
        raise _lib.FsnerfError(f"packed_points: rays must be [R,3], got {tuple(rays_o.shape)} / {tuple(rays_d.shape)}")
    x = torch.empty(N, 3, device=dev)
    dirs = torch.empty(N, 3, device=dev) if want_dirs else None
    check(_lib.load().fsnerf_packed_points(N, ptr(ray_indices.contiguous()), ptr(ts), ptr(te), ptr(rays_o),
                                           ptr(rays_d), ptr(x), ptr(dirs), _stream()), "fsnerf_packed_points")
    return x, dirs


def offsets_from_ray_indices(ray_indices, n_rays):
    """[R+1] int64 segment offsets of sorted packed ray indices"""
    if torch.are_deterministic_algorithms_enabled():
        # torch's CUDA bincount refuses to run in that mode; on sorted indices the offsets are
        # also where each ray's run starts (first index >= r), the same integers
        return torch.searchsorted(ray_indices, torch.arange(n_rays + 1, device=ray_indices.device))
    counts = torch.bincount(ray_indices, minlength=n_rays)
    offsets = torch.zeros(n_rays + 1, dtype=torch.int64, device=ray_indices.device)
    torch.cumsum(counts, 0, out=offsets[1:])
    return offsets


def composite_packed_forward(raw, t_starts, t_ends, offsets, bkgd=None):
    """raw [N,4] -> rgb [R,3], opacity [R,1], depth [R,1], weights [N], trans [N], alphas [N]"""
    raw, ts, te = _f32c(raw, "raw"), _f32c(t_starts, "t_starts"), _f32c(t_ends, "t_ends")
    R, N, dev = offsets.numel() - 1, ts.numel(), raw.device
    rgb, op, dp = torch.empty(R, 3, device=dev), torch.empty(R, 1, device=dev), torch.empty(R, 1, device=dev)
    w, tr, al = torch.empty(N, device=dev), torch.empty(N, device=dev), torch.empty(N, device=dev)
    check(_lib.load().fsnerf_composite_packed_forward(R, ptr(offsets), ptr(raw), ptr(ts), ptr(te),
                                                      ptr(_f32c(bkgd, "bkgd")), ptr(rgb), ptr(op), ptr(dp), ptr(w),
                                                      ptr(tr), ptr(al), _stream()), "fsnerf_composite_packed_forward")
    return rgb, op, dp, w, tr, al


def composite_packed_backward(raw, t_starts, t_ends, offsets, trans, d_rgb, d_opacity=None, d_depth=None,
                              d_weights=None, bkgd=None, want_d_bkgd=False):
    raw, ts, te = _f32c(raw, "raw"), _f32c(t_starts, "t_starts"), _f32c(t_ends, "t_ends")
    R = offsets.numel() - 1
    d_raw = torch.empty_like(raw)
    d_bkgd = torch.zeros(3, device=raw.device) if want_d_bkgd else None
    check(_lib.load().fsnerf_composite_packed_backward(
        R, ptr(offsets), ptr(raw), ptr(ts), ptr(te), ptr(_f32c(trans, "trans")), ptr(_f32c(bkgd, "bkgd")),
        ptr(_f32c(d_rgb, "d_rgb")), ptr(_f32c(d_opacity, "d_opacity")), ptr(_f32c(d_depth, "d_depth")),
        ptr(_f32c(d_weights, "d_weights")), ptr(d_raw), ptr(d_bkgd), _stream()), "fsnerf_composite_packed_backward")
    return d_raw, d_bkgd


def occgrid_update(occs, occ, cell_ids=None, decay=0.95):
    """in place: occs[c] = max(decay*occs[c], max of the candidates occ[i] in cell c)"""
    occ = _f32c(occ, "occ").reshape(-1)
    ws = torch.empty_like(occ)
    check(_lib.load().fsnerf_occgrid_update(occ.numel(), ptr(cell_ids), ptr(occ), float(decay), ptr(occs), ptr(ws),
                                            _stream()), "fsnerf_occgrid_update")


def occgrid_binarize(occs, threshold, binaries):
    check(_lib.load().fsnerf_occgrid_binarize(occs.numel(), ptr(occs), float(threshold), ptr(binaries), _stream()),
          "fsnerf_occgrid_binarize")


# -------------------------------------------------------------------- MLP
def make_cfg(n_layers=8, d_hidden=256, skip=(4,), n_freqs_pos=10, n_freqs_dir=4, log_space=True):
    mask = 0
    for s in skip:
        mask |= 1 << int(s)
    return NetCfg(n_layers, d_hidden, mask, n_freqs_pos, n_freqs_dir, int(bool(log_space)))


def mlp_param_count(cfg):
    n = _lib.load().fsnerf_mlp_param_count(C.byref(cfg))
    if n < 0:
        check(-1, "fsnerf_mlp_param_count")
    return n


def mlp_param_layout(cfg):
    """-> list of (offset, numel) in floats, one per state-dict tensor (reference order)."""
    off = (C.c_int64 * 64)()
    num = (C.c_int64 * 64)()
    n = _lib.load().fsnerf_mlp_param_layout(C.byref(cfg), off, num, 64)
    if n < 0:
        check(n, "fsnerf_mlp_param_layout")
    return [(off[i], num[i]) for i in range(n)]


def state_dict_names(cfg):
    """the reference's state_dict() keys, in order (src/core/models.py:96-108)"""
    mods = [f"layers.{i}" for i in range(cfg.n_layers)] + ["sigma", "connection", "branch", "rgb"]
    return [f"{m}.{k}" for m in mods for k in ("weight", "bias")]


def flatten_state_dict(cfg, sd, device):
    """state dict (reference keys) -> flat fp32 parameter buffer on `device`."""
    layout = mlp_param_layout(cfg)
    names = state_dict_names(cfg)
    if len(names) != len(layout) or set(names) != set(sd.keys()):
        raise _lib.FsnerfError("state dict keys do not match the network configuration")
    flat = torch.zeros(mlp_param_count(cfg), device=device)
    for (o, n), name in zip(layout, names):
        v = sd[name]
        if v.numel() != n:
            raise _lib.FsnerfError(f"state dict tensor {name}: {v.numel()} elements, expected {n}")
        flat[o:o + n] = v.detach().reshape(-1).to(device=device, dtype=torch.float32)
    return flat


def mlp_packed_bytes(cfg):
    n = _lib.load().fsnerf_mlp_packed_bytes(C.byref(cfg))
    if n < 0:
        check(-1, "fsnerf_mlp_packed_bytes")
    return n


def mlp_stash_bytes(cfg, n_samples):
    n = _lib.load().fsnerf_mlp_stash_bytes(C.byref(cfg), int(n_samples))
    if n < 0:
        check(-1, "fsnerf_mlp_stash_bytes")
    return n


def mlp_bwd_workspace_bytes(cfg, n_samples, deterministic=False):
    """bytes of the workspace mlp_backward needs (deterministic: that mode's, which is larger)"""
    lib = _lib.load()
    name = "fsnerf_mlp_bwd_workspace_bytes_deterministic" if deterministic else "fsnerf_mlp_bwd_workspace_bytes"
    n = getattr(lib, name)(C.byref(cfg), int(n_samples))
    if n < 0:
        check(-1, name)
    return n


def mlp_pack(cfg, params, packed=None):
    params = _f32c(params, "params")
    if packed is None:
        packed = torch.empty(mlp_packed_bytes(cfg), dtype=torch.uint8, device=params.device)
    check(_lib.load().fsnerf_mlp_pack(C.byref(cfg), ptr(params), ptr(packed), _stream()),
          "fsnerf_mlp_pack")
    return packed


def mlp_forward(cfg, params, packed, *, rays_o=None, rays_d=None, t_starts=None, t_ends=None,
                x=None, dirs=None, mask_pos=None, mask_dir=None, density_only=False, stash=None,
                out=None):
    """Either (rays_o, rays_d, t_starts[R,S], t_ends[R,S]) or (x[P,3], dirs[P,3]|None)."""
    params = _f32c(params, "params")
    if x is not None:
        x, dirs = _f32c(x, "x"), _f32c(dirs, "dirs")
        P, S = x.shape[0], 1
    else:
        rays_o, rays_d = _f32c(rays_o, "rays_o"), _f32c(rays_d, "rays_d")
        t_starts, t_ends = _f32c(t_starts, "t_starts"), _f32c(t_ends, "t_ends")
        P, S = t_starts.numel(), t_starts.shape[-1]
    if out is None:
        # density_only: False/0 full, True/1 sigma [P], 2 sigma into the .w slot of a zeroed [P,4]
        out = (torch.empty(P, device=params.device) if int(density_only) == 1 else
               torch.zeros(P, 4, device=params.device) if int(density_only) == 2 else
               torch.empty(P, 4, device=params.device))
    check(_lib.load().fsnerf_mlp_forward(
        C.byref(cfg), ptr(params), ptr(packed), P, S, ptr(rays_o), ptr(rays_d), ptr(t_starts),
        ptr(t_ends), ptr(x), ptr(dirs), ptr(_f32c(mask_pos, "mask_pos")),
        ptr(_f32c(mask_dir, "mask_dir")), int(density_only), ptr(out), ptr(stash), _stream()),
        "fsnerf_mlp_forward")
    return out


def mlp_backward(cfg, params, packed, n_samples, stash, out, d_out, grads, workspace,
                 density_only=False, deterministic=False):
    """Adds the MLP gradient to grads.  deterministic=True: bitwise reproducible gradients (same
    inputs, library build and GPU model); the workspace must then have
    mlp_bwd_workspace_bytes(cfg, n_samples, deterministic=True) bytes."""
    lib = _lib.load()
    name = "fsnerf_mlp_backward_deterministic" if deterministic else "fsnerf_mlp_backward"
    check(getattr(lib, name)(
        C.byref(cfg), ptr(params), ptr(packed), int(n_samples), ptr(stash), ptr(out),
        ptr(_f32c(d_out, "d_out")), int(density_only), ptr(grads), ptr(workspace), _stream()),
        name)
    return grads


# ------------------------------------------------------------- train step
def mse_loss_grad(rgb, gt, grad_scale, loss_sum, want_grad=True):
    rgb, gt = _f32c(rgb, "rgb"), _f32c(gt, "gt")
    d = torch.empty_like(rgb) if want_grad else None
    check(_lib.load().fsnerf_mse_loss_grad(rgb.numel(), ptr(rgb), ptr(gt), float(grad_scale),
                                           ptr(loss_sum), ptr(d), _stream()), "fsnerf_mse_loss_grad")
    return d


def adam_step(params, grads, m, v, lr, step, beta1=0.9, beta2=0.999, eps=1e-8):
    check(_lib.load().fsnerf_adam_step(params.numel(), ptr(params), ptr(grads), ptr(m), ptr(v),
                                       float(lr), beta1, beta2, eps, int(step), _stream()),
          "fsnerf_adam_step")


def reg_segments(cfg, n_nets=1):
    """flat [begin, end) ranges of the tensors the reference's weight penalty covers:
    '"weight" in name and param.shape[0] > 3' (src/run-nerf.py:272-273) — every weight except
    sigma.weight [1,H] and rgb.weight [3,H/2] — for n_nets networks laid back to back."""
    n_net = mlp_param_count(cfg)
    segs = []
    for i in range(n_nets):
        for (off, numel), name in zip(mlp_param_layout(cfg), state_dict_names(cfg)):
            if "weight" in name and name not in ("sigma.weight", "rgb.weight"):
                segs.append((i * n_net + off, i * n_net + off + numel))
    return segs


def adam_step_reg(params, grads, m, v, lr, step, mode, alpha, segments, seg_sums,
                  beta1=0.9, beta2=0.999, eps=1e-8, deterministic=False):
    """Adam with the weight-norm penalty fused in; mode 'l1' or anything else (Frobenius),
    like the reference's `args.reg` switch.  seg_sums [len(segments)] device floats.
    deterministic=True: the per-tensor sums are added in one fixed order (reproducible update)."""
    n = len(segments)
    b = (C.c_int64 * n)(*[s[0] for s in segments])
    e = (C.c_int64 * n)(*[s[1] for s in segments])
    name = "fsnerf_adam_step_reg_deterministic" if deterministic else "fsnerf_adam_step_reg"
    check(getattr(_lib.load(), name)(params.numel(), ptr(params), ptr(grads), ptr(m), ptr(v),
                                     float(lr), beta1, beta2, eps, int(step),
                                     1 if mode == "l1" else 2, float(alpha), n, b, e,
                                     ptr(seg_sums), _stream()), name)


# -------------------------------------------------------------- profiling
def profile_enable(on=True):
    check(_lib.load().fsnerf_profile_enable(int(bool(on))), "fsnerf_profile_enable")


def profile_read():
    """-> {kernel name: (total_ms, launches)} since profile_enable(True)"""
    n_max = 32
    names = C.create_string_buffer(32 * n_max)
    ms = (C.c_float * n_max)()
    cnt = (C.c_int * n_max)()
    n = _lib.load().fsnerf_profile_read(n_max, names, ms, cnt)
    if n < 0:
        check(n, "fsnerf_profile_read")
    raw = names.raw
    return {raw[32 * i:32 * (i + 1)].split(b"\0")[0].decode(): (ms[i], cnt[i]) for i in range(n)}
