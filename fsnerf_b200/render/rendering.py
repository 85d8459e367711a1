"""Drop-in for the reference's ``render.rendering`` entry points
(/root/reference/src/render/rendering.py:25-248): ``render_rays``,
``render_frame``, ``render_path`` with the same signatures and return
structures.  Sampling (stratified + hierarchical sample_pdf, per
BASELINE.json north_star, standing in for nerfacc's occupancy-grid sampler),
the MLP and the compositor run in the CUDA kernels of libfsnerf_b200.so.
"""
import os
import weakref
from typing import Optional, Tuple

import numpy as np
import torch
from torch import nn, Tensor

from .. import ops
from .._lib import FsnerfError
from ..utils import utilities as U

to8b = lambda x: (255 * np.clip(x, 0, 1)).astype(np.uint8)  # noqa: E731  (reference :22)


class _Token:
    """lifetime marker of one forward's claim on a model's cached scratch buffers"""
    __slots__ = ("__weakref__",)


def _claim(model, key, nbytes, device):
    """A device scratch buffer cached on the model (the multi-GB activation stash and the backward
    ring are the same size every step of the reference's loop: no allocator round trip per step).
    A buffer still claimed by a live autograd graph (two forwards before a backward) is left alone
    and a fresh one is handed out.  -> (buffer, token); drop the token to release the claim."""
    cache = model.__dict__.setdefault("_scratch", {})
    buf, owner = cache.get(key, (None, None))
    busy = owner is not None and owner() is not None
    if buf is None or busy or buf.numel() < nbytes or buf.device != device:
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        if busy:
            return buf, _Token()  # one-off: the cached buffer stays with its owner
    tok = _Token()
    cache[key] = (buf, weakref.ref(tok))
    return buf, tok


class _RenderFunction(torch.autograd.Function):
    """rays + intervals -> MLP (fused encode + tcgen05 MLP) -> compositing.
    One autograd node so that loss.backward() (src/run-nerf.py:282) reaches the
    model parameters and the background colour."""

    @staticmethod
    def forward(ctx, model, rays_o, rays_d, ts, te, bkgd, flags, need_grad, *params):
        ctx.set_materialize_grads(False)  # unused outputs (weights, raw, ...) arrive as None, not as zero tensors
        R, S = ts.shape
        packed = model._refresh_packed()
        stash = tok = None
        if need_grad:
            stash, tok = _claim(model, "stash", ops.mlp_stash_bytes(model.cfg, R * S), ts.device)
        raw = ops.mlp_forward(model.cfg, model._flat, packed, rays_o=rays_o, rays_d=rays_d,
                              t_starts=ts, t_ends=te, mask_pos=model.mask_pos,
                              mask_dir=model.mask_dir, stash=stash)
        bk = None if bkgd is None else bkgd.detach()
        rgb, op, dp, w, _, _ = ops.composite_forward(raw.view(R, S, 4), ts, te, bkgd=bk, flags=flags)
        ctx.model, ctx.packed, ctx.stash, ctx.tok, ctx.flags, ctx.shape = model, packed, stash, tok, flags, (R, S)
        ctx.has_bkgd = bkgd is not None
        ctx.save_for_backward(raw, ts, te, bk if bk is not None else raw.new_empty(0))
        return rgb, op, dp, w, raw

    @staticmethod
    def backward(ctx, d_rgb, d_op, d_dp, d_w, d_raw_in):
        model = ctx.model
        raw, ts, te, bk = ctx.saved_tensors
        R, S = ctx.shape
        bk = bk if ctx.has_bkgd else None
        cont = lambda g: None if g is None else g.contiguous()  # noqa: E731  (the kernel takes NULL for an absent gradient)
        if d_rgb is None:
            d_rgb = torch.zeros(R, 3, device=raw.device)
        d_raw, d_bk = ops.composite_backward(raw.view(R, S, 4), ts, te, d_rgb.contiguous(), cont(d_op), cont(d_dp),
                                             cont(d_w), bkgd=bk, flags=ctx.flags, want_d_bkgd=ctx.has_bkgd)
        if d_raw_in is not None:
            # gradients that reach the raw samples directly, e.g. the occlusion regulariser on
            # extras["sigmas"] (src/run-nerf.py:260-264): added to the compositor's
            d_raw = d_raw.view(-1, 4).add_(d_raw_in.reshape(-1, 4))
        grads = torch.zeros_like(model._flat)
        ws, wtok = _claim(model, "bwd_ws", ops.mlp_bwd_workspace_bytes(model.cfg, R * S), raw.device)
        ops.mlp_backward(model.cfg, model._flat, ctx.packed, R * S, ctx.stash, raw, d_raw.view(-1, 4), grads, ws)
        del wtok
        ctx.tok = ctx.stash = None  # the stash can be reused by the next forward
        model._last_flat_grad = grads  # parallel.allreduce_module_gradients reduces this buffer in one collective
        views = [grads[o:o + n].view(p.shape) for (o, n), p in zip(model._layout, model._param_list())]
        return (None, None, None, None, None, d_bk, None, None, *views)


class _LazyExtras(dict):
    """nerfacc's extras dict (weights / alphas / trans / sigmas / rgbs).  The reference's loop reads
    only ``sigmas`` (src/run-nerf.py:262): ``alphas`` and ``trans`` are computed on first access
    instead of being written by every compositing launch."""

    def __init__(self, lazy, *a, **kw):
        super().__init__(*a, **kw)
        self._lazy = lazy

    def _materialise(self):
        if self._lazy is not None:
            raw, ts, te, bk, flags = self._lazy
            self._lazy = None
            with torch.no_grad():
                *_, al, tr = ops.composite_forward(raw.detach().view(ts.shape[0], ts.shape[1], 4), ts, te, bkgd=bk,
                                                   flags=flags, extras=True)
            dict.__setitem__(self, "alphas", al.reshape(-1))
            dict.__setitem__(self, "trans", tr.reshape(-1))

    def __missing__(self, key):
        if key in ("alphas", "trans") and self._lazy is not None:
            self._materialise()
            return dict.__getitem__(self, key)
        raise KeyError(key)

    def __contains__(self, key):
        return dict.__contains__(self, key) or (key in ("alphas", "trans") and self._lazy is not None)

    def get(self, key, default=None):
        return self[key] if key in self else default

    # enumerating the dict shows every key nerfacc's has
    def __iter__(self):
        self._materialise()
        return dict.__iter__(self)

    def __len__(self):
        self._materialise()
        return dict.__len__(self)

    def keys(self):
        self._materialise()
        return dict.keys(self)

    def items(self):
        self._materialise()
        return dict.items(self)

    def values(self):
        self._materialise()
        return dict.values(self)


def volume_render(model, rays_o, rays_d, t_starts, t_ends, render_bkgd=None, flags=0):
    """Stands in for ``nerfacc.volrend.rendering`` + the ``rgb_sigma_fn`` closure
    (reference :76-96) on a dense [R,S] sample layout.
    -> (rgb[R,3], opacity[R,1], depth[R,1], weights[R,S], raw[R*S,4])"""
    params = model._param_list()
    # (grad mode is always off inside Function.forward, so decide here)
    need_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in params) or (
        render_bkgd is not None and render_bkgd.requires_grad))
    return _RenderFunction.apply(model, rays_o, rays_d, t_starts, t_ends, render_bkgd, flags, need_grad,
                                 *params)


class HierarchicalEstimator(nn.Module):
    """Estimator-shaped object (the reference builds an
    ``OccGridEstimator(roi_aabb, resolution, levels)``, src/run-nerf.py:96-98, and
    calls ``.sampling`` / ``.update_every_n_steps`` / ``.train`` / ``.eval`` /
    ``.to``).  Sampling is stratified in [near, far] (``n_coarse`` points) and,
    when ``n_fine > 0``, refined by sample_pdf over the weights of a coarse pass
    through ``proposal_model`` (the canonical coarse network)."""

    def __init__(self, roi_aabb=None, resolution: int = 128, levels: int = 1, *, near: float = 2.0,
                 far: float = 6.0, n_coarse: int = 64, n_fine: int = 0,
                 proposal_model: Optional[nn.Module] = None) -> None:
        super().__init__()
        self.roi_aabb, self.resolution, self.levels = roi_aabb, resolution, levels
        self.near, self.far = float(near), float(far)
        self.n_coarse, self.n_fine = int(n_coarse), int(n_fine)
        if self.n_fine > 0 and proposal_model is None:
            raise FsnerfError("HierarchicalEstimator: n_fine > 0 needs a proposal (coarse) model")
        self.proposal_model = proposal_model
        self._u_strat = self._u_pdf = None
        self.last = {}
        self._const = {}  # per (device, shape) constants: white background, packed ray indices

    def set_uniforms(self, u_strat: Optional[Tensor], u_pdf: Optional[Tensor]) -> None:
        """Explicit uniforms for the next sampling() call (parity tests feed the same
        ones to the oracle); otherwise the samplers draw them in-kernel, keyed by a 64-bit seed
        taken from torch's CPU generator (so torch.manual_seed reproduces a run, as it does for
        the reference's torch.rand)."""
        self._u_strat, self._u_pdf = u_strat, u_pdf

    @property
    def samples_per_ray(self) -> int:
        return self.n_coarse + self.n_fine

    def sampling(self, rays_o, rays_d, sigma_fn=None, render_step_size=None, stratified=False,
                 near_plane=None, far_plane=None, white_bkgd=False):
        """-> packed (ray_indices[N] int64, t_starts[N], t_ends[N]), N = R*S
        (same triple as OccGridEstimator.sampling, reference :66-74).  The
        reference passes near_plane=0 / far_plane=1e10 and ignores the dataset
        bounds (App. C3): bounds come from this object."""
        R = rays_o.shape[0]
        dev = rays_o.device
        us, up = self._u_strat, self._u_pdf
        self._u_strat = self._u_pdf = None
        seeds = (None, None)
        if stratified and (us is None or (up is None and self.n_fine > 0)):
            seeds = [int(v) for v in torch.empty(2, dtype=torch.int64).random_()]
        ts, te = ops.sample_stratified(R, self.n_coarse, self.near, self.far, us if stratified else None,
                                       device=dev, seed=seeds[0] if stratified and us is None else None)
        self.last = {}
        if self.n_fine > 0:
            bk = None
            if white_bkgd:
                bk = self._const.get(("white", dev))
                if bk is None:
                    bk = self._const[("white", dev)] = torch.ones(3, device=dev)
            if torch.is_grad_enabled() or stratified:
                rgb_c, op_c, dp_c, w_c, _ = volume_render(self.proposal_model, rays_o, rays_d, ts, te, bk)
                self.last = dict(rgb_coarse=rgb_c, opacity_coarse=op_c, depth_coarse=dp_c,
                                 weights_coarse=w_c, t_starts_coarse=ts, t_ends_coarse=te)
            else:
                # inference (render_frame / render_path / evaluation: train=False under no_grad): only the
                # WEIGHTS of the proposal pass are needed — skip its view branch (density-only
                # forward writing sigma into the compositor's (rgb, sigma) layout)
                pm = self.proposal_model
                raw_c = ops.mlp_forward(pm.cfg, pm._flat, pm._refresh_packed(), rays_o=rays_o, rays_d=rays_d,
                                        t_starts=ts, t_ends=te, mask_pos=pm.mask_pos, mask_dir=pm.mask_dir,
                                        density_only=2)
                _, op_c, dp_c, w_c, _, _ = ops.composite_forward(raw_c.view(R, self.n_coarse, 4), ts, te, bkgd=bk)
                self.last = dict(opacity_coarse=op_c, depth_coarse=dp_c, weights_coarse=w_c,
                                 t_starts_coarse=ts, t_ends_coarse=te)
            ts, te, *_ = ops.sample_pdf(ts, w_c.detach(), self.n_fine, self.far,
                                        up if stratified else None, want_aux=False,
                                        seed=seeds[1] if stratified and up is None else None)
        S = ts.shape[1]
        ray_indices = self._const.get(("ri", dev, R, S))  # the same packed index vector every step
        if ray_indices is None:
            self._const = {k: v for k, v in self._const.items() if k[0] != "ri"}
            ray_indices = self._const[("ri", dev, R, S)] = torch.arange(R, device=dev).repeat_interleave(S)
        self._dense = (ts, te)
        return ray_indices, ts.reshape(-1), te.reshape(-1)

    def update_every_n_steps(self, step=None, occ_eval_fn=None, occ_thre=None, **kw) -> None:
        """No occupancy grid on this path (SURVEY.md §8 row a9): kept so that the
        reference's train loop (src/run-nerf.py:293-295) runs unchanged."""
        return None


class _PackedCompositeFunction(torch.autograd.Function):
    """nerfacc.volrend.rendering on packed samples (reference :89-96) as one autograd node:
    raw [N,4] = (rgb, sigma) of the samples, ray r owning [offsets[r], offsets[r+1])."""

    @staticmethod
    def forward(ctx, raw, ts, te, offsets, bkgd):
        ctx.set_materialize_grads(False)
        bk = None if bkgd is None else bkgd.detach()
        rgb, op, dp, w, tr, al = ops.composite_packed_forward(raw, ts, te, offsets, bkgd=bk)
        ctx.has_bkgd = bkgd is not None
        ctx.save_for_backward(raw, ts, te, offsets, tr, bk if bk is not None else raw.new_empty(0))
        ctx.mark_non_differentiable(tr, al)
        return rgb, op, dp, w, tr, al

    @staticmethod
    def backward(ctx, d_rgb, d_op, d_dp, d_w, _d_tr, _d_al):
        raw, ts, te, offsets, tr, bk = ctx.saved_tensors
        R = offsets.numel() - 1
        zero = lambda g, shape: torch.zeros(shape, device=raw.device) if g is None else g.contiguous()  # noqa: E731
        d_raw, d_bk = ops.composite_packed_backward(raw, ts, te, offsets, tr, zero(d_rgb, (R, 3)), zero(d_op, (R, 1)),
                                                    zero(d_dp, (R, 1)), None if d_w is None else d_w.contiguous(),
                                                    bkgd=bk if ctx.has_bkgd else None, want_d_bkgd=ctx.has_bkgd)
        return d_raw, None, None, None, d_bk


class OccGridEstimator(nn.Module):
    """Drop-in for ``nerfacc.estimators.occ_grid.OccGridEstimator`` as the reference uses it
    (construction src/run-nerf.py:92-98, ``.sampling`` src/render/rendering.py:66-74,
    ``.update_every_n_steps`` src/run-nerf.py:288-295): multi-level binary occupancy grid,
    fixed-step ray marching through the occupied cells, transmittance visibility filter,
    EMA grid update.  Kernels: csrc/occgrid.cu; semantics: oracle/occgrid.py (nerfacc 0.5.3 is
    not on the box — parity unpinned against it)."""

    def __init__(self, roi_aabb, resolution: int = 128, levels: int = 1, **kwargs) -> None:
        super().__init__()
        roi = torch.as_tensor(roi_aabb, dtype=torch.float32).flatten()
        assert roi.numel() == 6, f"Expected [6] aabb, got {tuple(roi.shape)}"
        assert isinstance(resolution, int), "cubic grids only: resolution must be an int"
        centre, half = (roi[:3] + roi[3:]) / 2, (roi[3:] - roi[:3]) / 2
        aabbs = torch.stack([torch.cat([centre - half * 2 ** l, centre + half * 2 ** l]) for l in range(levels)])
        self.levels, self.resolution = int(levels), int(resolution)
        self.cells_per_lvl = self.resolution ** 3
        self.register_buffer("aabbs", aabbs)
        self.register_buffer("occs", torch.zeros(self.levels * self.cells_per_lvl))
        self.register_buffer("binaries", torch.zeros((self.levels,) + (self.resolution,) * 3, dtype=torch.bool))
        self._jitter = None

    def set_uniforms(self, jitter: Optional[Tensor]) -> None:
        """explicit per-ray U[0,1) for the next stratified sampling() call (parity tests)"""
        self._jitter = jitter

    @torch.no_grad()
    def sampling(self, rays_o: Tensor, rays_d: Tensor, sigma_fn=None, alpha_fn=None, near_plane: float = 0.0,
                 far_plane: float = 1e10, t_min: Optional[Tensor] = None, t_max: Optional[Tensor] = None,
                 render_step_size: float = 1e-3, early_stop_eps: float = 1e-4, alpha_thre: float = 0.0,
                 stratified: bool = False, cone_angle: float = 0.0, **kwargs):
        """-> packed (ray_indices int64 [N], t_starts [N], t_ends [N])"""
        if cone_angle != 0.0 or alpha_fn is not None or t_max is not None:
            raise FsnerfError("OccGridEstimator.sampling: cone_angle / alpha_fn / t_max are not used by the "
                              "reference and not implemented")
        R, dev = rays_o.shape[0], rays_o.device
        near_planes = torch.full((R,), float(near_plane), device=dev)
        if t_min is not None:
            near_planes = torch.clamp(near_planes, min=t_min)
        if stratified:
            u = self._jitter if self._jitter is not None else torch.rand(R, device=dev)
            near_planes = near_planes + u * render_step_size
        self._jitter = None
        ri, ts, te, offsets = ops.occgrid_march(rays_o, rays_d, self.binaries.view(torch.uint8), self.aabbs,
                                                render_step_size, far=far_plane, near_planes=near_planes)
        if (alpha_thre > 0.0 or early_stop_eps > 0.0) and sigma_fn is not None:
            if alpha_thre > 0.0:  # min(alpha_thre, mean) <= 0 disables the alpha test either way
                alpha_thre = min(alpha_thre, self.occs.mean().item())
            sigmas = sigma_fn(ts, te, ri) if ts.numel() else ts.new_empty(0)
            assert sigmas.shape == ts.shape, f"sigmas must have shape of (N,)! Got {tuple(sigmas.shape)}"
            ri, ts, te, _ = ops.occgrid_filter(ts, te, offsets, sigmas, early_stop_eps, alpha_thre)
        return ri, ts, te

    @torch.no_grad()
    def update_every_n_steps(self, step: int, occ_eval_fn=None, occ_thre: float = 1e-2, ema_decay: float = 0.95,
                             warmup_steps: int = 256, n: int = 16, generator: Optional[torch.Generator] = None) -> None:
        """generator: draws the cell subset and the in-cell points (torch's default generator when None)"""
        if not self.training:
            raise RuntimeError("You should only call this function only during training. Please call "
                               "_update() directly if you want to update the field during inference.")
        if step % n == 0 and self.training:
            self._update(step, occ_eval_fn, occ_thre, ema_decay, warmup_steps, generator=generator)

    def _sample_cells(self, step, warmup_steps, lvl, generator=None):
        """cell ids evaluated this round: all during warm-up, else 1/4 uniform + up to 1/4 occupied"""
        dev = self.occs.device
        if step < warmup_steps:
            return None
        n = self.cells_per_lvl // 4
        uniform = torch.randint(self.cells_per_lvl, (n,), device=dev, generator=generator)
        occupied = torch.nonzero(self.binaries[lvl].flatten())[:, 0]
        if occupied.numel() > n:
            occupied = occupied[torch.randint(occupied.numel(), (n,), device=dev, generator=generator)]
        return torch.cat([uniform, occupied])

    @torch.no_grad()
    def _update(self, step, occ_eval_fn, occ_thre=1e-2, ema_decay=0.95, warmup_steps=256, rand=None,
                generator=None) -> None:
        res, dev = self.resolution, self.occs.device
        for lvl in range(self.levels):
            ids = self._sample_cells(step, warmup_steps, lvl, generator)
            flat = torch.arange(self.cells_per_lvl, device=dev) if ids is None else ids
            coords = torch.stack([flat // (res * res), (flat // res) % res, flat % res], -1).float()
            u = torch.rand(coords.shape, device=dev, generator=generator) if rand is None else rand[lvl]
            x = (coords + u) / res
            x = self.aabbs[lvl, :3] + x * (self.aabbs[lvl, 3:] - self.aabbs[lvl, :3])
            occ = occ_eval_fn(x).reshape(-1)
            ops.occgrid_update(self.occs[lvl * self.cells_per_lvl:(lvl + 1) * self.cells_per_lvl], occ,
                               cell_ids=ids, decay=ema_decay)
        thre = torch.clamp(self.occs[self.occs >= 0].mean(), max=occ_thre).item()
        ops.occgrid_binarize(self.occs, thre, self.binaries.view(torch.uint8))


def _render_rays_packed(rays_o, rays_d, estimator, model, train, white_bkgd, render_step_size, device):
    """the reference's own structure (src/render/rendering.py:56-107) on packed samples"""
    R = rays_o.shape[0]

    def sigma_fn(t_starts, t_ends, ray_indices):  # :58-64
        x = rays_o[ray_indices] + rays_d[ray_indices] * (t_starts + t_ends)[:, None] / 2.0
        return model(x).squeeze(-1)

    ray_indices, t_starts, t_ends = estimator.sampling(
        rays_o, rays_d, sigma_fn=sigma_fn, render_step_size=render_step_size, stratified=train,
        near_plane=0.0, far_plane=1e10)
    render_bkgd = white_bkgd * torch.ones((3,), device=device, requires_grad=train)
    t_vals = (t_starts + t_ends) / 2.0
    try:  # :88-103 — nerfacc's shape assertions and the reference's answer to them
        if t_starts.numel():  # :76-84
            dirs = rays_d[ray_indices]
            x = rays_o[ray_indices] + dirs * (t_starts + t_ends)[:, None] / 2.0
            out = model(x, dirs)
            rgbs, sigmas = out[..., :3], out[..., -1].squeeze(-1)  # one surviving sample: squeeze -> 0-d
            assert rgbs.shape[-1] == 3, f"rgbs must have 3 channels, got {rgbs.shape}"
            assert sigmas.shape == t_starts.shape, f"sigmas must have shape of (N,)! Got {sigmas.shape}"
            raw = out
        else:
            raw = torch.zeros(0, 4, device=device)
        offsets = ops.offsets_from_ray_indices(ray_indices, R)
        rgb, opacity, depth, weights, trans, alphas = _PackedCompositeFunction.apply(raw, t_starts, t_ends, offsets,
                                                                                     render_bkgd)
        extras = dict(weights=weights, alphas=alphas, trans=trans, sigmas=raw[:, 3], rgbs=raw[:, :3])
        output = (rgb, opacity, depth, extras)
    except AssertionError:
        if os.environ.get("FSNERF_DEBUG_FALLBACK"):  # the reference swallows it silently
            import traceback
            traceback.print_exc()
        output = (torch.ones_like(rays_o) * white_bkgd, None,
                  torch.zeros_like(rays_o[:, 0].unsqueeze(1), dtype=torch.float32), None)
    return output, ray_indices, t_vals


def render_rays(rays_o: Tensor, rays_d: Tensor, estimator, model: nn.Module, train: bool = False,
                white_bkgd: bool = False, render_step_size: float = 5e-3,
                device: torch.device = torch.device("cuda")) -> Tuple[Tensor]:
    """reference: src/render/rendering.py:25-107.
    -> ((rgb[R,3], opacity[R,1], depth[R,1], extras), ray_indices[N], t_vals[N])
    extras: weights/alphas/trans/sigmas/rgbs (packed [N]) like nerfacc's, plus
    rgb_coarse/opacity_coarse/depth_coarse when the estimator is hierarchical."""
    device = torch.device(device)
    if device.type != "cuda":
        raise FsnerfError("render_rays: fsnerf_b200 has no CPU path; pass a CUDA device")
    rays_o = rays_o.to(device=device, dtype=torch.float32).contiguous()  # also un-expands stride-0 origins
    rays_d = rays_d.to(device=device, dtype=torch.float32).contiguous()
    R = rays_o.shape[0]
    if isinstance(estimator, OccGridEstimator):
        return _render_rays_packed(rays_o, rays_d, estimator, model, train, white_bkgd, render_step_size, device)
    ray_indices, t_starts, t_ends = estimator.sampling(
        rays_o, rays_d, sigma_fn=None, render_step_size=render_step_size, stratified=train,
        near_plane=0.0, far_plane=1e10, white_bkgd=white_bkgd)
    S = t_starts.numel() // max(R, 1)
    ts, te = t_starts.view(R, S), t_ends.view(R, S)
    render_bkgd = white_bkgd * torch.ones((3,), device=device, requires_grad=train)
    rgb, opacity, depth, weights, raw = volume_render(model, rays_o, rays_d, ts, te, render_bkgd)
    extras = _LazyExtras((raw, ts, te, render_bkgd.detach(), 0), weights=weights.reshape(-1),
                         sigmas=raw[:, 3], rgbs=raw[:, :3])
    extras.update(getattr(estimator, "last", {}))
    t_vals = (t_starts + t_ends) / 2.0
    return (rgb, opacity, depth, extras), ray_indices, t_vals


def render_frame(hwf, near: float, far: float, pose: Tensor, chunksize: int, estimator, model: nn.Module,
                 train: bool = False, ndc: bool = False, white_bkgd: bool = False,
                 render_step_size: float = 5e-3, device: torch.device = torch.device("cuda"),
                 compat_positional_bug: bool = False, pixel_range: Optional[Tuple[int, int]] = None):
    """reference: src/render/rendering.py:110-177 -> (img[H,W,3], depth[H,W]).
    The reference passes ``white_bkgd`` positionally into render_rays' ``train``
    slot (:160-168; SURVEY.md App. C1); that is reproduced only with
    ``compat_positional_bug=True``.  ``pixel_range=(a,b)`` renders the flattened
    pixels [a,b) only (multi-GPU pixel partition) and returns flat [b-a,3],[b-a]."""
    H, W, focal = hwf
    H, W = int(H), int(W)
    device = torch.device(device)
    a, b = (0, H * W) if pixel_range is None else pixel_range
    pose = pose.to(device=device, dtype=torch.float32)
    rays_o, rays_d, _ = ops.gen_rays(pose[None].contiguous(), H, W, float(focal), first_id=a, n_rays=b - a,
                                     ndc=ndc, ndc_near=1.0)
    img, depth_map = [], []
    for ro, rd in zip(U.get_chunks(rays_o, chunksize), U.get_chunks(rays_d, chunksize)):
        if compat_positional_bug:
            out = render_rays(ro, rd, estimator, model, white_bkgd, render_step_size=render_step_size,
                              device=device)
        else:
            out = render_rays(ro, rd, estimator, model, train=train, white_bkgd=white_bkgd,
                              render_step_size=render_step_size, device=device)
        (rgb, _, dpt, _), *_ = out
        img.append(rgb)
        depth_map.append(dpt)
    img = torch.cat(img, dim=0)
    depth = torch.cat(depth_map, dim=0).clamp(near, far)
    if pixel_range is not None:
        return img, depth.reshape(-1)
    return img.reshape(H, W, 3), depth.reshape(H, W)


def render_path(render_poses: Tensor, hwf, near: float, far: float, chunksize: int, model: nn.Module,
                estimator, ndc: bool = False, train: bool = False, white_bkgd: bool = False,
                render_step_size: float = 5e-3, device: torch.device = torch.device("cuda"),
                rank: int = 0, world_size: int = 1):
    """reference: src/render/rendering.py:180-248 -> (frames[F,H,W,3], d_frames[F,H,W])
    numpy fp32.  With world_size > 1 the flattened F*H*W pixel range is split in
    contiguous slices, rank r renders slice r and returns only its flat slice
    (frames[n_r,3], d_frames[n_r], (start, stop)): no collective is needed."""
    H, W, _ = hwf
    H, W = int(H), int(W)
    F = len(render_poses)
    total = F * H * W
    start, stop = (total * rank) // world_size, (total * (rank + 1)) // world_size
    frames, d_frames = [], []
    dev_rgb, dev_dep = [], []

    def flush():  # frames stay on the device and cross to the host in batches: no per-frame sync
        if dev_rgb:
            frames.append(torch.cat(dev_rgb).cpu().numpy())
            d_frames.append(torch.cat(dev_dep).cpu().numpy())
            dev_rgb.clear()
            dev_dep.clear()
    with torch.no_grad():
        for i, pose in enumerate(render_poses):
            a, b = max(start, i * H * W), min(stop, (i + 1) * H * W)
            if a >= b:
                continue
            rng = None if (a == i * H * W and b == (i + 1) * H * W) else (a - i * H * W, b - i * H * W)
            rgb, depth = render_frame(hwf, near, far, pose, chunksize, estimator, model, train=train, ndc=ndc,
                                      white_bkgd=white_bkgd, render_step_size=render_step_size,
                                      device=device, pixel_range=rng)
            dev_rgb.append(rgb.reshape(-1, 3).detach())
            dev_dep.append(depth.reshape(-1).detach())
            if sum(t.shape[0] for t in dev_rgb) >= 64 * 1024 * 1024:  # <= 1 GiB of rgb resident
                flush()
        flush()
    frames = [np.concatenate(frames, 0)] if frames else []
    d_frames = [np.concatenate(d_frames, 0)] if d_frames else []
    if world_size == 1:
        return frames[0].reshape(F, H, W, 3), d_frames[0].reshape(F, H, W)
    if not frames:
        return np.zeros((0, 3), np.float32), np.zeros((0,), np.float32), (start, stop)
    return frames[0], d_frames[0], (start, stop)
