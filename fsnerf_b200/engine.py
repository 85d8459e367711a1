"""Fused host driver of the hot path: one training step / one render chunk as a
fixed sequence of kernel launches on the current stream, no autograd, no
per-step allocation after warm-up.  This is what ``bench.py`` times; the
drop-in modules (render.rendering / core.models) wrap the same kernels in
autograd for the reference's own train loop.

Train step (src/run-nerf.py:232-285 with the sampler replaced per north_star):
  gen_rays* -> stratified -> coarse MLP -> composite -> sample_pdf -> fine MLP
  -> composite -> MSE grads -> composite bwd x2 -> MLP bwd x2 (heads + one fused
  dgrad/wgrad launch each) -> [NCCL all-reduce of the flat gradient] -> Adam on the flat buffer.
With sampler="occgrid" (the reference's own sampler, src/run-nerf.py:92-98,288-295):
  occgrid_march -> packed_points -> density MLP -> occgrid_filter -> packed_points -> MLP
  -> packed composite -> MSE grads -> packed composite bwd -> MLP bwd -> [all-reduce] -> Adam
  -> grid update every 16th step.
Coarse and fine networks live in ONE flat fp32 parameter/gradient/moment buffer
so the data-parallel exchange is a single collective (SURVEY.md §8e).
"""
import math
from typing import Optional

import torch

from . import ops
from ._lib import FsnerfError
from .core.models import NeRF, freq_mask
from .parallel import allreduce_gradients, loss_grad_scale
from .render.rendering import OccGridEstimator

_M64 = (1 << 64) - 1


def jitter_seeds(seed: int, rank: int, draw: int):
    """Keys of the (stratified, pdf) uniform streams of one step: splitmix64 of (construction
    seed, rank, draw counter), so ranks and steps never share a stream."""
    keys = []
    for which in (0, 1):
        z = (seed * 0x9E3779B97F4A7C15 + (rank << 40) + 2 * draw + which) & _M64
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
        keys.append(z ^ (z >> 31))
    return keys


def grid_seed(seed: int, step: int) -> int:
    """Key of the occupancy-grid update of train step `step`: (seed, step) only, never the rank,
    so every rank of a data-parallel run draws the same cells and points and holds the same grid."""
    return jitter_seeds(seed, 0, -1 - step)[0]


class HotPath:
    """sampler="hierarchical" (default): stratified + sample_pdf, coarse and fine networks.
    sampler="occgrid": the reference's own configuration (src/run-nerf.py:92-98,232-295): ONE
    network, an owned render.rendering.OccGridEstimator(roi_aabb, grid_resolution, grid_levels) for the
    grid, fixed-step marching (render_step_size, near 0, far 1e10) with the transmittance visibility
    filter (early_stop_eps 1e-4, alpha_thre 0) on a density-only forward, then a training forward of
    the survivors.  Its train_step reads two sizes on the host: N (candidates) and M (survivors).
    near / far / n_coarse / n_fine do not apply to it.

    deterministic=True: the MLP backward and the weight-norm penalty run in their deterministic
    mode, so on one GPU two engines built from the same seed and fed the same rays hold bitwise
    identical parameters, Adam moments, occupancy grid and renders after any number of steps
    (same library build and GPU model).  The loss sums stay atomics: they are only reported."""

    def __init__(self, n_coarse=64, n_fine=128, near=2.0, far=6.0, white_bkgd=True, device="cuda",
                 n_layers=8, d_hidden=256, skip=(4,), n_freqs=10, n_freqs_dir=4, log_space=True,
                 seed=42, lr=5e-4, process_group=None, world_size=None, sampler="hierarchical",
                 roi_aabb=None, grid_resolution=128, grid_levels=1, render_step_size=5e-3, deterministic=False):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise FsnerfError("HotPath: CUDA device required (no CPU path)")
        if sampler not in ("hierarchical", "occgrid"):
            raise FsnerfError(f"HotPath: unknown sampler {sampler!r} (hierarchical | occgrid)")
        ops.require_device(self.device.index if self.device.index is not None else torch.cuda.current_device())
        self.occgrid = sampler == "occgrid"
        self.deterministic = bool(deterministic)
        self.n_coarse, self.n_fine = int(n_coarse), int(n_fine)
        self.near, self.far, self.white_bkgd = float(near), float(far), bool(white_bkgd)
        self.cfg = ops.make_cfg(n_layers, d_hidden, skip, n_freqs, n_freqs_dir, log_space)
        self.layout = ops.mlp_param_layout(self.cfg)
        self.names = ops.state_dict_names(self.cfg)
        self.n_net = ops.mlp_param_count(self.cfg)
        self.hier = self.n_fine > 0 and not self.occgrid
        n_nets = 2 if self.hier else 1
        kw = {"pos_fn": {"n_freqs": n_freqs, "log_space": log_space},
              "dir_fn": {"n_freqs": n_freqs_dir, "log_space": log_space}}
        # seed-42 construction exactly like the reference (src/run-nerf.py:35-36,65-80);
        # the fine network, which the reference does not have, continues the same RNG stream
        self.params = torch.zeros(n_nets * self.n_net, device=self.device)
        with torch.random.fork_rng(devices=[]):  # weights are initialised on the CPU
            torch.manual_seed(seed)
            for i in range(n_nets):
                net = NeRF(3, 3, n_layers, d_hidden, list(skip), **kw)
                self.params[i * self.n_net:(i + 1) * self.n_net].copy_(net.flat_parameters())
        # gradient buffer with the two loss accumulators behind it: ONE fill zeroes both every step.
        # The occgrid sampler puts this rank's trained survivor count between them, so the gradient
        # all-reduce also tells every rank whether any rank trained (one collective, one decision).
        n_grad = self.params.numel() + (1 if self.occgrid else 0)
        self._grads_and_loss = torch.zeros(n_grad + 2, device=self.device)
        self.grads = self._grads_and_loss[:self.params.numel()]
        self._reduced = self._grads_and_loss[:n_grad]
        self.m = torch.zeros_like(self.params)
        self.v = torch.zeros_like(self.params)
        self.packed = [torch.empty(ops.mlp_packed_bytes(self.cfg), dtype=torch.uint8, device=self.device)
                       for _ in range(n_nets)]
        self.bkgd = torch.ones(3, device=self.device) if self.white_bkgd else None
        self.step = 0
        self._seed, self._draws = int(seed), 0
        self.lr = lr
        self.pg = process_group
        if world_size is not None:
            self.world = int(world_size)
        else:
            self.world = torch.distributed.get_world_size(process_group) if process_group is not None or (
                torch.distributed.is_available() and torch.distributed.is_initialized()) else 1
        self.rank = torch.distributed.get_rank(process_group) if self.world > 1 and (
            torch.distributed.is_available() and torch.distributed.is_initialized()) else 0
        self.loss_sums = self._grads_and_loss[n_grad:]
        # in-step regularisers (SURVEY.md §8 f2): occlusion (src/core/loss.py:26-60) fused into the
        # compositing backward, weight-norm penalty (src/run-nerf.py:266-279) fused into Adam
        self.occ_sum = torch.zeros(1, device=self.device)
        self.reg_segs = ops.reg_segments(self.cfg, n_nets)
        self.reg_sums = torch.zeros(len(self.reg_segs), device=self.device)
        self.mask_pos = self.mask_dir = None
        self._buf = {}
        self._packed_fresh = False
        self.launches = 0  # kernels of ours launched (bench.py reports it)
        if self.occgrid:
            if roi_aabb is None:
                raise FsnerfError("HotPath(sampler='occgrid') needs roi_aabb")
            self.estimator = OccGridEstimator(roi_aabb, resolution=int(grid_resolution),
                                              levels=int(grid_levels)).to(self.device)
            self.render_step_size = float(render_step_size)
            self.early_stop_eps, self.alpha_thre = 1e-4, 0.0  # OccGridEstimator.sampling's defaults
            self.k = 0  # train_step calls so far: the reference's loop counter (src/run-nerf.py:288-295)
            self._grid_gen = torch.Generator(device=self.device)
            self.last_counts = (0, 0)  # (candidates N, survivors M) of the last occgrid forward

    # ------------------------------------------------------------------ helpers
    def net_params(self, i):
        return self.params[i * self.n_net:(i + 1) * self.n_net]

    def net_grads(self, i):
        return self.grads[i * self.n_net:(i + 1) * self.n_net]

    def state_dict(self, i):
        """reference-format state dict of network i (0 = coarse, 1 = fine / only)."""
        flat = self.net_params(i)
        shapes = NeRF_shapes(self.cfg)
        return {n: flat[o:o + k].view(shapes[n]).clone() for (o, k), n in zip(self.layout, self.names)}

    def load_state_dict(self, i, sd):
        self.net_params(i).copy_(ops.flatten_state_dict(self.cfg, sd, self.device))
        self._packed_fresh = False

    def set_freq_mask(self, step, reg_steps):
        """FreeNeRF annealed mask (App. B4) for this step; None when expired."""
        if reg_steps <= 0 or step >= reg_steps:
            self.mask_pos = self.mask_dir = None
        else:
            self.mask_pos = freq_mask(3 * (1 + 2 * self.cfg.n_freqs_pos), step, reg_steps).to(self.device)
            self.mask_dir = freq_mask(3 * (1 + 2 * self.cfg.n_freqs_dir), step, reg_steps).to(self.device)

    def _bytes(self, key, n):
        b = self._buf.get(key)
        if b is None or b.numel() < n:
            b = torch.empty(n, dtype=torch.uint8, device=self.device)
            self._buf[key] = b
        return b

    def _zeros4(self, key, n):
        """cached zero-initialised [n,4] buffer (rgb slots stay 0: only sigma is written)"""
        b = self._buf.get(key)
        if b is None or b.shape[0] != n:
            b = torch.zeros(n, 4, device=self.device)
            self._buf[key] = b
        return b

    def _pack(self):
        if not self._packed_fresh:
            for i, pk in enumerate(self.packed):
                ops.mlp_pack(self.cfg, self.net_params(i), pk)
                self.launches += 1
            self._packed_fresh = True

    # ------------------------------------------------------------------ forward
    def _jitter_seeds(self):
        """Two fresh 64-bit keys (stratified, pdf) for the in-kernel uniform stream."""
        self._draws += 1
        return jitter_seeds(self._seed, self.rank, self._draws)

    def _forward(self, rays_o, rays_d, u_strat, u_pdf, train, seeds=(None, None)):
        cfg, R = self.cfg, rays_o.shape[0]
        self._pack()
        ts_c, te_c = ops.sample_stratified(R, self.n_coarse, self.near, self.far, u_strat, device=self.device,
                                           seed=seeds[0] if u_strat is None else None)
        st_c = self._bytes("stash_c", ops.mlp_stash_bytes(cfg, R * self.n_coarse)) if train else None
        # rendering a hierarchical model needs only the WEIGHTS of the coarse pass: skip its view
        # branch (17 % of its FLOPs) and write sigma straight into the compositor's (rgb, sigma) layout
        sigma_only = (not train) and self.hier
        raw_c = ops.mlp_forward(cfg, self.net_params(0), self.packed[0], rays_o=rays_o, rays_d=rays_d,
                                t_starts=ts_c, t_ends=te_c, mask_pos=self.mask_pos, mask_dir=self.mask_dir,
                                stash=st_c, density_only=2 if sigma_only else 0,
                                out=self._zeros4("raw_c", R * self.n_coarse) if sigma_only else None)
        rgb_c, op_c, dp_c, w_c, _, _ = ops.composite_forward(raw_c.view(R, self.n_coarse, 4), ts_c, te_c,
                                                             bkgd=self.bkgd)
        self.launches += 3
        out = dict(ts_c=ts_c, te_c=te_c, raw_c=raw_c, rgb_c=rgb_c, op_c=op_c, dp_c=dp_c, w_c=w_c, st_c=st_c)
        if not self.hier:
            out.update(rgb=rgb_c, opacity=op_c, depth=dp_c)
            return out
        S = self.n_coarse + self.n_fine
        ts_f, te_f, *_ = ops.sample_pdf(ts_c, w_c, self.n_fine, self.far, u_pdf, want_aux=False,
                                        seed=seeds[1] if u_pdf is None else None)
        st_f = self._bytes("stash_f", ops.mlp_stash_bytes(cfg, R * S)) if train else None
        raw_f = ops.mlp_forward(cfg, self.net_params(1), self.packed[1], rays_o=rays_o, rays_d=rays_d,
                                t_starts=ts_f, t_ends=te_f, mask_pos=self.mask_pos, mask_dir=self.mask_dir,
                                stash=st_f)
        rgb_f, op_f, dp_f, w_f, _, _ = ops.composite_forward(raw_f.view(R, S, 4), ts_f, te_f, bkgd=self.bkgd)
        self.launches += 3
        out.update(ts_f=ts_f, te_f=te_f, raw_f=raw_f, rgb=rgb_f, opacity=op_f, depth=dp_f, w_f=w_f, st_f=st_f)
        return out

    def _forward_occgrid(self, rays_o, rays_d, u, train):
        """occgrid sampler: march -> density forward of the candidates -> visibility filter -> forward
        of the survivors (stashed when train) -> packed compositing.  u: per-ray jitter U[0,1) or None.
        Every step matches render.rendering.render_rays on OccGridEstimator bit for bit (same kernels,
        same operands), including its answer to exactly one survivor (src/render/rendering.py:97-103):
        a constant background, zero opacity and depth, and no raw samples to train."""
        cfg, R = self.cfg, rays_o.shape[0]
        self._pack()
        est, step = self.estimator, self.render_step_size
        near_planes = None if u is None else u * step  # the drop-in's 0 + u * step, bit for bit
        ri, ts, te, offsets = ops.occgrid_march(rays_o, rays_d, est.binaries.view(torch.uint8), est.aabbs, step,
                                                near=0.0, far=1e10, near_planes=near_planes)
        N = ts.numel()
        self.launches += 2
        if N > 0:
            x, _ = ops.packed_points(ri, ts, te, rays_o, rays_d)
            sigmas = ops.mlp_forward(cfg, self.net_params(0), self.packed[0], x=x, mask_pos=self.mask_pos,
                                     mask_dir=self.mask_dir, density_only=1)
            ri, ts, te, offsets = ops.occgrid_filter(ts, te, offsets, sigmas, self.early_stop_eps, self.alpha_thre)
            self.launches += 4
        M = ts.numel()
        self.last_counts = (N, M)
        out = dict(ri=ri, ts=ts, te=te, offsets=offsets, M=M, raw=None, st=None)
        if M == 1:
            bk = 1.0 if self.white_bkgd else 0.0
            out.update(rgb=torch.full((R, 3), bk, device=self.device), opacity=torch.zeros(R, 1, device=self.device),
                       depth=torch.zeros(R, 1, device=self.device))
            return out
        if M > 0:
            x, dirs = ops.packed_points(ri, ts, te, rays_o, rays_d, want_dirs=True)
            out["st"] = self._bytes("stash", ops.mlp_stash_bytes(cfg, M)) if train else None
            raw = ops.mlp_forward(cfg, self.net_params(0), self.packed[0], x=x, dirs=dirs, mask_pos=self.mask_pos,
                                  mask_dir=self.mask_dir, stash=out["st"])
            self.launches += 2
        else:
            raw = torch.zeros(0, 4, device=self.device)
        rgb, op, dp, _, tr, _ = ops.composite_packed_forward(raw, ts, te, offsets, bkgd=self.bkgd)
        self.launches += 1
        out.update(raw=raw, trans=tr, rgb=rgb, opacity=op, depth=dp)
        return out

    def _occ_eval(self, x):
        """occ_eval_fn of the reference's grid update: density of the current weights x step size"""
        self._pack()
        sigma = ops.mlp_forward(self.cfg, self.net_params(0), self.packed[0], x=x, mask_pos=self.mask_pos,
                                mask_dir=self.mask_dir, density_only=1)
        return sigma * self.render_step_size

    @torch.no_grad()
    def update_grid(self, step: int) -> None:
        """occgrid sampler: OccGridEstimator.update_every_n_steps(step) (src/run-nerf.py:288-295; updates
        when step % 16 == 0) with occ_eval_fn = density of the current weights x render_step_size.  The
        cells and points are drawn from grid_seed(seed, step), so equal weights give equal grids."""
        self._grid_gen.manual_seed(grid_seed(self._seed, step))
        self.estimator.update_every_n_steps(step=step, occ_eval_fn=self._occ_eval, occ_thre=1e-2,
                                            generator=self._grid_gen)

    @torch.no_grad()
    def render(self, rays_o, rays_d):
        """deterministic (eval) render of a ray chunk -> rgb[R,3], opacity[R,1], depth[R,1]"""
        if self.occgrid:
            o = self._forward_occgrid(rays_o, rays_d, None, train=False)
        else:
            o = self._forward(rays_o, rays_d, None, None, train=False)
        return o["rgb"], o["opacity"], o["depth"]

    # --------------------------------------------------------------- train step
    @torch.no_grad()
    def train_step(self, rays_o, rays_d, rgb_gt, u_strat=None, u_pdf=None, lr: Optional[float] = None,
                   global_rays: Optional[int] = None, apply_update: bool = True,
                   occ_reg=None, weight_reg=None):
        """One optimisation step on this rank's ray shard.  Returns a device
        tensor [2] = (sum sq err coarse, sum sq err fine) over the local shard;
        mean loss = value / (3 * global_rays).  u_*: explicit uniforms (parity tests); by default
        the samplers draw them in-kernel from the counter-based stream (ops.rng_uniform), so
        the step launches no generator kernel and writes no uniform buffer.

        occ_reg = (a, b, func): adds core.loss.OcclusionRegularizer(a, b, func) of the output
        pass (the fine network's samples; the coarse ones when n_fine == 0) to the loss exactly
        as src/run-nerf.py:260-264 does (NOT scaled by beta, which only gates it there);
        self.occ_sum / global_rays is its value.  weight_reg = (mode, alpha): the weight-norm
        penalty of src/run-nerf.py:266-279 ('l1' or Frobenius) on every network of the flat
        buffer; the caller applies the reference's `k < int(reg_ratio*Td)` gate by passing
        None.  self.reg_sums holds sum|w| (l1) / sum w^2 (l2) per regularised tensor."""
        if self.occgrid:
            return self._train_step_occgrid(rays_o, rays_d, rgb_gt, u_strat, lr, global_rays, apply_update,
                                            occ_reg, weight_reg)
        cfg, R = self.cfg, rays_o.shape[0]
        G = int(global_rays) if global_rays is not None else R * self.world
        o = self._forward(rays_o, rays_d, u_strat, u_pdf, train=True, seeds=self._jitter_seeds())
        self._grads_and_loss.zero_()
        scale = loss_grad_scale(G)  # F.mse_loss 'mean' over the GLOBAL batch (src/run-nerf.py:256)
        occ = None
        if occ_reg is not None:
            self.occ_sum.zero_()
            occ = (occ_reg[0], occ_reg[1], occ_reg[2], 1.0 / G, self.occ_sum)
        d_rgb_c = ops.mse_loss_grad(o["rgb_c"], rgb_gt, scale, self.loss_sums[0:1])
        d_raw_c, _ = ops.composite_backward(o["raw_c"].view(R, self.n_coarse, 4), o["ts_c"], o["te_c"], d_rgb_c,
                                            bkgd=self.bkgd, occ=None if self.hier else occ)
        # one ring for both passes (they run back to back on the stream): it stays L2 resident
        det = self.deterministic
        ws_c = self._bytes("bwd_ws", max(ops.mlp_bwd_workspace_bytes(cfg, R * self.n_coarse, det),
                                         ops.mlp_bwd_workspace_bytes(cfg, R * (self.n_coarse + self.n_fine), det)))
        ops.mlp_backward(cfg, self.net_params(0), self.packed[0], R * self.n_coarse, o["st_c"], o["raw_c"],
                         d_raw_c.view(-1, 4), self.net_grads(0), ws_c, deterministic=det)
        self.launches += 2 + 2  # mse, composite bwd, heads, fused dgrad+wgrad
        if self.hier:
            S = self.n_coarse + self.n_fine
            d_rgb_f = ops.mse_loss_grad(o["rgb"], rgb_gt, scale, self.loss_sums[1:2])
            d_raw_f, _ = ops.composite_backward(o["raw_f"].view(R, S, 4), o["ts_f"], o["te_f"], d_rgb_f,
                                                bkgd=self.bkgd, occ=occ)
            ws_f = ws_c
            ops.mlp_backward(cfg, self.net_params(1), self.packed[1], R * S, o["st_f"], o["raw_f"],
                             d_raw_f.view(-1, 4), self.net_grads(1), ws_f, deterministic=det)
            self.launches += 2 + 2  # mse, composite bwd, heads, fused dgrad+wgrad
        if self.world > 1:
            # the path's one real exchange: SUM of the flat fp32 gradient (both nets)
            allreduce_gradients(self.grads, self.pg)
        if apply_update:
            self.step += 1
            if weight_reg is not None:
                ops.adam_step_reg(self.params, self.grads, self.m, self.v, self.lr if lr is None else lr,
                                  self.step, weight_reg[0], weight_reg[1], self.reg_segs, self.reg_sums,
                                  deterministic=self.deterministic)
                self.launches += 2
            else:
                ops.adam_step(self.params, self.grads, self.m, self.v, self.lr if lr is None else lr, self.step)
                self.launches += 1
            self._packed_fresh = False
        return self.loss_sums

    def _train_step_occgrid(self, rays_o, rays_d, rgb_gt, u, lr, global_rays, apply_update, occ_reg, weight_reg):
        """train_step of the occgrid sampler: the step of examples/train_dropin.py --sampler occgrid
        (src/run-nerf.py:232-295) on the fused kernels.  u: explicit per-ray jitter [R] (else drawn
        in-kernel from the step's stratified key).  The loss goes to loss_sums[0].  The host reads
        two sizes, N and M (ops.occgrid_march / ops.occgrid_filter); a data-parallel rank that
        trained nothing also reads the all-reduced survivor count.

        Fewer than two survivors (the empty grid of the first steps, or the one-survivor
        background fallback) write no MLP gradient; when that holds on every rank, Adam does not
        step and its step count stays, as torch.optim.Adam skips parameters whose .grad is None.
        With apply_update the grid update of loop step k (the number of earlier train_step calls)
        follows on the fresh weights."""
        if occ_reg is not None:
            raise FsnerfError("HotPath(sampler='occgrid'): occ_reg is not fused into the packed backward")
        cfg, R = self.cfg, rays_o.shape[0]
        G = int(global_rays) if global_rays is not None else R * self.world
        k, self.k = self.k, self.k + 1
        seed = self._jitter_seeds()[0]
        if u is None:
            u = ops.rng_uniform(R, seed, device=self.device)
            self.launches += 1
        o = self._forward_occgrid(rays_o, rays_d, u, train=True)
        self._grads_and_loss.zero_()
        M = o["M"]
        trained = M >= 2
        d_rgb = ops.mse_loss_grad(o["rgb"], rgb_gt, loss_grad_scale(G), self.loss_sums[0:1], want_grad=trained)
        self.launches += 1
        if trained:
            d_raw, _ = ops.composite_packed_backward(o["raw"], o["ts"], o["te"], o["offsets"], o["trans"], d_rgb,
                                                     bkgd=self.bkgd)
            ws = self._bytes("bwd_ws", ops.mlp_bwd_workspace_bytes(cfg, M, self.deterministic))
            ops.mlp_backward(cfg, self.net_params(0), self.packed[0], M, o["st"], o["raw"], d_raw, self.net_grads(0),
                             ws, deterministic=self.deterministic)
            self._reduced[-1:].fill_(float(M))
            self.launches += 3
        any_trained = trained
        if self.world > 1:
            allreduce_gradients(self._reduced, self.pg)
            if not trained:
                any_trained = float(self._reduced[-1].item()) > 0
        if apply_update:
            if any_trained:
                self.step += 1
                if weight_reg is not None:
                    ops.adam_step_reg(self.params, self.grads, self.m, self.v, self.lr if lr is None else lr,
                                      self.step, weight_reg[0], weight_reg[1], self.reg_segs, self.reg_sums,
                                  deterministic=self.deterministic)
                    self.launches += 2
                else:
                    ops.adam_step(self.params, self.grads, self.m, self.v, self.lr if lr is None else lr, self.step)
                    self.launches += 1
                self._packed_fresh = False
            self.update_grid(k)
        return self.loss_sums

    @staticmethod
    def psnr(loss_sum: float, n_rays: int) -> float:
        """reference: psnr = -10 log10(mse) (src/run-nerf.py:257-258)"""
        return -10.0 * math.log10(max(loss_sum / (3.0 * n_rays), 1e-20))


def NeRF_shapes(cfg):
    H = cfg.d_hidden
    d_pe, d_de = 3 * (1 + 2 * cfg.n_freqs_pos), 3 * (1 + 2 * cfg.n_freqs_dir)
    shapes = {}
    for i in range(cfg.n_layers):
        n_in = d_pe if i == 0 else (H + d_pe if (cfg.skip_mask >> (i - 1)) & 1 else H)
        shapes[f"layers.{i}.weight"], shapes[f"layers.{i}.bias"] = (H, n_in), (H,)
    shapes["sigma.weight"], shapes["sigma.bias"] = (1, H), (1,)
    shapes["connection.weight"], shapes["connection.bias"] = (H, H), (H,)
    shapes["branch.weight"], shapes["branch.bias"] = (H // 2, H + d_de), (H // 2,)
    shapes["rgb.weight"], shapes["rgb.bias"] = (3, H // 2), (3,)
    return shapes
