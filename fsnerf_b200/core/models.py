"""Drop-in for the reference's ``core.models`` (NeRF + PositionalEncoder,
/root/reference/src/core/models.py:10-143): same constructor signatures, same
``state_dict()`` keys/shapes (24 tensors, 595 844 parameters for the default
net), same seed-42 initial values, same ``forward(x, dirs=None)`` contract —
but the arithmetic runs in the fused tcgen05 kernels of libfsnerf_b200.so
(bf16 operands, fp32 accumulation).  There is no CPU path.
"""
from typing import Tuple

import torch
from torch import nn, Tensor

from .. import ops
from .._lib import FsnerfError


class PositionalEncoder(nn.Module):
    """reference: src/core/models.py:10-50.  Holds the encoding configuration;
    inside NeRF the encoding is computed in registers by the MLP kernel and never
    materialised.  ``d_output = d_input * (1 + 2 * n_freqs)``."""

    def __init__(self, d_input, n_freqs, log_space=False):
        super().__init__()
        self.d_input = d_input
        self.n_freqs = n_freqs
        self.log_space = log_space
        self.d_output = d_input * (1 + 2 * n_freqs)

    def frequencies(self) -> Tensor:
        """reference :31-34: 2^linspace(0, L-1, L) (log space) or linspace(1, 2^(L-1), L)"""
        if self.log_space:
            return 2.0 ** torch.linspace(0.0, self.n_freqs - 1, self.n_freqs)
        return torch.linspace(2.0 ** 0.0, 2.0 ** (self.n_freqs - 1), self.n_freqs)

    def forward(self, x, mask=None):
        """[..., d_input] -> [..., d_output] on the device (standalone kernel ``fsnerf_encode``; inside
        NeRF the same encoding is fused into the first layer's operand staging and never materialised).
        Inference only, like every direct use in the reference."""
        if not x.is_cuda:
            raise FsnerfError("PositionalEncoder.forward: CUDA tensor required (no CPU path)")
        out = ops.encode(x.reshape(-1, self.d_input), self.frequencies().to(x.device), mask)
        return out.reshape(*x.shape[:-1], self.d_output)


class _NeRFFunction(torch.autograd.Function):
    """model(x, dirs): one fused forward launch; backward = dgrad + wgrad + heads.
    The parameter tensors are passed so autograd routes gradients to them; the
    kernels read the shared flat buffer they are views of."""

    @staticmethod
    def forward(ctx, module, x, dirs, need_grad, *params):
        ctx.set_materialize_grads(False)
        density_only = dirs is None
        if need_grad and density_only:
            raise FsnerfError("NeRF(x) (density only) is inference-only on the B200 path; the "
                              "reference calls it under no_grad (src/render/rendering.py:58-64)")
        P = x.shape[0]
        packed = module._refresh_packed()
        stash = None
        if need_grad:
            stash = torch.empty(ops.mlp_stash_bytes(module.cfg, P), dtype=torch.uint8, device=x.device)
        out = ops.mlp_forward(module.cfg, module._flat, packed, x=x, dirs=dirs,
                              mask_pos=module.mask_pos, mask_dir=module.mask_dir,
                              density_only=density_only, stash=stash)
        ctx.module, ctx.P, ctx.stash, ctx.packed = module, P, stash, packed
        ctx.save_for_backward(out)
        return out.reshape(P, 1) if density_only else out

    @staticmethod
    def backward(ctx, d_out):
        module = ctx.module
        (out,) = ctx.saved_tensors
        if d_out is None:
            return (None,) * (4 + len(module._layout))
        grads = torch.zeros_like(module._flat)
        # torch.use_deterministic_algorithms(True) selects the bitwise reproducible backward
        det = torch.are_deterministic_algorithms_enabled()
        ws = torch.empty(ops.mlp_bwd_workspace_bytes(module.cfg, ctx.P, det), dtype=torch.uint8,
                         device=out.device)
        ops.mlp_backward(module.cfg, module._flat, ctx.packed, ctx.P, ctx.stash, out,
                         d_out.contiguous(), grads, ws, deterministic=det)
        module._last_flat_grad = grads
        views = [grads[o:o + n].view(p.shape) for (o, n), p in zip(module._layout, module._param_list())]
        return (None, None, None, None, *views)


class NeRF(nn.Module):
    """reference: src/core/models.py:53-143 (8x256 ReLU MLP, skip concat after
    layer 4, un-activated sigma head, 256->256 connection, 283->128 view branch,
    128->3 sigmoid rgb).  forward(x[N,3], dirs[N,3]|None) -> [N,4]=(rgb,sigma)
    or [N,1]=sigma."""

    def __init__(self, d_pos: int = 3, d_dir: int = 3, n_layers: int = 8, d_hidden: int = 256,
                 skip: Tuple[int] = (4,), **kwargs) -> None:
        super().__init__()
        if d_pos != 3 or d_dir != 3:
            raise FsnerfError("NeRF: the B200 path supports d_pos == d_dir == 3")
        self.d_pos, self.d_dir, self.skip = d_pos, d_dir, skip
        skip = [int(s) for s in skip]  # parser quirk: --skip yields ['4'] (SURVEY.md App. C7)
        n_freqs, log_space = kwargs["pos_fn"]["n_freqs"], kwargs["pos_fn"]["log_space"]
        self._pos_encoder = PositionalEncoder(d_pos, n_freqs, log_space)
        n_freqs_d, log_space_d = kwargs["dir_fn"]["n_freqs"], kwargs["dir_fn"]["log_space"]
        self._dir_encoder = PositionalEncoder(d_dir, n_freqs_d, log_space_d)
        if bool(log_space) != bool(log_space_d):
            raise FsnerfError("NeRF: pos_fn and dir_fn must share log_space")
        d_pe, d_de = self._pos_encoder.d_output, self._dir_encoder.d_output
        self.cfg = ops.make_cfg(n_layers, d_hidden, skip, n_freqs, n_freqs_d, log_space)
        # same construction order as the reference so torch.manual_seed(42) gives
        # the same initial weights (hidden 1..n-1 first, then layers.0; :96-102)
        hidden = [nn.Linear(d_hidden + d_pe, d_hidden) if i in skip else nn.Linear(d_hidden, d_hidden)
                  for i in range(n_layers - 1)]
        self.layers = nn.ModuleList([nn.Linear(d_pe, d_hidden)] + hidden)
        self.sigma = nn.Linear(d_hidden, 1)
        self.connection = nn.Linear(d_hidden, d_hidden)
        self.branch = nn.Linear(d_hidden + d_de, d_hidden // 2)
        self.rgb = nn.Linear(d_hidden // 2, 3)
        self.mask_pos = None  # FreeNeRF masks (set_freq_mask)
        self.mask_dir = None
        self._layout = ops.mlp_param_layout(self.cfg)
        self._flat = None
        self._packed = None
        self._rehome(torch.device("cpu"))

    # ---- flat parameter buffer ------------------------------------------------
    def _param_list(self):
        """parameters in state-dict order (cached: the kernels' layout is fixed at construction)"""
        pl = self.__dict__.get("_plist")
        if pl is None:
            pl = [p for _, p in self.named_parameters()]
            self.__dict__["_plist"] = pl
        return pl

    def _rehome(self, device, dtype=torch.float32):
        """(Re)create the flat fp32 buffer on `device` and make every parameter a
        view into it (state_dict keys/shapes unchanged)."""
        self.__dict__.pop("_plist", None)
        plist = self._param_list()
        if [tuple(p.shape) for p in plist] and len(plist) != len(self._layout):
            raise FsnerfError("NeRF: parameter list does not match the kernel layout")
        flat = torch.zeros(ops.mlp_param_count(self.cfg), device=device, dtype=dtype)
        for (o, n), p in zip(self._layout, plist):
            flat[o:o + n].copy_(p.detach().reshape(-1))
            p.data = flat[o:o + n].view(p.shape)
            p.grad = None
        self._flat = flat
        self._packed = None

    def _apply(self, fn, recurse=True):
        probe = fn(torch.empty(0, dtype=self._flat.dtype, device=self._flat.device))
        if probe.dtype != torch.float32:
            raise FsnerfError("NeRF: parameters stay fp32 (bf16 operand copies are made by the kernels)")
        if probe.device != self._flat.device:
            self._rehome(probe.device)
            if self.mask_pos is not None:
                self.mask_pos, self.mask_dir = self.mask_pos.to(probe.device), self.mask_dir.to(probe.device)
        return self

    def flat_parameters(self) -> Tensor:
        """the flat fp32 buffer all parameters are views of (kernel layout)"""
        return self._flat

    def _refresh_packed(self):
        """fp32 -> packed bf16 operand image (cheap: one small launch)."""
        if self._flat.device.type != "cuda":
            raise FsnerfError("NeRF: move the model to a CUDA device first (no CPU path)")
        # copy.deepcopy(model) / load_state_dict(assign=True) give the parameters their own storage:
        # the kernels would then read a stale flat buffer.  Re-home (copies the parameters' current
        # values into a fresh flat buffer and re-views them) when the aliasing is broken.
        base = self._flat.data_ptr()
        for (o, _), p in zip(self._layout, self._param_list()):
            if p.data_ptr() != base + 4 * o:
                self._rehome(p.device)
                break
        self._packed = ops.mlp_pack(self.cfg, self._flat, self._packed)
        return self._packed

    def set_freq_mask(self, step: int, reg_steps: int) -> None:
        """FreeNeRF annealed frequency mask (SURVEY.md App. B4) for both encodings;
        step >= reg_steps (or reg_steps <= 0) removes it."""
        if reg_steps <= 0 or step >= reg_steps:
            self.mask_pos = self.mask_dir = None
            return
        self.mask_pos = freq_mask(self._pos_encoder.d_output, step, reg_steps).to(self._flat.device)
        self.mask_dir = freq_mask(self._dir_encoder.d_output, step, reg_steps).to(self._flat.device)

    def forward(self, x, dirs=None):
        x = x.reshape(-1, 3)
        if dirs is not None:
            dirs = dirs.reshape(-1, 3)
        params = self._param_list()
        # (grad mode is always off inside Function.forward, so decide here)
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        return _NeRFFunction.apply(self, x, dirs, need_grad, *params)


def freq_mask(d_out: int, step: int, reg_steps: int) -> Tensor:
    """FreeNeRF mask over `d_out` channels laid out in groups of 3 (App. B4):
    ptr = min(G*step/reg_steps + 1, G); first floor(ptr) groups 1, next group
    ptr - floor(ptr), rest 0.  Host-side schedule (a 63-float vector)."""
    G = d_out // 3
    m = torch.zeros(d_out)
    if reg_steps <= 0 or step >= reg_steps:
        return torch.ones(d_out)
    ptr = min(G * float(step) / float(reg_steps) + 1.0, float(G))
    k = int(ptr)
    m[:3 * k] = 1.0
    if k < G:
        m[3 * k:3 * k + 3] = ptr - k
    return m


# ------------------------------------------------------------------ SiNeRF (module mirror)
class Sine(nn.Module):
    """reference: src/core/models.py:145-169 — sin(w x)"""

    def __init__(self, w: float = 1.) -> None:
        super().__init__()
        self.w = w

    def forward(self, x: Tensor) -> Tensor:
        return torch.sin(self.w * x)


class SirenLinear(nn.Module):
    """reference: src/core/models.py:171-236 — Linear + Sine with the SIREN initialisation
    (uniform(-1/d, 1/d) for the first layer, uniform(-sqrt(6/d), sqrt(6/d)) otherwise; weights
    drawn before biases, like the reference, so a seeded construction reproduces it)."""

    def __init__(self, in_dim: int = 256, out_dim: int = 256, use_bias: bool = True, w: float = 1.,
                 is_first: bool = False) -> None:
        super().__init__()
        self.fc_layer = nn.Linear(in_dim, out_dim, bias=use_bias)
        self.use_bias, self.is_first, self.in_dim, self.w, self.c = use_bias, is_first, in_dim, w, 6.
        self.activation = Sine(w)
        with torch.no_grad():
            bound = (1 / in_dim) if is_first else (6. / in_dim) ** 0.5
            self.fc_layer.weight.uniform_(-bound, bound)
            if use_bias and self.fc_layer.bias is not None:
                self.fc_layer.bias.uniform_(-bound, bound)

    def forward(self, x) -> Tensor:
        return self.activation(self.fc_layer(x))


class SiNeRF(nn.Module):
    """Drop-in for the reference's ``SiNeRF`` (src/core/models.py:238-309; selected by
    ``--model sinerf``, src/run-nerf.py:81-88): same constructor, state-dict keys and
    ``forward(x, dirs=None) -> [N,4] = (rgb, relu(sigma))`` or ``[N,1]``.

    NOT on the fused tcgen05 kernels: the sine activations need their own epilogue and a
    cos-based backward (DESIGN.md §8), so this mirror runs on PyTorch's CUDA ops.  It composes with
    the packed path (``OccGridEstimator`` + ``render_rays``), which calls ``model(x)`` /
    ``model(x, dirs)`` generically; the hierarchical / fused paths require ``NeRF``."""

    def __init__(self, pos_dim: int = 3, dir_dim: int = 3, width: int = 256,
                 alpha=(30., 1., 1., 1., 1., 1., 1., 1.)) -> None:
        super().__init__()
        self.pos_dim, self.dir_dim, self.alpha = pos_dim, dir_dim, list(alpha)
        hidden = [SirenLinear(width, width, True, a) for a in self.alpha[1:]]
        self.first_layers = nn.Sequential(SirenLinear(pos_dim, width, True, self.alpha[0], True), *hidden)
        self.sigma_layers = nn.Sequential(SirenLinear(width, width // 2, True), nn.Linear(width // 2, 1, True),
                                          nn.ReLU())
        self.fc_feature = nn.Linear(width, width)
        self.rgb_layers = nn.Sequential(SirenLinear(width + dir_dim, width // 2, True),
                                        nn.Linear(width // 2, 3, True), nn.Sigmoid())

    def forward(self, x: Tensor, dirs: Tensor = None) -> Tensor:
        x = self.first_layers(x)
        if dirs is None:
            return self.sigma_layers(x)
        sigma = self.sigma_layers(x)
        x = torch.cat([self.fc_feature(x), dirs], dim=-1)
        return torch.cat([self.rgb_layers(x), sigma], dim=-1)
