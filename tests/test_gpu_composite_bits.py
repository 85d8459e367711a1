"""Alpha compositing (csrc/composite.cu) bit for bit: seeded inputs reproduce recorded SHA-256
digests of every output of

  (a) the dense forward (extras on) for the flag sets 0, 1, 2, 4 and 7, with delta_scale and a
      background colour, at sample counts that select each register-block count (NB 2 / 4 / 6 / 8)
      and are not multiples of 32;
  (b) the dense backward's d_raw for the same flags, without and with the fused occlusion term,
      with d_opacity / d_depth / d_weights, including S = 300 (NB 16);
  (c) the packed forward and backward on ragged rays, some empty and one over 1000 samples;
  (d) the visibility filter's count and fill passes.

None of these outputs goes through an atomic, so each is deterministic.  d_bkgd and the occlusion
loss sum are float atomics and are left out.  A product-form digest that moves means an FMA
contraction moved in the compositing arithmetic.

`python tests/test_gpu_composite_bits.py` prints the digests of the current build (to re-record
them after a deliberate change of the compositing arithmetic)."""
import hashlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLAGS = [0, 1, 2, 4, 7]
SIZES = [(203, 45), (131, 100), (97, 170), (66, 250), (41, 300)]  # NB 2, 4, 6, 8, 8 fwd / 16 bwd
OCC = {None: None, "linear": (0.5, 2.0), "exp": (1.5, 0.7)}

DIGESTS = {
    "fwd-0": "456ccc44e4dfb3783f66fbae3a1324c01edc270e7f12d51c897c721218b877a2",
    "bwd-0-None": "ec2ff83ca3b6acea2be4f58465c5bb4b428c0952b546e38017c658d8a76abfd2",
    "bwd-0-linear": "ded3301159971ee17846aa884d8ae2f84b7263da2c8a38c758341c015423779a",
    "bwd-0-exp": "c39e97537cbb324fce68a45b1f48d3080023ff37a5c33c3bce122be1e05c5edc",
    "fwd-1": "dc5731120e05a0866f5b9256fc7518018e11a420caf52e5a680a3d61a0470172",
    "bwd-1-None": "71838e42f526d21be124243580870b6e41637d56be39e6183c91a8bf3e8f7bda",
    "bwd-1-linear": "6c6252cc8c6ee711f3e816a1ecd06587ef9819bd31968ac052e920b68b458022",
    "bwd-1-exp": "5f93f38afac80f411845137393fc197bd3bde0608b49d98d9f1f642905ee1a37",
    "fwd-2": "780448c1f6bd83fa4574245143c546aa2b46d5a09fdf8a50b4bfc49dea149192",
    "bwd-2-None": "13cf4b9d295783e767c5bc736f3371f13d530b764cb038859eb1e65e058b803e",
    "bwd-2-linear": "984dbb8a7ba9ebee2b02b7b13d5e83e1ef1533972fad092e2719fe6d8b986f68",
    "bwd-2-exp": "4b0e655d8869f590c13b453281738c604023a6fe26165544d5b18a33cdcf72e0",
    "fwd-4": "c6fbd4c7d97af0bce498ac244d4216a9be85da5295e52d2b6ee2c6a16ea8185b",
    "bwd-4-None": "9b99cf09412e5fc4a13791f66fadc3088960d44fc52d01c30737885d6516442e",
    "bwd-4-linear": "90a9b0fe56cf2f30779091fe3582433d0a5a20262c4d9959e1c999a9a895575a",
    "bwd-4-exp": "822e9f3ee37546f0a14e12d53065417331392230cf931a45c457971057cf0ac1",
    "fwd-7": "a3df1963cf679287b858164f426d88d4e4dc0d9bc2a36eb45ab8b2d45361132f",
    "bwd-7-None": "e0c22c5e48cdb1c70c7ae58574ff38262ffc0837257cebba3704da483daf3b64",
    "bwd-7-linear": "ec8eb8f3f96ae2b4574f0a66b17f66baf75422714676d3861c9bd98acfe8ad41",
    "bwd-7-exp": "8b7adcfc710a4cce6cc737698d2ded79e8f47a91cf55190f376274745429c37c",
    "packed-fwd": "45c93dec6ec9cc1ee8d87bd30205e707d77f19a403ad2a3f4f751f6200ab6b48",
    "packed-bwd": "b01e1649999fafc94a5f2b73e105afd4f64c8c4c380427a6fce4f51a4feaa526",
    "filter-0.0": "f976779d4f154e03e810cf826755688a8e7be68b82e487b90b8966add6558fa6",
    "filter-0.01": "5059861863023066cd0163cf2ec6369e0f0cb1d974d7d481954c3d75056357a2",
}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fsnerf_b200 import ops
    ops.require_device(0)
    return torch.device("cuda:0")


def _sha(tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def _dense_inputs(R, S, flags, seed, device):
    rng = np.random.default_rng(seed)
    e = np.sort(2 + 4 * rng.random((R, S + 1), dtype=np.float32), axis=-1)
    raw = rng.random((R, S, 4), dtype=np.float32)
    raw[..., 3] = rng.standard_normal((R, S), dtype=np.float32) * 6
    if flags & 4:
        raw[..., 3] = np.abs(raw[..., 3])  # product form: keep 1 - alpha positive
    ds = 1 + rng.random(R, dtype=np.float32)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)  # noqa: E731
    return cu(raw), cu(e[:, :-1]), cu(e[:, 1:]), cu(ds), rng


def _dense_forward(flags, device):
    from fsnerf_b200 import ops
    out = []
    for R, S in SIZES:
        raw, ts, te, ds, _ = _dense_inputs(R, S, flags, 100 * R + S, device)
        bk = torch.tensor([1.0, 0.5, 0.25], device=device)
        out += ops.composite_forward(raw, ts, te, bkgd=bk, delta_scale=ds, flags=flags, extras=True)
    return _sha(out)


def _dense_backward(flags, occ, device):
    from fsnerf_b200 import ops
    out = []
    for R, S in SIZES:
        raw, ts, te, ds, rng = _dense_inputs(R, S, flags, 100 * R + S + 1, device)
        cu = lambda a: torch.from_numpy(a).to(device)  # noqa: E731
        d_rgb = cu(rng.standard_normal((R, 3), dtype=np.float32))
        d_op = cu(rng.standard_normal((R, 1), dtype=np.float32))
        d_dp = cu(rng.standard_normal((R, 1), dtype=np.float32))
        d_w = cu(rng.standard_normal((R, S), dtype=np.float32))
        bk = torch.tensor([1.0, 0.5, 0.25], device=device)
        o = None if occ is None else (*OCC[occ], occ, 1.0 / (4 * R), torch.zeros(1, device=device))
        d_raw, _ = ops.composite_backward(raw, ts, te, d_rgb, d_op, d_dp, d_w, bkgd=bk, delta_scale=ds,
                                          flags=flags, want_d_bkgd=True, occ=o)
        out.append(d_raw)
    return _sha(out)


def _packed_inputs(device):
    rng = np.random.default_rng(11)
    counts = rng.integers(0, 90, 300)
    counts[rng.choice(300, 40, replace=False)] = 0
    counts[123] = 1037
    offsets = np.zeros(301, np.int64)
    offsets[1:] = np.cumsum(counts)
    N = int(offsets[-1])
    t = 2 + 4 * rng.random(N + 300, dtype=np.float32)
    ts, te = np.empty(N, np.float32), np.empty(N, np.float32)
    for r in range(300):
        e = np.sort(t[offsets[r] + r: offsets[r + 1] + r + 1])
        ts[offsets[r]: offsets[r + 1]], te[offsets[r]: offsets[r + 1]] = e[:-1], e[1:]
    raw = rng.random((N, 4), dtype=np.float32)
    raw[:, 3] = rng.standard_normal(N, dtype=np.float32) * 6
    cu = lambda a: torch.from_numpy(a).to(device)  # noqa: E731
    return cu(raw), cu(ts), cu(te), cu(offsets), rng


def _packed(device):
    from fsnerf_b200 import ops
    raw, ts, te, offsets, rng = _packed_inputs(device)
    R, N = offsets.numel() - 1, ts.numel()
    bk = torch.tensor([1.0, 0.5, 0.25], device=device)
    fwd = ops.composite_packed_forward(raw, ts, te, offsets, bkgd=bk)
    trans = fwd[4]
    cu = lambda a: torch.from_numpy(a).to(device)  # noqa: E731
    d_raw, _ = ops.composite_packed_backward(
        raw, ts, te, offsets, trans, cu(rng.standard_normal((R, 3), dtype=np.float32)),
        cu(rng.standard_normal((R, 1), dtype=np.float32)), cu(rng.standard_normal((R, 1), dtype=np.float32)),
        cu(rng.standard_normal(N, dtype=np.float32)), bkgd=bk, want_d_bkgd=True)
    return _sha(fwd), _sha([d_raw])


def _filter(alpha_thre, device):
    from fsnerf_b200 import ops
    raw, ts, te, offsets, _ = _packed_inputs(device)
    return _sha(ops.occgrid_filter(ts, te, offsets, raw[:, 3].contiguous(), 1e-4, alpha_thre))


def _all(device):
    d = {}
    for f in FLAGS:
        d[f"fwd-{f}"] = _dense_forward(f, device)
        for occ in OCC:
            d[f"bwd-{f}-{occ}"] = _dense_backward(f, occ, device)
    d["packed-fwd"], d["packed-bwd"] = _packed(device)
    for a in (0.0, 0.01):
        d[f"filter-{a}"] = _filter(a, device)
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAGS)
def test_dense_forward_matches_recorded_digests(dev, flags):
    assert _dense_forward(flags, dev) == DIGESTS[f"fwd-{flags}"]


@pytest.mark.gpu
@pytest.mark.parametrize("occ", list(OCC))
@pytest.mark.parametrize("flags", FLAGS)
def test_dense_backward_matches_recorded_digests(dev, flags, occ):
    assert _dense_backward(flags, occ, dev) == DIGESTS[f"bwd-{flags}-{occ}"]


@pytest.mark.gpu
def test_packed_forward_backward_match_recorded_digests(dev):
    assert _packed(dev) == (DIGESTS["packed-fwd"], DIGESTS["packed-bwd"])


@pytest.mark.gpu
@pytest.mark.parametrize("alpha_thre", [0.0, 0.01])
def test_filter_matches_recorded_digests(dev, alpha_thre):
    assert _filter(alpha_thre, dev) == DIGESTS[f"filter-{alpha_thre}"]


if __name__ == "__main__":
    print("DIGESTS = {")
    for k, v in _all(torch.device("cuda:0")).items():
        print(f'    "{k}": "{v}",')
    print("}")
