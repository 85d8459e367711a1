"""The training forward's stash (csrc/mlp_fwd2.cu, kTrain): the bf16 SW128 operand images and
1-bit ReLU masks that the backward reads back.

  (a) a seeded run large enough that every CTA loops over several tiles (148 x 3 full tiles plus
      a partial one) reproduces recorded SHA-256 digests of the stash bytes and of `out` — the
      forward has no atomics, so both are deterministic bit for bit;
  (b) every mask bit equals `h > 0` of the bf16 activation image stored in the same record;
  (c) bytes past the last tile's record in an oversized stash buffer stay untouched.

`python tests/test_gpu_stash.py` prints the digests of the current build (to re-record them
after a deliberate change of the stash format or of the forward's arithmetic)."""
import hashlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import mlp as omlp  # noqa: E402

P_HASH = 128 * (148 * 3 + 5) + 37   # every CTA runs >= 3 tiles; the last tile is partial
SEED = 7
STASH_SHA256 = "f7efd271eb01b50a811d2cbfd023319b4008ef32ef292413cebf130a907a3afc"
OUT_SHA256 = "e9350c1048e96e30abb81a1ed802f7be6a875aca4fddf95c6a3ac6ed6f3f59f2"


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fsnerf_b200 import ops
    ops.require_device(0)
    return torch.device("cuda:0")


def _inputs(P, seed, device):
    from fsnerf_b200 import ops
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict(seed=seed)
    params = ops.flatten_state_dict(cfg, sd, device)
    packed = ops.mlp_pack(cfg, params)
    g = torch.Generator().manual_seed(1000 + seed)
    x = (torch.rand(P, 3, generator=g) * 2 - 1) * 2.5
    d = torch.nn.functional.normalize(torch.randn(P, 3, generator=g), dim=-1)
    return cfg, params, packed, x.to(device), d.to(device)


def _forward(P, seed, device, pad=0, fill=0):
    """-> (out, stash buffer of stash_bytes + pad bytes, filled with `fill` before the launch)"""
    from fsnerf_b200 import ops
    cfg, params, packed, x, d = _inputs(P, seed, device)
    nb = ops.mlp_stash_bytes(cfg, P)
    buf = torch.full((nb + pad,), fill, dtype=torch.uint8, device=device)
    out = ops.mlp_forward(cfg, params, packed, x=x, dirs=d, stash=buf[:nb])
    torch.cuda.synchronize()
    return cfg, out, buf


def _digests(out, stash):
    return (hashlib.sha256(stash.cpu().numpy().tobytes()).hexdigest(),
            hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest())


def _layout(cfg):
    """Per tile record (csrc/mlp_program.cu): [(image offset, chunks, mask offset)] of every layer
    whose output has a ReLU mask, and the record size."""
    H, n = cfg.d_hidden, cfg.n_layers
    CH = 128 * 128  # one [128 rows x 64 features] bf16 chunk image
    off = CH                                  # the position encoding image comes first
    layers = []                               # (image offset, chunks, has mask)
    for _ in range(n):
        layers.append((off, H // 64, True))
        off += (H // 64) * CH
    off += (H // 64) * CH                     # connection layer (no ReLU)
    off += CH                                 # view-direction encoding image
    layers.append((off, (H // 2) // 64, True))  # branch
    off += ((H // 2) // 64) * CH
    out = []
    for img, nch, _ in layers:
        out.append((img, nch, off))
        off += nch * 2 * 128 * 4
    return out, off


def _check_masks(cfg, stash, n_tiles):
    layers, rec = _layout(cfg)
    s = stash[: n_tiles * rec].view(n_tiles, rec).cpu().numpy()
    rows = np.arange(128)
    for img, nch, moff in layers:
        for c in range(nch):
            chunk = s[:, img + c * 128 * 128: img + (c + 1) * 128 * 128].reshape(n_tiles, 128, 8, 16)
            # undo the SW128 swizzle: 16-byte unit u of row r sits at unit u ^ (r & 7)
            units = chunk[:, rows[:, None], (np.arange(8)[None, :] ^ (rows[:, None] & 7))]
            h = units.reshape(n_tiles, 128, 64 * 2).view(np.uint16)            # [tile, row, feature] bf16 bits
            pos = (h != 0) & (h < 0x8000)                                       # bf16 > 0
            for half in range(2):
                words = s[:, moff + (c * 2 + half) * 512: moff + (c * 2 + half + 1) * 512].view(np.uint32)
                f = pos[:, :, 32 * half: 32 * half + 32]
                # feature 2q -> bit 15 - q, feature 2q + 1 -> bit 31 - q (mlp_issue.cuh: relu_bits_fold)
                want = np.zeros((n_tiles, 128), np.uint32)
                for q in range(16):
                    want |= f[:, :, 2 * q].astype(np.uint32) << np.uint32(15 - q)
                    want |= f[:, :, 2 * q + 1].astype(np.uint32) << np.uint32(31 - q)
                bad = np.argwhere(words != want)
                assert bad.size == 0, (img, c, half, bad[:4])
            assert pos.any() and not pos.all(), "the seeded activations should have both signs"


@pytest.mark.gpu
def test_stash_and_out_match_recorded_digests(dev):
    _, out, stash = _forward(P_HASH, SEED, dev)
    assert _digests(out, stash) == (STASH_SHA256, OUT_SHA256)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [P_HASH, 128 * 5 + 1])
def test_relu_masks_match_the_stashed_activations(dev, P):
    from fsnerf_b200 import ops
    cfg, _, stash = _forward(P, SEED, dev, fill=0xA5)
    n_tiles = (P + 127) // 128
    assert _layout(cfg)[1] * n_tiles == ops.mlp_stash_bytes(cfg, P)
    _check_masks(cfg, stash, n_tiles)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [P_HASH, 300])
def test_nothing_written_past_the_last_tile(dev, P):
    from fsnerf_b200 import ops
    pad = 1 << 20
    cfg, _, buf = _forward(P, SEED, dev, pad=pad, fill=0x3C)
    nb = ops.mlp_stash_bytes(cfg, P)
    assert bool((buf[nb:] == 0x3C).all())
    assert bool((buf[:nb] != 0x3C).any())


if __name__ == "__main__":
    _, out, stash = _forward(P_HASH, SEED, torch.device("cuda:0"))
    s, o = _digests(out, stash)
    print(f'STASH_SHA256 = "{s}"\nOUT_SHA256 = "{o}"')
