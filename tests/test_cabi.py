"""CPU tests: the C-ABI library loads and exports every symbol that
include/fsnerf_b200.h declares (no compute calls without a GPU)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "fsnerf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fsnerf_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from fsnerf_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in the header but not exported"
        assert s in _lib.SIGNATURES, f"{s} has no ctypes prototype"
    assert set(_lib.SIGNATURES) == set(syms)
    assert lib.fsnerf_version() >= 100
    assert isinstance(lib.fsnerf_last_error(), bytes)


def test_host_side_layout_queries():
    """param count / packed bytes are pure host arithmetic: safe without a GPU."""
    from fsnerf_b200 import ops
    cfg = ops.make_cfg()
    layout = ops.mlp_param_layout(cfg)
    assert len(layout) == 24 and sum(n for _, n in layout) == 595844  # reference state dict (SURVEY.md §8 a5)
    assert all(o % 4 == 0 for o, _ in layout) and ops.mlp_param_count(cfg) % 4 == 0
    assert ops.mlp_param_count(cfg) >= 595844
    # 73 forward + 68 transposed (dgrad) 16 KB operand blocks + the fp32 small-params block
    assert ops.mlp_packed_bytes(cfg) == (73 + 68) * 16384 + 4864 * 4
    # per 128-sample tile: 640 KB of bf16 operand images + 34 KB of 1-bit ReLU masks (8 x 4 KB + 2 KB)
    assert ops.mlp_stash_bytes(cfg, 128) == 640 * 1024 + 34 * 1024
    assert ops.mlp_stash_bytes(cfg, 129) == 2 * (640 + 34) * 1024
    bad = ops.make_cfg(d_hidden=128)
    from fsnerf_b200._lib import FsnerfError
    with pytest.raises(FsnerfError, match="d_hidden must be 256"):
        ops.mlp_param_count(bad)


def test_no_cpu_fallback():
    import torch
    from fsnerf_b200 import ops
    from fsnerf_b200._lib import FsnerfError
    with pytest.raises(FsnerfError, match="CUDA tensor"):
        ops.composite_forward(torch.zeros(2, 4, 4), torch.zeros(2, 4), torch.ones(2, 4))


def test_flatten_state_dict_layout():
    import torch
    from fsnerf_b200 import ops
    from oracle import mlp as omlp
    cfg = ops.make_cfg()
    sd = omlp.init_state_dict()
    assert list(sd.keys()) == ops.state_dict_names(cfg)
    flat = ops.flatten_state_dict(cfg, sd, "cpu")
    for (o, n), name in zip(ops.mlp_param_layout(cfg), ops.state_dict_names(cfg)):
        assert torch.equal(flat[o:o + n], sd[name].reshape(-1))


def test_deep_network_is_rejected_before_the_pack_table_overflows():
    """12 hidden layers (205 operand blocks > the 192-entry pack table): an error, not a host overflow"""
    from fsnerf_b200 import ops
    from fsnerf_b200._lib import FsnerfError
    cfg = ops.make_cfg(n_layers=12)
    with pytest.raises(FsnerfError):
        ops.mlp_param_count(cfg)
