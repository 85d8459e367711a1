"""CPU tests of the deterministic mode's host side: the entry points are exported, and the workspace
queries are pure host arithmetic (no GPU needed)."""
import pytest

# fsnerf_mlp_bwd_workspace_bytes(cfg, n) for n in N_SAMPLES, as the library returned it before the
# deterministic mode existed: the default query must not change
N_SAMPLES = (0, 1, 300, 54321, 4096 * 64, 4096 * 192, 10 ** 7)
DEFAULT_BYTES = {
    (8, (4,), 10, 4): [32768, 361472, 1016832, 29534208, 29560832, 29626368, 30778368],
    (4, (2,), 6, 2): [32768, 230400, 623616, 17737728, 17764352, 17829888, 18981888],
    (10, (4, 7), 10, 4): [32768, 427008, 1213440, 35432448, 35459072, 35524608, 36676608],
}


def _lib():
    from fsnerf_b200 import _lib
    return _lib.load()


def test_deterministic_symbols_are_exported():
    from fsnerf_b200 import _lib
    lib = _lib.load()
    for s in ("fsnerf_mlp_bwd_workspace_bytes_deterministic", "fsnerf_mlp_backward_deterministic",
              "fsnerf_adam_step_reg_deterministic"):
        assert hasattr(lib, s) and s in _lib.SIGNATURES


@pytest.mark.parametrize("net", sorted(DEFAULT_BYTES))
def test_workspace_sizes(net):
    from fsnerf_b200 import ops
    n_layers, skip, fp, fd = net
    cfg = ops.make_cfg(n_layers, 256, skip, fp, fd)
    default = [ops.mlp_bwd_workspace_bytes(cfg, n) for n in N_SAMPLES]
    assert default == DEFAULT_BYTES[net]
    det = [ops.mlp_bwd_workspace_bytes(cfg, n, deterministic=True) for n in N_SAMPLES]
    assert det[0] == default[0]
    for n, a, b in zip(N_SAMPLES[1:], default[1:], det[1:]):
        assert b > a and b % 1024 == 0, n
    # the partials stop growing once every CTA of the launch is busy: 16.9 MB for the default net
    if net == (8, (4,), 10, 4):
        assert 15e6 < det[-1] - default[-1] < 18e6


def test_deterministic_entry_points_check_their_arguments():
    import ctypes as C
    from fsnerf_b200 import ops
    lib = _lib()
    cfg = ops.make_cfg()
    # density_only stays unsupported; null pointers are refused before any device work
    assert lib.fsnerf_mlp_backward_deterministic(C.byref(cfg), None, None, 128, None, None, None, 1, None, None,
                                                 None) == -3
    assert lib.fsnerf_mlp_backward_deterministic(C.byref(cfg), None, None, 128, None, None, None, 0, None, None,
                                                 None) == -1
    assert lib.fsnerf_mlp_backward_deterministic(C.byref(cfg), None, None, 0, None, None, None, 0, None, None,
                                                 None) == 0
    assert lib.fsnerf_adam_step_reg_deterministic(10, None, None, None, None, 1e-3, 0.9, 0.999, 1e-8, 1, 2, 1e-3,
                                                  1, None, None, None, None) == -1
