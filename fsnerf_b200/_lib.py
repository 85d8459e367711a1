"""ctypes binding of libfsnerf_b200.so (the C ABI declared in include/fsnerf_b200.h).

There is no fallback: if the shared library is missing, or a compute entry
point is called without an sm_100 device, this raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfsnerf_b200.so")


class NetCfg(C.Structure):
    """mirror of fsnerf_net_cfg"""
    _fields_ = [("n_layers", C.c_int), ("d_hidden", C.c_int), ("skip_mask", C.c_int),
                ("n_freqs_pos", C.c_int), ("n_freqs_dir", C.c_int), ("log_space", C.c_int)]


class FsnerfError(RuntimeError):
    pass


_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_f = C.c_float

# name -> (restype, argtypes); must list every symbol of include/fsnerf_b200.h
SIGNATURES = {
    "fsnerf_version": (_i, []),
    "fsnerf_last_error": (C.c_char_p, []),
    "fsnerf_device_ok": (_i, [_i]),
    "fsnerf_gen_rays": (_i, [_p, _i, _i, _i, _i, _f, _p, _l, _l, _i, _f, _f, _f, _p, _p, _p, _p, _p]),
    "fsnerf_to_ndc": (_i, [_p, _p, _l, _f, _f, _f, _p, _p, _p]),
    "fsnerf_sample_stratified": (_i, [_l, _i, _f, _f, _p, _p, _p, _p]),
    "fsnerf_sample_pdf": (_i, [_l, _i, _i, _p, _p, _p, _f, _p, _p, _p, _p, _p, _p]),
    "fsnerf_sample_stratified_seeded": (_i, [_l, _i, _f, _f, C.c_uint64, _p, _p, _p]),
    "fsnerf_sample_pdf_seeded": (_i, [_l, _i, _i, _p, _p, C.c_uint64, _f, _p, _p, _p, _p, _p, _p]),
    "fsnerf_rng_uniform": (_i, [_l, C.c_uint64, _p, _p]),
    "fsnerf_composite_forward": (_i, [_l, _i, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p]),
    "fsnerf_composite_backward": (_i, [_l, _i, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p]),
    "fsnerf_composite_backward_occ": (_i, [_l, _i, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p,
                                          _i, _f, _f, _f, _p, _p]),
    "fsnerf_encode": (_i, [_l, _i, _i, _p, _p, _p, _p, _p]),
    "fsnerf_occgrid_march": (_i, [_l, _p, _p, _p, _f, _f, _f, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p]),
    "fsnerf_occgrid_filter": (_i, [_l, _p, _p, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p]),
    "fsnerf_packed_points": (_i, [_l, _p, _p, _p, _p, _p, _p, _p, _p]),
    "fsnerf_composite_packed_forward": (_i, [_l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "fsnerf_composite_packed_backward": (_i, [_l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "fsnerf_occgrid_update": (_i, [_l, _p, _p, _f, _p, _p, _p]),
    "fsnerf_occgrid_binarize": (_i, [_l, _p, _f, _p, _p]),
    "fsnerf_mlp_param_count": (_l, [C.POINTER(NetCfg)]),
    "fsnerf_mlp_param_layout": (_i, [C.POINTER(NetCfg), C.POINTER(_l), C.POINTER(_l), _i]),
    "fsnerf_mlp_packed_bytes": (_l, [C.POINTER(NetCfg)]),
    "fsnerf_mlp_stash_bytes": (_l, [C.POINTER(NetCfg), _l]),
    "fsnerf_mlp_bwd_workspace_bytes": (_l, [C.POINTER(NetCfg), _l]),
    "fsnerf_mlp_pack": (_i, [C.POINTER(NetCfg), _p, _p, _p]),
    "fsnerf_mlp_forward": (_i, [C.POINTER(NetCfg), _p, _p, _l, _i, _p, _p, _p, _p, _p, _p, _p, _p,
                                _i, _p, _p, _p]),
    "fsnerf_mlp_backward": (_i, [C.POINTER(NetCfg), _p, _p, _l, _p, _p, _p, _i, _p, _p, _p]),
    "fsnerf_mse_loss_grad": (_i, [_l, _p, _p, _f, _p, _p, _p]),
    "fsnerf_profile_enable": (_i, [_i]),
    "fsnerf_profile_read": (_i, [_i, C.c_char_p, C.POINTER(_f), C.POINTER(_i)]),
    "fsnerf_debug_set_trace": (_i, [_p]),
    "fsnerf_adam_step": (_i, [_l, _p, _p, _p, _p, _f, _f, _f, _f, _i, _p]),
    "fsnerf_adam_step_reg": (_i, [_l, _p, _p, _p, _p, _f, _f, _f, _f, _i, _i, _f, _i,
                                 C.POINTER(_l), C.POINTER(_l), _p, _p]),
}

_lib = None


def load():
    """dlopen the library (once) and declare every prototype."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FsnerfError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
                f"g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = load().fsnerf_last_error().decode(errors="replace")
        raise FsnerfError(f"{what} failed ({rc}): {msg}")


def ptr(t):
    """device pointer of a torch tensor (None -> NULL)"""
    return None if t is None else C.c_void_p(t.data_ptr())
