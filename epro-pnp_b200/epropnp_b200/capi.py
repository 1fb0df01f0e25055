"""ctypes binding of include/epropnp_b200.h.  There is no fallback: if the shared library is missing
or a call fails, a NativeError is raised."""
import ctypes
import os

import torch

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB_PATH = os.path.join(_PKG_ROOT, "lib", "libepropnp_b200.so")
_lib = None

c_float_p = ctypes.c_void_p


class NativeError(RuntimeError):
    pass


class EpnpParams(ctypes.Structure):
    _fields_ = [("dof", ctypes.c_int32), ("lm_iter", ctypes.c_int32), ("fast_mode", ctypes.c_int32),
                ("z_min", ctypes.c_float), ("min_lm_diagonal", ctypes.c_float),
                ("max_lm_diagonal", ctypes.c_float), ("min_relative_decrease", ctypes.c_float),
                ("initial_radius", ctypes.c_float), ("max_radius", ctypes.c_float), ("eps", ctypes.c_float),
                ("huber_eps", ctypes.c_float), ("mc_samples", ctypes.c_int32), ("mc_iter", ctypes.c_int32),
                ("amis_eps", ctypes.c_float), ("acg_mle_iter", ctypes.c_int32), ("acg_dispersion", ctypes.c_float)]


def lib_path():
    return _LIB_PATH


_P = ctypes.c_void_p
_I = ctypes.c_int
_F = ctypes.c_float
ABI_VERSION = 2            # EPNP_ABI_VERSION of include/epropnp_b200.h

_SIGNATURES = {
    "epnp_abi_version": (ctypes.c_int, []),
    "epnp_error_string": (ctypes.c_char_p, [_I]),
    "epnp_last_cuda_error": (ctypes.c_int, []),
    "epnp_default_params": (None, [ctypes.POINTER(EpnpParams), _I]),
    "epnp_max_points": (ctypes.c_int, [_I, _I, _I]),
    "epnp_adaptive_delta_f32": (ctypes.c_int, [_P, _P, _F, _P, _I, _I, _P]),
    "epnp_evaluate_cost_f32": (ctypes.c_int, [_P] * 9 + [_I, _I, _I, _I, _F, _P]),
    "epnp_evaluate_f32": (ctypes.c_int, [_P] * 11 + [_I, _I, _I, _I, _F, _F, _P]),
    "epnp_lm_solve_f32": (ctypes.c_int, [_P] * 13 + [_I, _I, ctypes.POINTER(EpnpParams), _P]),
    "epnp_gn_plus_backward_f32": (ctypes.c_int, [_P] * 13 + [_I, _I, _I, _F, _F, _F, _P]),
    "epnp_rslm_draw_f32": (ctypes.c_int, [_P] * 5 + [ctypes.c_uint64, ctypes.c_uint32, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
    "epnp_epnp_init_f32": (ctypes.c_int, [_P] * 4 + [_F, _P, _P, _I, _I, _P]),
    "epnp_rslm_f32": (ctypes.c_int, [_P] * 13 + [_I, _I, _I, _I, ctypes.POINTER(EpnpParams), _P]),
    "epnp_amis_f32": (ctypes.c_int, [_P] * 12 + [ctypes.c_uint64, ctypes.c_uint32] + [_P] * 3
                      + [_I, _I, ctypes.POINTER(EpnpParams), _P]),
    "epnp_lm_amis_fused_f32": (ctypes.c_int, [_P] * 11 + [ctypes.c_uint64, ctypes.c_uint32] + [_P] * 8
                               + [_I, _I, ctypes.POINTER(EpnpParams), _P]),
    "epnp_lm_amis_fused_push_f32": (ctypes.c_int, [_P] * 8 + [ctypes.c_uint64, ctypes.c_uint32] + [_P] * 5
                                    + [_P, _P, _I, _I, _I, ctypes.POINTER(EpnpParams), _P]),
    "epnp_cost_backward_f32": (ctypes.c_int, [_P] * 7 + [_P, _P, _I, _P, _P, _I] + [_P] * 4 + [_I, _I, _I, _F, _P]),
    "epnp_mc_epilogue_f32": (ctypes.c_int, [_P] * 8 + [_I, _I, _I, _P]),
    "epnp_mc_lse_backward_f32": (ctypes.c_int, [_P] * 4 + [_I, _I, _P]),
    "epnp_fused_workspace_bytes": (ctypes.c_size_t, [_I, _I, ctypes.POINTER(EpnpParams)]),
    "epnp_lm_amis_fused_host_f32": (ctypes.c_int, [_P] * 8 + [ctypes.c_uint64, ctypes.c_uint32] + [_P] * 5
                                    + [_P, ctypes.c_size_t, _I, _I, _I, ctypes.POINTER(EpnpParams), _P]),
}


def exported_symbols():
    return sorted(_SIGNATURES)


def lib():
    """The loaded shared library (built in-tree by __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise NativeError(
                f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU / PyTorch fallback for the EPro-PnP hot path.")
        handle = ctypes.CDLL(_LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.epnp_abi_version() != ABI_VERSION:
            raise NativeError(f"libepropnp_b200.so ABI version {handle.epnp_abi_version()}, this package binds version "
                              f"{ABI_VERSION}: rebuild it (python -c 'import __graft_entry__ as g; g.build()')")
        _lib = handle
    return _lib


def default_params(dof=6, **overrides):
    p = EpnpParams()
    lib().epnp_default_params(ctypes.byref(p), int(dof))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def check(rc, what="epnp call"):
    if rc != 0:
        msg = lib().epnp_error_string(rc).decode()
        if rc == -4:
            msg += f" [cudaError {lib().epnp_last_cuda_error()}]"
        raise NativeError(f"{what} failed: {msg} (code {rc})")


def ptr(t):
    """Device (or host) pointer of a contiguous float32 tensor, None -> NULL."""
    if t is None:
        return None
    assert t.dtype == torch.float32 and t.is_contiguous(), "native path needs contiguous float32"
    return ctypes.c_void_p(t.data_ptr())


def iptr(t):
    """Pointer of a contiguous int32 tensor."""
    assert t.dtype == torch.int32 and t.is_contiguous(), "index arguments are contiguous int32"
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
