"""ctypes binding of ``libdotaclient_b200.so`` (the C-ABI in ``include/dotaclient_b200.h``).

There is NO fallback: if the library is missing or a call fails, a ``RuntimeError`` is raised.
The library is built in-tree by ``dotaclient_b200.build`` (``__graft_entry__.build()``).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdotaclient_b200.so")

_c = ctypes
_vp, _i32, _i64, _f32, _f64, _sz = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float, _c.c_double, _c.c_size_t
_ptr5 = _c.c_void_p * 5

# name -> (restype, argtypes); must list every symbol include/dotaclient_b200.h declares.
SIGNATURES = {
    "dc_version": (_i32, []),
    "dc_last_error": (_c.c_char_p, []),
    "dc_device_info": (_i32, [_c.POINTER(_i32)] * 3),
    "dc_gae_scan": (_i32, [_vp, _i32, _vp, _vp, _i32, _vp, _vp, _f64, _f64, _vp, _vp, _vp]),
    "dc_rnn_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "dc_rnn_seq_fwd": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "dc_rnn_seq_bwd": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "dc_gemm_tf32x3_supported": (_i32, [_i64, _i32, _i32]),
    "dc_gemm_tf32x3": (_i32, [_vp, _i32, _vp, _i32, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _vp]),
    "dc_gemm_wgrad_workspace_bytes": (_sz, [_i32, _i32]),
    "dc_gemm_wgrad_tf32x3": (_i32, [_vp, _i32, _vp, _i32, _i64, _i32, _i32, _vp, _i32, _vp, _i32, _vp, _vp]),
    "dc_gemm_tf32x3_blocked": (_i32, [_vp, _i32, _i64, _i64, _vp, _i32, _vp, _vp, _i32, _i64, _i64, _i64, _i32, _i32, _i32,
                                      _vp]),
    "dc_gemm_wgrad_tf32x3_blocked": (_i32, [_vp, _i32, _i64, _i64, _vp, _i32, _i64, _i32, _i32, _vp, _i32, _vp, _i32, _vp,
                                            _vp]),
    "dc_unit_basic_fwd": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "dc_unit_basic_fwd_mask": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "dc_unit_basic_bwd_workspace_bytes": (_sz, []),
    "dc_env_fwd": (_i32, [_vp, _vp, _vp, _vp, _i32, _i64, _vp]),
    "dc_env_bwd_workspace_bytes": (_sz, []),
    "dc_env_bwd": (_i32, [_vp, _vp, _i32, _vp, _vp, _vp, _i64, _vp, _vp]),
    "dc_unit_wgrad_routed": (_i32, [_vp, _vp, _i32, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    "dc_unit_dgrad_fused": (_i32, [_vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _i32, _vp, _vp]),
    "dc_unit_dgrad_fused_mask": (_i32, [_vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _i32, _vp, _vp]),
    "dc_gemm_unit_max": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _i64, _i32, _vp]),
    "dc_target_unit_q_fwd": (_i32, [_vp, _i32, _c.c_void_p * 6, _vp, _i64, _vp]),
    "dc_target_unit_q_bwd": (_i32, [_vp, _c.c_void_p * 6, _vp, _i32, _i64, _vp]),
    "dc_target_unit_fwd": (_i32, [_vp, _vp, _vp, _i64, _vp]),
    "dc_target_unit_bwd": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "dc_ppo_loss_fwd_bwd": (_i32, [_ptr5, _ptr5, _ptr5, _vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _ptr5, _vp, _vp,
                                   _vp, _vp, _vp]),
    "dc_ppo_loss_fwd_bwd_strided": (_i32, [_ptr5, _c.c_int64 * 5, _ptr5, _ptr5, _vp, _vp, _vp, _vp, _i64, _i64, _f32, _f32, _f32,
                                           _ptr5, _c.c_int64 * 5, _vp, _i64, _vp, _vp, _vp, _vp]),
    "dc_selected_logp": (_i32, [_ptr5, _ptr5, _ptr5, _i64, _vp, _vp]),
    "dc_select_actions": (_i32, [_ptr5, _c.c_int64 * 5, _ptr5, _vp, _i64, _vp, _vp, _vp]),
    "dc_grad_flags": (_i32, [_vp, _i64, _vp, _i32, _vp, _vp]),
    "dc_grad_finish": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _f64, _f64, _f64, _f64, _f64, _vp, _vp,
                              _vp, _vp]),
}

PPO_WORKSPACE_BYTES = 512
FINISH_WORKSPACE_BYTES = 1024
LOSS_SLOTS = 16

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load():
    """Loads the shared library (once).  Raises if it has not been built -- no silent fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            "%s not found: build it with `python -m dotaclient_b200.build` (needs nvcc, sm_100a). "
            "dotaclient_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            continue
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported(name):
    lib = load()
    return hasattr(lib, name)


def check(rc, what):
    if rc != 0:
        msg = load().dc_last_error()
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def ptr5(tensors):
    return _ptr5(*[t.data_ptr() if t is not None else None for t in tensors])


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
