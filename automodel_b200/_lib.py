"""ctypes binding of libb200_train.so (C ABI: include/b200_train.h).  Fails loudly if the library is missing."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libb200_train.so")

_lib = None

_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/b200_train.h declares
SIGNATURES = {
    "b200_last_error": (C.c_char_p, []),
    "b200_abi_version": (_i, []),
    "b200_device_check": (_i, []),
    "b200_set_option": (_i, [C.c_char_p, _i]),
    "b200_gemm_bf16": (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_gemm_bf16_cublaslt": (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    "b200_rmsnorm_fwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "b200_rmsnorm_bwd_workspace_floats": (_i, [_i, _i]),
    "b200_rmsnorm_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _vp]),
    "b200_rope_inplace": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200_bias_rope_inplace": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200_colsum_workspace_floats": (_i, [_i, _i]),
    "b200_colsum_bf16": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i, _vp]),
    "b200_swiglu_fwd": (_i, [_vp, _vp, _i64, _i, _vp]),
    "b200_swiglu_bwd": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "b200_embed_fwd": (_i, [_vp, _vp, _vp, _i, _i, _vp]),
    "b200_embed_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "b200_attn_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i64, _i64, _i64, _i64, _i, _i, _i, _i, _f, _vp]),
    "b200_attn_bwd_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "b200_attn_bwd": (_i, [_vp] * 10 + [_sz, _vp] + [_i, _i] + [_i64] * 8 + [_i, _i, _i, _i, _f, _vp]),
    "b200_ce_fwd_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i64, _i64, _i, _vp]),
    "b200_sumsq_workspace_floats": (_i, []),
    "b200_sumsq_bf16": (_i, [_vp, _i64, _vp, _vp, _i, _vp]),
    "b200_adamw_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _i, _f, _vp, _i, _vp]),
    "b200_add_inplace_bf16": (_i, [_vp, _vp, _i64, _vp]),
    "b200_ctx_create": (_i, [C.POINTER(_vp), _i, _i]),
    "b200_ctx_destroy": (_i, [_vp]),
    "b200_ctx_set_timeout_ms": (_i, [_vp, _i64]),
    "b200_ctx_signal_pad_bytes": (_sz, []),
    "b200_ctx_set_signal_pad": (_i, [_vp, C.POINTER(_vp), _sz]),
    "b200_ctx_register_buffer": (_i, [_vp, _i, C.POINTER(_vp), _vp, _sz]),
    "b200_ctx_has_multicast": (_i, [_vp, _i]),
    "b200_reducescatter_layer": (_i, [_vp, _i, _sz, _i64, _i, _i, _vp]),
    "b200_allgather_layer": (_i, [_vp, _i, _sz, _i64, _i, _i, _vp]),
    "b200_allreduce_scalars": (_i, [_vp, _vp, _i, _vp]),
}


class B200Error(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle.  No fallback: a missing build is an error."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  automodel_b200 has no CPU or library fallback.")
        try:
            import torch  # noqa: F401  (makes torch's libcublasLt resident so the rpath lookup is not needed)
        except Exception:
            pass
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().b200_last_error().decode(errors="replace")
        raise B200Error(f"{what} failed (code {rc}): {msg}")
