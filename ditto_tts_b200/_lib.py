"""ctypes binding of libditto_b200.so (include/ditto_b200.h).  There is no fallback: if the library
is missing or no B200 is visible, the product path raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libditto_b200.so")

PREC_FP32, PREC_BF16 = 0, 1
F_FUSED_ROPE, F_FOLD_CROSS, F_FUSED_ATTN, F_DEFER_LN, F_BLOCKS_ONLY = 1, 2, 4, 8, 16


class DittoError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("hidden_dim", C.c_int32), ("num_layers", C.c_int32), ("num_heads", C.c_int32),
                ("time_dim", C.c_int32), ("text_dim", C.c_int32), ("diffusion_steps", C.c_int32),
                ("precision", C.c_int32), ("max_seq_len", C.c_int32), ("flags", C.c_int32),
                ("reserved", C.c_int32 * 7)]


class SeqGroup(C.Structure):
    """ditto_seq_group_t: one group of equal-length sequences of a ragged batch."""
    _fields_ = [("n_seq", C.c_int64), ("n_x", C.c_int64), ("T", C.c_int64), ("S", C.c_int64), ("ctx", C.c_void_p)]


_P, _I64, _I32, _F = C.c_void_p, C.c_int64, C.c_int32, C.c_float

# name -> (restype, argtypes); mirrors include/ditto_b200.h one to one
SIGNATURES = {
    "ditto_abi_version": (_I32, []),
    "ditto_last_error": (C.c_char_p, []),
    "ditto_kernel_launch_count": (_I64, []),
    "ditto_profile_start": (_I32, []),
    "ditto_profile_stop": (_I32, []),
    "ditto_profile_num_classes": (_I32, []),
    "ditto_profile_class_name": (C.c_char_p, [_I32]),
    "ditto_profile_get": (_I32, [_I32, C.POINTER(_I64), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                 C.POINTER(C.c_double)]),
    "ditto_debug_set_counters": (_I32, [_P]),
    "ditto_debug_option": (_I32, [C.c_char_p, _I32]),
    "ditto_engine_create": (_I32, [C.POINTER(Config), C.POINTER(_P)]),
    "ditto_engine_destroy": (_I32, [_P]),
    "ditto_engine_load_weight": (_I32, [_P, C.c_char_p, _P, _I64, _P]),
    "ditto_engine_load_schedule": (_I32, [_P, _P, _P, _P, _I64, _P]),
    "ditto_engine_load_update_table": (_I32, [_P, _P, _I64, _P]),
    "ditto_engine_load_multistep_table": (_I32, [_P, _P, _I64, _P]),
    "ditto_engine_load_known_table": (_I32, [_P, _P, _I64, _P]),
    "ditto_engine_finalize": (_I32, [_P, _P]),
    "ditto_text_context_bytes": (_I64, [_P, _I64, _I64]),
    "ditto_workspace_bytes": (_I64, [_P, _I64, _I64, _I64]),
    "ditto_text_context": (_I32, [_P, _P, _I64, _I64, _P, _P, _I64, _P]),
    "ditto_forward": (_I32, [_P, _P, _I64, _P, _P, _I64, _I64, _I64, _P, _P, _I64, _P]),
    "ditto_cfg_ddpm_update": (_I32, [_P, _P, _P, _P, _P, _P, _F, _P, _I64, _I64, _P]),
    "ditto_p_sample": (_I32, [_P, _P, _P, _P, _P, _I32, _F, _I64, _I64, _I64, _P, _P, _P, _I64, _P]),
    "ditto_p_sample_rng": (_I32, [_P, _P, _P, _P, _P, _I32, _F, _I64, _I64, _I64, _P, _P, _P, _I64, _I32, _P]),
    "ditto_cfg_ddpm_update_rng": (_I32, [_P, _P, _P, _P, _P, _P, _I64, _F, _P, _I64, _I64, _I32, _P]),
    "ditto_randn": (_I32, [_P, _I64, _P, _I64, _P]),
    "ditto_cfg_multistep_update": (_I32, [_P, _P, _P, _P, _P, _P, _F, _P, _P, _I64, _I64, _P]),
    "ditto_cfg_multistep_update_rng": (_I32, [_P, _P, _P, _P, _P, _P, _I64, _F, _P, _P, _I64, _I64, _I32, _P]),
    "ditto_p_sample_multistep": (_I32, [_P, _P, _P, _P, _P, _I32, _F, _I64, _I64, _I64, _P, _P, _P, _P, _I64, _P]),
    "ditto_p_sample_multistep_rng": (_I32, [_P, _P, _P, _P, _P, _I32, _F, _I64, _I64, _I64, _P, _P, _P, _P, _I64, _I32, _P]),
    "ditto_cfg_update_known": (_I32, [_P, _P, _P, _P, _P, _P, _P, _I64, _F, _P, _P, _P, _P, _I64, _I64, _I32, _P]),
    "ditto_p_sample_known": (_I32, [_P, _P, _P, _P, _P, _P, _I32, _F, _I64, _I64, _I64, _P, _P, _P, _P, _P, _P, _I64, _I32, _P]),
    "ditto_q_sample": (_I32, [_P, _P, _P, _P, _P, _I64, _I64, _P]),
    "ditto_workspace_bytes_ragged": (_I64, [_P, C.POINTER(SeqGroup), _I64]),
    "ditto_forward_ragged": (_I32, [_P, _P, C.POINTER(SeqGroup), _I64, _P, _P, _P, _I64, _P]),
    "ditto_p_sample_ragged": (_I32, [_P, _P, C.POINTER(SeqGroup), _I64, _P, _P, _I32, _F, _P, _P, _P, _I64, _P]),
    "ditto_p_sample_ragged_rng": (_I32, [_P, _P, C.POINTER(SeqGroup), _I64, _P, _P, _I32, _F, _P, _P, _P, _I64, _I32, _P]),
    "ditto_p_sample_ragged_multistep": (_I32, [_P, _P, C.POINTER(SeqGroup), _I64, _P, _P, _I32, _F, _P, _P, _P, _P, _I64, _P]),
    "ditto_p_sample_ragged_multistep_rng": (_I32, [_P, _P, C.POINTER(SeqGroup), _I64, _P, _P, _I32, _F, _P, _P, _P, _P, _I64, _I32,
                                                   _P]),
    "ditto_p_sample_ragged_known": (_I32, [_P, _P, C.POINTER(SeqGroup), _I64, _P, _P, _P, _I32, _F, _P, _P, _P, _P, _P, _P, _I64,
                                           _I32, _P]),
    "ditto_dit_block": (_I32, [_P, _I32, _P, _P, _I64, _I64, _I64, _P, _P, _I64, _P]),
    "ditto_attn_self": (_I32, [_P, _I32, _P, _P, _I64, _I64, _I64, _P, _P, _I64, _P]),
    "ditto_attn_cross": (_I32, [_P, _I32, _P, _P, _I64, _I64, _I64, _P, _P, _I64, _P]),
    "ditto_gated_mlp": (_I32, [_P, _I32, _P, _P, _I64, _I64, _I64, _P, _P, _I64, _P]),
    "ditto_adaln_workspace_bytes": (_I64, [_I64, _I64, _I64, _I64]),
    "ditto_adaln": (_I32, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _P, _I64, _P]),
    "ditto_rope": (_I32, [_P, _P, _P, _I64, _I64, _I64, _I64, _P]),
    "ditto_attn_self768": (_I32, [_P, _I64, _I64, _I64, _F, _P, _P, _P, _P, _I32, _P]),
    "ditto_layernorm": (_I32, [_P, _P, _P, _P, _I32, _I64, _I64, _P]),
    "ditto_gemm_f32": (_I32, [_P, _I64, _I64, _P, _I64, _I64, _I32, _P, _I64, _I64, _P, _P, _F, _I64, _I64, _I64,
                              _I64, _P]),
    "ditto_gemm_resid_ln_weight_row": (_I32, [_I32]),
    "ditto_gemm_resid_ln": (_I32, [_P, _I64, _P, _I64, _P, _P, _I64, _P, _P, _P, _I64, _I64, _I64, _I64, _P]),
    "ditto_gemm_bf16": (_I32, [_P, _I64, _P, _I64, _P, _I64, _I32, _P, _P, _I64, _F, _I64, _I64, _I64, _P]),
    "ditto_cast_bf16": (_I32, [_P, _P, _I64, _P]),
    "ditto_vq_code_sqnorm": (_I32, [_P, _I64, _I64, _P, _P]),
    "ditto_vq_encode": (_I32, [_P, _I64, _I64, _I64, _P, _I64, _P, _I64, _P, _P]),
    "ditto_pool_latents": (_I32, [_P, _I64, _I64, _I64, _I64, _I64, _P, _P]),
    "ditto_mse_workspace_bytes": (_I64, []),
    "ditto_mse_loss": (_I32, [_P, _P, _I64, _P, _P, _I64, _P]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises DittoError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DittoError(f"{LIB_PATH} not found: build it with `python -m ditto_tts_b200.build` "
                         "(nvcc, sm_100a).  There is no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ditto_abi_version() != 1:
        raise DittoError("libditto_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().ditto_last_error().decode("utf-8", "replace")
        raise DittoError(f"{what or 'libditto_b200'} failed (code {rc}): {msg}")


def debug_option(name: str, value: int):
    """Developer A/B switch of the kernels (DESIGN.md section 9); ``debug_option("reset", 0)`` restores the product path.
    Engine-level options are sampled when an engine is created."""
    check(load().ditto_debug_option(name.encode(), int(value)), f"ditto_debug_option({name})")


def launch_count() -> int:
    return int(load().ditto_kernel_launch_count())


def profile_start():
    check(load().ditto_profile_start(), "ditto_profile_start")


def profile_stop():
    """Returns {class_name: dict(launches, ms, flops, bytes)} for the classes that launched."""
    lib = load()
    check(lib.ditto_profile_stop(), "ditto_profile_stop")
    out = {}
    for i in range(lib.ditto_profile_num_classes()):
        n, ms, fl, by = _I64(), C.c_double(), C.c_double(), C.c_double()
        check(lib.ditto_profile_get(i, C.byref(n), C.byref(ms), C.byref(fl), C.byref(by)))
        if n.value:
            out[lib.ditto_profile_class_name(i).decode()] = dict(launches=n.value, ms=ms.value, flops=fl.value,
                                                                 bytes=by.value)
    return out
