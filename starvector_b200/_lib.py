"""ctypes binding of the C-ABI in include/starvector_b200.h (the whole product boundary).

No torch types cross this boundary: tensors are passed as raw device pointers plus sizes and
the current CUDA stream handle.  Loading fails loudly when the library has not been built —
there is no Python/CPU fallback for any entry point.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SV_LIB_PATH") or os.path.join(_HERE, "libstarvector_b200.so")   # SV_LIB_PATH: A/B builds

SV_OK, SV_ERR_INVALID, SV_ERR_CUDA, SV_ERR_UNSUPPORTED, SV_ERR_STATE = 0, -1, -2, -3, -4
SV_DTYPE_BF16, SV_DTYPE_F32, SV_DTYPE_F16 = 0, 1, 2
SV_ACT_NONE, SV_ACT_QUICKGELU, SV_ACT_GELU_TANH, SV_ACT_SILU = 0, 1, 2, 3
SV_LINEAR_AUTO, SV_LINEAR_ROWGROUP, SV_LINEAR_TCGEN05 = 0, 1, 2
SV_ATTN_DECODE_CLUSTER, SV_ATTN_DECODE_SPLIT = 0, 1
SV_GEMV_EPI_PLAIN, SV_GEMV_EPI_QKV, SV_GEMV_EPI_LMHEAD = 0, 1, 2
SV_SELECT_GREEDY, SV_SELECT_FUSED, SV_SELECT_FUSED_PARTIALS, SV_SELECT_SAMPLE = 0, 1, 2, 3
ABI_VERSION = 6
SV_ALPHA_WHITE, SV_ALPHA_DROP = 0, 1


class ModelDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "variant", "image_size", "patch_size", "vit_width", "vit_layers", "vit_heads", "vit_mlp", "adapter_norm",
        "hidden", "n_layer", "n_head", "n_kv_head", "head_dim", "n_inner", "n_positions", "vocab")] + [
        ("ln_eps", C.c_float), ("max_batch", C.c_int32), ("max_len", C.c_int32),
        ("rope_theta", C.c_float), ("sliding_window", C.c_int32), ("vit_ln_eps", C.c_float)]


class GenParams(C.Structure):
    _fields_ = [
        ("max_new_tokens", C.c_int32), ("do_sample", C.c_int32), ("temperature", C.c_float), ("top_p", C.c_float),
        ("repetition_penalty", C.c_float), ("eos_token_id", C.c_int32), ("pad_token_id", C.c_int32),
        ("n_stop_ids", C.c_int32), ("stop_ids", C.c_int32 * 8), ("stop_row0_only", C.c_int32),
        ("seed", C.c_uint64), ("poll_interval", C.c_int32),
    ]


class BeamParams(C.Structure):
    _fields_ = [
        ("num_beams", C.c_int32), ("max_new_tokens", C.c_int32), ("do_sample", C.c_int32), ("early_stopping", C.c_int32),
        ("temperature", C.c_float), ("top_p", C.c_float), ("repetition_penalty", C.c_float), ("length_penalty", C.c_float),
        ("eos_token_id", C.c_int32), ("pad_token_id", C.c_int32), ("n_stop_ids", C.c_int32), ("stop_ids", C.c_int32 * 8),
        ("poll_interval", C.c_int32), ("seed", C.c_uint64),
    ]


class PreprocDesc(C.Structure):
    _fields_ = [("out_size", C.c_int32), ("alpha_mode", C.c_int32), ("pad_square", C.c_int32), ("out_dtype", C.c_int32),
                ("mean", C.c_float * 3), ("std", C.c_float * 3)]


class ImageU8(C.Structure):
    _fields_ = [("data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("channels", C.c_int32),
                ("row_stride", C.c_int32)]


TOKEN_CALLBACK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int32)   # sv_token_callback

# name -> (restype, argtypes); must list every SV_API symbol of the header (tests check this)
_P, _I, _F = C.c_void_p, C.c_int32, C.c_float
SIGNATURES = {
    "sv_abi_version": (C.c_int, []),
    "sv_engine_create": (C.c_int, [C.POINTER(ModelDesc), C.c_int, C.POINTER(_P)]),
    "sv_engine_destroy": (None, [_P]),
    "sv_last_error": (C.c_char_p, [_P]),
    "sv_engine_load_weight": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), _I, _I]),
    "sv_engine_missing_weights": (C.c_int, [_P]),
    "sv_encode_images": (C.c_int, [_P, _P, _I, _P, _P, _P]),
    "sv_prefill": (C.c_int, [_P, _P, _I, _I, _P, _P]),
    "sv_prefill_embeds": (C.c_int, [_P, _P, _I, _I, _P, _P]),
    "sv_decode_step": (C.c_int, [_P, _P, _P, _P]),
    "sv_reorder_cache": (C.c_int, [_P, _P, _P]),
    "sv_expand_batch": (C.c_int, [_P, _P, C.c_int32, _P]),
    "sv_extend": (C.c_int, [_P, _P, _I, _P, _I, _P, _F, _P]),
    "sv_beam_search": (C.c_int, [_P, C.POINTER(BeamParams), _I, _P, _P, _P]),
    "sv_beam_params_check": (C.c_int, [C.POINTER(BeamParams), _I]),
    "sv_beam_state_bytes": (C.c_int, []),
    "sv_beam_state_init_host": (C.c_int, [C.POINTER(BeamParams), _I, _I, _P]),
    "sv_beam_state_read_host": (C.c_int, [_P, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(C.c_float)]),
    "sv_beam_row_candidates_host": (C.c_int, [C.POINTER(BeamParams), C.POINTER(C.c_float), _I, C.POINTER(_I), _I, _F, _I, _I,
                                              C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(_I)]),
    "sv_beam_step_host": (C.c_int, [C.POINTER(BeamParams), _I, _I, _I, _P, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                    C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "sv_generate": (C.c_int, [_P, C.POINTER(GenParams), _P, _P, _P]),
    "sv_generate_stream": (C.c_int, [_P, C.POINTER(GenParams), _P, _P, TOKEN_CALLBACK, _P, _P]),
    "sv_generate_im2svg_host": (C.c_int, [_P, _P, _I, _P, _I, C.POINTER(GenParams), _P, _P, _P]),
    "sv_launch_count": (C.c_int64, [_P]),
    "sv_engine_describe": (C.c_char_p, [_P]),
    "sv_debug_read_timeline": (C.c_int, [_P, C.POINTER(C.c_longlong), _I]),
    "sv_last_decode_timing": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "sv_op_layernorm": (C.c_int, [_P, _P, _P, _P, _I, _I, _F, _P]),
    "sv_op_linear": (C.c_int, [_I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "sv_op_attention_vit": (C.c_int, [_P, _P, _I, _I, _I, _P]),
    "sv_op_attention_mqa": (C.c_int, [_P, _P, _I, _I, _I, _P]),
    "sv_op_attention_prefill": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "sv_op_attention_decode": (C.c_int, [_I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "sv_op_gemv_ring": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _I, _I, _P, _P, _I, _I, _I, _I, _P, _P, _I,
                                  C.POINTER(_I), _P]),
    "sv_op_lm_head_logps": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _F, _P]),
    "sv_op_select": (C.c_int, [_I, _P, _P, C.POINTER(GenParams), _I, _I, _I, _I, _P, _P, _I, _P, _P, _I, _I, _P, _P, _P]),
    "sv_preproc_create": (C.c_int, [C.POINTER(PreprocDesc), C.c_int, C.POINTER(_P)]),
    "sv_preproc_destroy": (None, [_P]),
    "sv_preproc_last_error": (C.c_char_p, [_P]),
    "sv_preproc_run_host": (C.c_int, [_P, C.POINTER(ImageU8), _I, _P, _P]),
    "sv_preproc_launch_count": (C.c_longlong, [_P]),
    "sv_resample_coeffs_host": (C.c_int, [_I, _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), _I]),
    "sv_preproc_lut_host": (C.c_int, [C.POINTER(PreprocDesc), C.POINTER(C.c_float)]),
    "sv_preproc_plan_host": (C.c_int, [C.POINTER(PreprocDesc), C.POINTER(ImageU8), _I, _P, C.c_int64, C.POINTER(C.c_int64)]),
}

_lib = None


def load() -> C.CDLL:
    """Load libstarvector_b200.so (built by `python -m starvector_b200.build` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA library has not been built. Run `python -m starvector_b200.build` "
            "(needs nvcc). starvector_b200 has no CPU or PyTorch fallback path."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.sv_abi_version() != ABI_VERSION:
        raise RuntimeError(f"ABI mismatch: library {lib.sv_abi_version()} vs binding {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


class EngineError(RuntimeError):
    """Any non-zero return of the C-ABI (SV_ERR_INVALID is raised as ValueError instead)."""


def check(lib, code: int, handle=None) -> None:
    if code == SV_OK:
        return
    msg = lib.sv_last_error(handle)
    text = msg.decode("utf-8", "replace") if msg else ""
    if code == SV_ERR_INVALID:
        raise ValueError(f"starvector_b200: {text}")
    if code == SV_ERR_UNSUPPORTED:
        raise NotImplementedError(f"starvector_b200: {text}")
    raise EngineError(f"starvector_b200 (code {code}): {text}")
