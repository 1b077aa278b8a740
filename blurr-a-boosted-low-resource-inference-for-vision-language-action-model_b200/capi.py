"""ctypes binding of `include/blurr_pi0.h` (libblurr_pi0.so).

The library is the product: if it is missing or cannot be loaded this module raises — there is
no Python/CPU fallback for the compute path.
"""

from __future__ import annotations

import ctypes as C
import os
from typing import Optional

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "lib", "libblurr_pi0.so")

ABI_VERSION = 1
BLURR_BF16, BLURR_F32, BLURR_I64 = 1, 0, 2
EPI_STORE, EPI_GELU, EPI_GEGLU, EPI_PARTIAL = 0, 1, 2, 3


class BlurrError(RuntimeError):
    """A non-zero status from the C ABI (message from `blurr_last_error`)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"blurr_pi0 status {status}: {message}")
        self.status = status


class Pi0ConfigC(C.Structure):
    """`blurr_pi0_config` (include/blurr_pi0.h)."""

    _fields_ = [
        ("abi_version", C.c_int32),
        ("vision_layers", C.c_int32), ("vision_hidden", C.c_int32), ("vision_intermediate", C.c_int32),
        ("vision_heads", C.c_int32), ("image_size", C.c_int32), ("patch_size", C.c_int32),
        ("num_image_tokens", C.c_int32), ("layer_norm_eps", C.c_float),
        ("joint_layers", C.c_int32), ("num_heads", C.c_int32), ("num_kv_heads", C.c_int32),
        ("head_dim", C.c_int32), ("vlm_hidden", C.c_int32), ("vlm_intermediate", C.c_int32),
        ("expert_hidden", C.c_int32), ("expert_intermediate", C.c_int32), ("rms_norm_eps", C.c_float),
        ("max_image_text_tokens", C.c_int32), ("num_proprio_tokens", C.c_int32),
        ("num_action_tokens", C.c_int32), ("action_dim", C.c_int32), ("proprio_dim", C.c_int32),
        ("vocab_size", C.c_int64), ("image_token_index", C.c_int64), ("pad_token_id", C.c_int64),
        ("num_inference_steps", C.c_int32), ("has_clip", C.c_int32),
        ("final_action_clip_value", C.c_float),
    ]


class LlmConfigC(C.Structure):
    """`blurr_llm_config` (include/blurr_llm.h)."""

    _fields_ = [
        ("abi_version", C.c_int32), ("num_layers", C.c_int32), ("hidden", C.c_int32), ("num_heads", C.c_int32),
        ("num_kv_heads", C.c_int32), ("head_dim", C.c_int32), ("intermediate", C.c_int32), ("vocab", C.c_int32),
        ("max_positions", C.c_int32), ("rms_eps", C.c_float),
    ]


LLM_ABI_VERSION = 2


class LlmSamplingC(C.Structure):
    """`blurr_llm_sampling` (include/blurr_llm.h): 24 bytes, seed at 0, temperature 8, top_k 12, top_p 16."""

    _fields_ = [("seed", C.c_uint64), ("temperature", C.c_float), ("top_k", C.c_int32), ("top_p", C.c_float)]


class VitConfigC(C.Structure):
    """`blurr_vit_config` (include/blurr_vit.h)."""

    _fields_ = [
        ("abi_version", C.c_int32), ("num_layers", C.c_int32), ("hidden", C.c_int32), ("num_heads", C.c_int32),
        ("mlp_dim", C.c_int32), ("image_size", C.c_int32), ("patch_size", C.c_int32), ("num_prefix_tokens", C.c_int32),
        ("use_layerscale", C.c_int32), ("gelu_erf", C.c_int32), ("ln_eps", C.c_float),
    ]


VIT_ABI_VERSION = 1


class Pi0InputsC(C.Structure):
    """`blurr_pi0_inputs` (include/blurr_pi0.h)."""

    _fields_ = [
        ("input_ids", C.c_void_p),
        ("pixel_values", C.c_void_p),
        ("pixel_strides", C.c_int64 * 4),
        ("image_text_proprio_mask", C.c_void_p),
        ("itp_mask_bstride", C.c_int64), ("itp_mask_rstride", C.c_int64),
        ("action_mask", C.c_void_p),
        ("action_mask_bstride", C.c_int64), ("action_mask_rstride", C.c_int64),
        ("vlm_position_ids", C.c_void_p),
        ("proprio_position_ids", C.c_void_p),
        ("action_position_ids", C.c_void_p),
        ("proprios", C.c_void_p),
        ("noise", C.c_void_p),
    ]


# every symbol `include/blurr_pi0.h` declares: (name, restype, argtypes)
_SIGNATURES = [
    ("blurr_abi_version", C.c_int, []),
    ("blurr_last_error", C.c_char_p, []),
    ("blurr_pi0_create", C.c_int, [C.POINTER(Pi0ConfigC), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("blurr_pi0_destroy", None, [C.c_void_p]),
    ("blurr_pi0_set_weight", C.c_int,
     [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.c_int]),
    ("blurr_pi0_set_rope_inv_freq", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_float), C.c_int]),
    ("blurr_pi0_set_time_table", C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    ("blurr_pi0_finalize_weights", C.c_int, [C.c_void_p]),
    ("blurr_pi0_infer_action", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(Pi0InputsC), C.c_void_p]),
    ("blurr_pi0_set_option", C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    ("blurr_pi0_check", C.c_int, [C.c_void_p, C.c_void_p]),
    ("blurr_pi0_debug_tap", C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    ("blurr_pi0_last_launch_count", C.c_int64, [C.c_void_p]),
    ("blurr_pi0_profile_report", C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t]),
    ("blurr_pi0_trace_report", C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t]),
    ("blurr_pi0_weight_bytes", C.c_int64, [C.c_void_p]),
    ("blurr_preproc_create", C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("blurr_preproc_destroy", None, [C.c_void_p]),
    ("blurr_preproc_build_tables", C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int16)]),
    ("blurr_preproc_tables", C.c_int,
     [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int16), C.POINTER(C.c_int32), C.POINTER(C.c_int16)]),
    ("blurr_preproc_frame", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    ("blurr_op_normalize_proprio", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("blurr_set_global_option", C.c_int, [C.c_char_p, C.c_int64]),
    ("blurr_op_pack_weight", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("blurr_op_gemm", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
      C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    ("blurr_op_gemm_async", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
      C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    ("blurr_op_pair_raster", C.c_int,
     [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int32), C.c_int]),
    ("blurr_op_siglip_attention", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    ("blurr_op_joint_attention", C.c_int,
     [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
      C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    # include/blurr_llm.h
    ("blurr_llm_create", C.c_int, [C.POINTER(LlmConfigC), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("blurr_llm_destroy", None, [C.c_void_p]),
    ("blurr_llm_set_weight", C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int]),
    ("blurr_llm_set_rope_table", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    ("blurr_llm_finalize", C.c_int, [C.c_void_p]),
    ("blurr_llm_embed", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    ("blurr_llm_generate", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(LlmSamplingC), C.c_int, C.c_void_p,
      C.c_void_p]),
    ("blurr_llm_sample", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(LlmSamplingC), C.c_int, C.c_void_p, C.c_void_p]),
    ("blurr_llm_set_option", C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    ("blurr_llm_check", C.c_int, [C.c_void_p, C.c_void_p]),
    ("blurr_llm_trace_report", C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t]),
    ("blurr_llm_last_launch_count", C.c_int64, [C.c_void_p]),
    ("blurr_llm_weight_bytes_per_token", C.c_int64, [C.c_void_p]),
    # include/blurr_vit.h
    ("blurr_vit_create", C.c_int, [C.POINTER(VitConfigC), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("blurr_vit_destroy", None, [C.c_void_p]),
    ("blurr_vit_set_weight", C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int]),
    ("blurr_vit_finalize", C.c_int, [C.c_void_p]),
    ("blurr_vit_forward", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p, C.c_int]),
    ("blurr_vit_set_option", C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    ("blurr_vit_last_launch_count", C.c_int64, [C.c_void_p]),
    ("blurr_mlp_create", C.c_int, [C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("blurr_mlp_destroy", None, [C.c_void_p]),
    ("blurr_mlp_set_weight", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    ("blurr_mlp_forward", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    ("blurr_vla_preproc_create", C.c_int,
     [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
      C.POINTER(C.c_float), C.POINTER(C.c_void_p)]),
    ("blurr_vla_preproc_destroy", None, [C.c_void_p]),
    ("blurr_vla_preproc_frame", C.c_int,
     [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    ("blurr_vla_preproc_build_coeffs", C.c_int,
     [C.c_int, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int]),
]
DECLARED_SYMBOLS = [s[0] for s in _SIGNATURES]

_lib: Optional[C.CDLL] = None


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load libblurr_pi0.so and bind every declared symbol. Raises if it is missing."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("BLURR_PI0_LIB", LIB_PATH)
    if not os.path.isfile(p):
        raise ImportError(
            f"{p} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; "
            "g.build()' or python <package>/build.py). The Pi-0 path has no CPU fallback."
        )
    lib = C.CDLL(p)
    lenient = bool(os.environ.get("BLURR_PI0_LIB_LENIENT"))      # tooling only: A/B against an older build
    for name, restype, argtypes in _SIGNATURES:
        if lenient and not hasattr(lib, name):
            continue
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.blurr_abi_version() != ABI_VERSION:
        raise ImportError(f"{p}: ABI version {lib.blurr_abi_version()} != {ABI_VERSION}; rebuild")
    if path is None:
        _lib = lib
    return lib


def check(status: int) -> int:
    if status < 0:
        msg = load_library().blurr_last_error()
        raise BlurrError(status, msg.decode("utf-8", "replace") if msg else "")
    return status
