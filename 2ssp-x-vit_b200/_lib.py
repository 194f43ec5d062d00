"""ctypes binding of libtssp_b200.so (C ABI declared in include/tssp.h).

The library is the product: if it is missing or a call fails, this module raises -- there is no
PyTorch/CPU fallback for any compute step.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

TSSP_MAX_BLOCKS = 64
TSSP_ABI_VERSION = 2

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = _PKG_DIR / "lib" / "libtssp_b200.so"

# weight table layout (include/tssp.h: enum tssp_weight_index / tssp_block_weight_index)
(W_PATCH_W, W_PATCH_B, W_CLS, W_POS, W_FINAL_LN_W, W_FINAL_LN_B, W_HEAD0_W, W_HEAD_W, W_HEAD_B,
 W_DIST_TOKEN, W_HEAD_DIST_W, W_HEAD_DIST_B, W_REG_TOKENS, W_NORM_PRE_W, W_NORM_PRE_B, W_GLOBAL_COUNT) = range(16)
(BW_LN1_W, BW_LN1_B, BW_Q_W, BW_Q_B, BW_K_W, BW_K_B, BW_V_W, BW_V_B, BW_PROJ_W, BW_PROJ_B,
 BW_LN2_W, BW_LN2_B, BW_FC1_W, BW_FC1_B, BW_FC2_W, BW_FC2_B, BW_LS1, BW_LS2, BW_COUNT) = range(19)
TSSP_MAX_REGISTER_TOKENS = 7

# GEMM epilogue modes (csrc/gemm_tcgen05.cuh: enum GemmMode)
(EPI_BF16, EPI_BF16_GELU, EPI_BF16_GELU_SCORE, EPI_BF16_GELU_SCORE_PRE, EPI_F32, EPI_BF16_ROWNORM, EPI_F32_SCALED,
 EPI_BF16_QGELU, EPI_BF16_QGELU_SCORE_PRE) = range(9)
# MLP activations of tssp_config_t.ffn_act
FFN_ACTS = {"gelu": 0, "quick_gelu": 1}


PROFILE_CLASSES = ["fc1_gelu_score", "qkv", "proj", "fc2", "patch_embed", "head", "attention", "layernorm", "score_finish", "misc"]


class TsspConfig(C.Structure):
    _fields_ = [
        ("n_blocks", C.c_int32),
        ("hidden", C.c_int32),
        ("heads", C.c_int32),
        ("image_size", C.c_int32),
        ("patch_size", C.c_int32),
        ("channels", C.c_int32),
        ("n_classes", C.c_int32),
        ("head_hidden", C.c_int32),
        ("max_images", C.c_int32),
        ("score_point", C.c_int32),
        ("cache_blocks", C.c_int32),
        ("ln_eps", C.c_float),
        ("dist_token", C.c_int32),
        ("register_tokens", C.c_int32),
        ("pos_patches_only", C.c_int32),
        ("layer_scale", C.c_int32),
        ("pre_norm", C.c_int32),
        ("ffn_act", C.c_int32),
        ("ffn_dims", C.c_int32 * TSSP_MAX_BLOCKS),
        ("attn_present", C.c_int32 * TSSP_MAX_BLOCKS),
    ]


# pixel formats of tssp_pixel_input_t.format
PIXELS_F32, PIXELS_U8 = 0, 1
TSSP_MAX_PIXEL_CHANNELS = 4


class TsspPixelInput(C.Structure):
    _fields_ = [
        ("format", C.c_int32),
        ("rescale", C.c_float),
        ("mean", C.c_float * TSSP_MAX_PIXEL_CHANNELS),
        ("std", C.c_float * TSSP_MAX_PIXEL_CHANNELS),
    ]


def pixel_input(fmt: int, mean=(), std=(), rescale: float = 1.0) -> TsspPixelInput:
    """A tssp_pixel_input_t; mean / std hold one value per channel (at most four), the rest stay 0 / 1."""
    out = TsspPixelInput()
    out.format, out.rescale = fmt, rescale
    for c in range(TSSP_MAX_PIXEL_CHANNELS):
        out.mean[c] = mean[c] if c < len(mean) else 0.0
        out.std[c] = std[c] if c < len(std) else 1.0
    return out


class TsspError(RuntimeError):
    """A call into libtssp_b200.so failed; the message comes from tssp_last_error()."""


_P = C.c_void_p
_I = C.c_int
_I64 = C.c_int64

# name -> (restype, argtypes); every symbol include/tssp.h declares
SIGNATURES = {
    "tssp_abi_version": (_I, []),
    "tssp_last_error": (C.c_char_p, []),
    "tssp_create": (_I, [C.POINTER(TsspConfig), _I, C.POINTER(_P)]),
    "tssp_destroy": (_I, [_P]),
    "tssp_trim_pool": (_I, []),
    "tssp_load_weights": (_I, [_P, C.POINTER(_P), _I, _P]),
    "tssp_update_ffn": (_I, [_P, _I, _I, _P, _P, _P, _P]),
    "tssp_set_attention": (_I, [_P, C.POINTER(C.c_int32)]),
    "tssp_set_pixel_input": (_I, [_P, C.POINTER(TsspPixelInput)]),
    "tssp_s1_reset": (_I, [_P, _P]),
    "tssp_s1_batch": (_I, [_P, _P, _I, _I, _P, _P]),
    "tssp_s1_scores": (_I, [_P, _P, _I, _P]),
    "tssp_forward_logits": (_I, [_P, _P, _I, _I, C.POINTER(C.c_int32), _P, _I, _P]),
    "tssp_eval_batch": (_I, [_P, _P, _P, _I, _I, C.POINTER(C.c_int32), _P, _P]),
    "tssp_s2_reset": (_I, [_P, _P]),
    "tssp_s2_batch": (_I, [_P, _P, _P, _I, _I, C.POINTER(C.c_int32), _I, _P]),
    "tssp_s2_counts": (_I, [_P, C.POINTER(_I64), _P]),
    "tssp_ffn_gather": (_I, [_P, _P, _P, _I, _I, _P, _I, _P, _P, _P, _P]),
    "tssp_ffn_gather_batch": (_I, [_I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_int32), _I, C.POINTER(_P),
                                   C.POINTER(C.c_int32), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), _P]),
    "tssp_op_gemm": (_I, [_I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _P, _P, _I, _I, _I, _P]),
    "tssp_op_gemm_scaled": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P, _P, _I, _P]),
    "tssp_op_gemm_rownorm": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P, _P, _I, _I, _P]),
    "tssp_op_score_finish": (_I, [_P, _I, _P, _I, _I, _I, _I, _P, _P]),
    "tssp_op_layernorm": (_I, [_P, _I64, _P, _P, _P, _I, _I, C.c_float, _P]),
    "tssp_op_layernorm_f32": (_I, [_P, _I64, _P, _P, _P, _I64, _I, _I, C.c_float, _P]),
    "tssp_op_attention": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "tssp_op_im2col": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, C.POINTER(TsspPixelInput), _P]),
    "tssp_op_cast_bf16": (_I, [_P, _I, _I, _I, _P, _I, _I, _I, _P]),
    "tssp_op_argmax_count": (_I, [_P, _I, _I, _I, _P, _P, _P, _P]),
    "tssp_op_stable_rank_f64": (_I, [_P, _I, _I, _I, _P, _P]),
    "tssp_mask_consensus_prepare": (_I, [_P, _I, _I, _P, _I, _I, _P, _P, _P, _P]),
    "tssp_mask_count_less": (_I, [_P, _I, _P, _I, _P, _P, _P]),
    "tssp_mask_consensus_select": (_I, [_P, _P, _I, _I, _P, _I, _I, _P, _I, _P, _P]),
    "tssp_mask_summation": (_I, [_P, _I, _I, _P, _I, _I, _I, _P, _P, _P, _P]),
    "tssp_op_minmax_normalize_f64": (_I, [_P, C.c_longlong, _P, _P, _P]),
    "tssp_format_ffn_scores": (C.c_longlong, [_P, C.POINTER(C.c_int32), _I, _P, C.c_longlong]),
    "tssp_debug_attention_trace": (_I, [_P]),
    "tssp_debug_gemm_trace": (_I, [_P]),
    "tssp_set_gemm_form": (_I, [_I]),
    "tssp_set_graphs": (_I, [_I]),
    "tssp_launch_count": (C.c_uint64, []),
    "tssp_graph_capture_count": (C.c_uint64, []),
    "tssp_profile_begin": (_I, []),
    "tssp_profile_end": (_I, [C.POINTER(C.c_double), C.POINTER(C.c_uint64), _I]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (once) and bind every prototype. Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("TSSP_B200_LIB", str(LIB_PATH))
    if not os.path.exists(path):
        raise TsspError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no fallback path."
        )
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.tssp_abi_version() != TSSP_ABI_VERSION:
        raise TsspError(f"ABI mismatch: library {lib.tssp_abi_version()} vs binding {TSSP_ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().tssp_last_error()
        raise TsspError(msg.decode("utf-8", "replace") if msg else f"libtssp_b200 call failed with status {rc}")


def ptr(t) -> C.c_void_p:
    """Device/host address of a torch tensor (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    return C.c_void_p(t.data_ptr())


def current_stream() -> C.c_void_p:
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
