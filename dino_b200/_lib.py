"""ctypes binding of libdinoseg.so (C ABI declared in include/dinoseg.h).

There is no fallback: if the shared object is missing or does not load, importing the
symbols raises.  The library itself refuses to create a handle on anything but sm_100.
"""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

_lib = None


class DinosegCfg(C.Structure):
    _fields_ = [
        ("embed_dim", C.c_int32), ("num_heads", C.c_int32), ("mlp_hidden", C.c_int32),
        ("n_blocks", C.c_int32), ("patch", C.c_int32), ("pos_grid", C.c_int32),
        ("n_classes", C.c_int32), ("head_h1", C.c_int32), ("head_h2", C.c_int32),
        ("head_kind", C.c_int32), ("ln_eps", C.c_float),
    ]


# name -> (restype, argtypes); must list every symbol of include/dinoseg.h
SIGNATURES = {
    "dinoseg_create": (C.c_int, [C.POINTER(DinosegCfg), C.c_int, C.POINTER(C.c_void_p)]),
    "dinoseg_destroy": (None, [C.c_void_p]),
    "dinoseg_last_error": (C.c_char_p, [C.c_void_p]),
    "dinoseg_set_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.c_void_p]),
    "dinoseg_missing_weights": (C.c_int, [C.c_void_p]),
    "dinoseg_set_resolution": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "dinoseg_set_resolution_hw": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "dinoseg_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int]),
    "dinoseg_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_size_t, C.c_void_p]),
    "dinoseg_predict_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dinoseg_forward_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                     C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                     C.c_void_p]),
    "dinoseg_predict_host_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                          C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_void_p]),
    "dinoseg_predict_host_submit": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dinoseg_predict_host_submit_u8": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                                   C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_void_p]),
    "dinoseg_predict_host_wait": (C.c_int, [C.c_void_p, C.c_int64]),
    "dinoseg_set_host_chunk": (C.c_int, [C.c_void_p, C.c_int]),
    "dinoseg_cls_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dinoseg_features": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                   C.c_void_p]),
    "dinoseg_features_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                      C.POINTER(C.c_float), C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dinoseg_embeddings": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
    "dinoseg_embeddings_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                        C.POINTER(C.c_float), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.c_void_p]),
    "dinoseg_argmax_replicate": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "dinoseg_copy_buffer": (C.c_int64, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dinoseg_set_debug_stop": (C.c_int, [C.c_void_p, C.c_int]),
    "dinoseg_last_launch_count": (C.c_int, [C.c_void_p]),
    "dinoseg_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "dinoseg_profile_set_mask": (C.c_int, [C.c_void_p, C.c_uint32]),
    "dinoseg_debug_pending_kinds": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]),
    "dinoseg_debug_heartbeat": (C.c_int, [C.POINTER(C.c_int), C.c_int]),
    "dinoseg_profile_num_kinds": (C.c_int, []),
    "dinoseg_profile_kind_name": (C.c_char_p, [C.c_int]),
    "dinoseg_profile_gaps": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "dinoseg_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int), C.c_int]),
    "dinoseg_op_gemm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "dinoseg_op_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dinoseg_debug_set_attn_timing": (C.c_int, [C.c_void_p]),
    "dinoseg_op_mlp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                 C.c_void_p]),
    "dinoseg_op_mlp_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                    C.c_int, C.c_void_p]),
    "dinoseg_op_fold_ln": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "dinoseg_op_mlp_ln": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                    C.c_int, C.c_void_p]),
    "dinoseg_op_gemm_pair": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "dinoseg_set_pair_kernels": (C.c_int, [C.c_void_p, C.c_int]),
    "dinoseg_debug_host_pool": (C.c_int, [C.c_int, C.c_int]),
    "dinoseg_debug_attn_redone": (C.c_int, []),
    "dinoseg_debug_attn_items": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "dinoseg_expand_labels_host": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dinoseg_get_pair_kernels": (C.c_int, [C.c_void_p]),
    "dinoseg_set_host_expand": (C.c_int, [C.c_void_p, C.c_int]),
    "dinoseg_get_host_expand": (C.c_int, [C.c_void_p]),
    "dinoseg_half_counts": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "dinoseg_set_fused_mlp": (C.c_int, [C.c_void_p, C.c_int]),
    "dinoseg_set_fused_head": (C.c_int, [C.c_void_p, C.c_int]),
    "dinoseg_op_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                       C.c_float, C.c_void_p]),
    "dinoseg_op_layernorm_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                           C.c_float, C.c_void_p]),
    "dinoseg_op_posembed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dinoseg_op_im2col": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "dinoseg_op_f32_to_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
}

EPI_BF16, EPI_GELU_BF16, EPI_RESID_F32, EPI_PATCH_F32, EPI_RELU_F32 = range(5)


def lib_path() -> str:
    return LIB_PATH


def load() -> C.CDLL:
    """Load libdinoseg.so (once) and declare the prototypes. Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("DINOSEG_LIB", LIB_PATH)    # measurement aid: another build of the SAME library (A/B runs)
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with `python -m dino_b200.build` "
            "(there is no CPU / PyTorch fallback for the DINOSeg hot path)")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error(handle=None) -> str:
    msg = load().dinoseg_last_error(handle)
    return msg.decode() if msg else ""
