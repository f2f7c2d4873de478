"""ctypes binding of libmrd_b200.so (the C ABI declared in include/mrd_b200.h).

There is no fallback: if the shared library is missing or a call fails, a Python exception is
raised.  The library is built in-tree by build.py (nvcc, sm_100a) and shipped with the snapshot.
"""

from __future__ import annotations

import ctypes as C
import os
import threading

from . import build as _build

ACT_NONE, ACT_RELU, ACT_GELU = 0, 1, 2
DT_I64, DT_I32, DT_F32, DT_U8, DT_BF16 = 0, 1, 2, 3, 4
ABI_VERSION = 1


class MrdError(RuntimeError):
    """A libmrd_b200 call returned a non-zero status."""


_lock = threading.Lock()
_lib = None

_vp, _i, _ll, _f, _d = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_double

# name -> (restype, argtypes); every symbol include/mrd_b200.h declares
SIGNATURES = {
    "mrd_last_error": (C.c_char_p, []),
    "mrd_abi_version": (_i, []),
    "mrd_ctx_create": (_i, [C.POINTER(_vp)]),
    "mrd_ctx_destroy": (_i, [_vp]),
    "mrd_ctx_configure": (_i, [_vp, _i, _i]),
    "mrd_ctx_set_option": (_i, [_vp, C.c_char_p, _d]),
    "mrd_ctx_load_weights": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_vp), C.POINTER(_ll), _vp]),
    "mrd_cnn_encoder_fwd": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mrd_text_encoder_fwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mrd_text_encoder_fwd_ex": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "mrd_fusion_fwd": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "mrd_head_fwd": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "mrd_fusion_head_fwd": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "mrd_multimodal_fwd": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _vp]),
    "mrd_ctx_profile": (_i, [_vp, _i]),
    "mrd_ctx_profile_report": (_i, [_vp, C.c_char_p, _i]),
    "mrd_ctx_launch_count": (_ll, [_vp]),
    "mrd_ctx_device_bytes": (_ll, [_vp]),
    "mrd_gemm_bf16": (_i, [_vp, _ll, _i, _i, _vp, _i, _vp, _vp, _ll, _vp, _ll, _vp, _ll, _i, _vp]),
    "mrd_gemm_ln_bf16": (_i, [_vp, _ll, _i, _i, _vp, _i, _vp, _vp, _ll, _vp, _ll, _vp, _vp, _f, _vp, _vp]),
    "mrd_gemm_ln_ws_bytes": (_ll, [_i]),
    "mrd_gemm_splitk_f32": (_i, [_vp, _ll, _i, _i, _vp, _i, _vp, _ll, _vp, _vp]),
    "mrd_conv2d_nhwc_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _i, _vp]),
    "mrd_conv1x1_dual_bf16": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp, _i, _vp]),
    "mrd_conv_chain_bf16": (_i, [_vp, _i, _vp, _i, _i, _vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _i, _vp]),
    "mrd_conv3x3_flat_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _i, _vp]),
    "mrd_stem_conv_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "mrd_stem_pool_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "mrd_repack_images": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "mrd_maxpool3x3s2": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "mrd_global_avgpool": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
    "mrd_layernorm_residual": (_i, [_vp, _ll, _vp, _ll, _vp, _vp, _f, _i, _i, _vp, _ll, _vp, _ll, _vp]),
    "mrd_bert_embed_layernorm": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp]),
    "mrd_attention_bf16": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "mrd_attention_probs_bf16": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "mrd_mask_to_bias": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "mrd_compact_tokens": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mrd_attention_varlen_bf16": (_i, [_vp, _vp, _vp, _i, _i, _i, _ll, _vp, _vp]),
    "mrd_attention_use_tcgen05": (_i, [_i]),
    "mrd_train_forward": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, C.c_ulonglong, _vp, _vp]),
    "mrd_train_backward": (_i, [_vp, _vp, _i, C.POINTER(C.c_char_p), C.POINTER(_vp), _vp]),
    "mrd_train_forward_ex": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, C.c_ulonglong, _vp, _vp, _vp, _vp, _vp,
                                  _vp]),
    "mrd_train_backward_ex": (_i, [_vp, _vp, _i, C.POINTER(C.c_char_p), C.POINTER(_vp), _vp, _vp]),
    "mrd_train_backward_begin": (_i, [_vp, _vp, _i, C.POINTER(C.c_char_p), C.POINTER(_vp), _vp]),
    "mrd_train_backward_stages": (_i, [_vp, _i, _i, _vp]),
    "mrd_train_backward_num_stages": (_i, [_vp]),
    "mrd_train_forward_dg": (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, C.c_ulonglong, _vp, _vp, _vp, _vp, _vp,
                                  _vp]),
    "mrd_train_backward_dg": (_i, [_vp, _vp, _i, C.POINTER(C.c_char_p), C.POINTER(_vp), _vp, _vp, _i, _vp, _vp, _vp]),
    "mrd_conv_dgrad_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _ll, _i, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "mrd_relu_mask_bf16": (_i, [_vp, _vp, _ll, _vp, _vp]),
    "mrd_maxpool3x3s2_bwd_bf16": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "mrd_pack_stem_dgrad": (_i, [_vp, _vp, _vp, _f, _vp, _vp]),
    "mrd_stem_dgrad_f32": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "mrd_dropout_mask": (_i, [C.c_ulonglong, C.c_uint, _d, _ll, _vp, _vp]),
    "mrd_attention_train_bf16": (_i, [_vp, _vp, _i, _i, _i, C.c_ulonglong, C.c_uint, _d, _vp, _vp]),
    "mrd_attention_train_varlen_bf16": (_i, [_vp, _vp, _vp, _i, _i, _i, _ll, C.c_ulonglong, C.c_uint, _d, _vp, _vp]),
    "mrd_attention_bwd_bf16": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, C.c_ulonglong, C.c_uint, _d, _vp, _vp,
                                    _ll, _vp]),
    "mrd_adamw_step": (_i, [_vp, _i, _vp, _vp, _i, _i, _f, _f, _f, _ll, _f, _vp, _vp]),
    "mrd_layernorm_bwd_bf16": (_i, [_vp, _vp, _vp, _f, _i, _i, _vp, _vp, _vp, _vp]),
    "mrd_dropout_bf16": (_i, [_vp, _ll, _i, _i, _vp, C.c_ulonglong, C.c_uint, _d, _vp, _ll, _vp]),
    "mrd_dropout_f32": (_i, [_vp, _i, _i, C.c_ulonglong, C.c_uint, _d, _vp, _vp]),
    "mrd_relu_dropout_f32": (_i, [_vp, _i, _i, C.c_ulonglong, C.c_uint, _d, _vp, _vp]),
    "mrd_head_dropout_f32": (_i, [_vp, _i, _i, _i, C.c_ulonglong, C.c_uint, _d, _vp, _vp, _vp]),
    "mrd_drop_add_layernorm_bf16": (_i, [_vp, _vp, _i, _i, _vp, C.c_ulonglong, C.c_uint, _d, _vp, _vp, _f, _vp, _vp, _vp]),
    "mrd_layernorm_f32": (_i, [_vp, _ll, _vp, _vp, _f, _i, _i, _vp, _ll, _vp]),
    "mrd_layernorm_bwd_f32": (_i, [_vp, _ll, _vp, _ll, _vp, _f, _i, _i, _vp, _ll, _vp, _vp, _vp]),
    "mrd_gelu_fwd_bf16": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "mrd_gelu_bwd_bf16": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "mrd_transpose_pad2_bf16": (_i, [_vp, _ll, _i, _vp, _vp, _ll, _i, _vp, _i, _vp, _i, _vp, _vp]),
    "mrd_colsum_bf16": (_i, [_vp, _ll, _i, _i, _vp, _f, _vp, _vp]),
    "mrd_colsum_f32": (_i, [_vp, _ll, _i, _i, _vp, _vp]),
    "mrd_relu_bwd_f32": (_i, [_vp, _vp, _ll, _vp, _vp]),
    "mrd_scatter_cls_rows_bf16": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "mrd_gather_cls_rows_f32": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "mrd_embed_layernorm_bwd": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _vp, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _vp]),
    "mrd_bn_stats_bf16": (_i, [_vp, _ll, _i, _vp, _vp, _vp, _vp]),
    "mrd_bn_apply_stats_bf16": (_i, [_vp, _ll, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _i, _vp]),
    "mrd_bn_update_running": (_i, [_vp, _i, _i, _f, _vp]),
}


def library_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if the sources changed and nvcc is available) and type the library."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        if build_if_missing and os.environ.get("MRD_B200_NO_BUILD") != "1":
            path = _build.build()
        if not os.path.exists(path):
            raise MrdError(
                f"{path} not found: the CUDA extension is not built (run `python -m __graft_entry__` "
                "or multimodal-rare-disease_b200/build.py); there is no CPU fallback")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        if lib.mrd_abi_version() != ABI_VERSION:
            raise MrdError(f"libmrd_b200 ABI {lib.mrd_abi_version()} != binding {ABI_VERSION}")
        _lib = lib
        return lib


def check(rc: int, what: str = "libmrd_b200") -> None:
    if rc != 0:
        msg = load().mrd_last_error()
        raise MrdError(f"{what} failed ({rc}): {msg.decode(errors='replace') if msg else ''}")
