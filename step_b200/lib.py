"""ctypes binding of libstep_b200.so (the C ABI in include/step_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libstep_b200.so")

f32p = C.c_void_p          # device pointers travel as integers
vp = C.c_void_p
ll = C.c_longlong
ull = C.c_ulonglong


class TsLayerWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "lin1_w", "lin1_b", "lin2_w", "lin2_b",
        "norm1_w", "norm1_b", "norm2_w", "norm2_b")]


class TsLayerImages(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("in_proj", "out_proj", "lin1", "lin2", "fused")]


class GwLayerParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "filter_w", "filter_b", "gate_w", "gate_b", "skip_w", "skip_b", "mlp_w", "mlp_b", "bn_w", "bn_b")]


class GwLayerGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "filter_w", "filter_b", "gate_w", "gate_b", "skip_w", "skip_b", "mlp_w", "mlp_b", "bn_w", "bn_b")]


# name -> (restype, argtypes); must list every symbol include/step_b200.h declares
SIGNATURES = {
    "step_abi_version": (C.c_int, []),
    "step_set_device": (C.c_int, [C.c_int]),
    "step_last_error_string": (C.c_char_p, []),
    "step_launch_count": (C.c_ulonglong, []),
    "step_ts_embed_fwd": (C.c_int, [f32p, ll, ll, ll, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p, f32p, C.c_float, ull, vp]),
    "step_linear_f32": (C.c_int, [f32p, f32p, f32p, f32p, ll, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p, C.c_float, ull,
                                  C.c_uint, vp]),
    "step_attn_fwd_f32": (C.c_int, [f32p, f32p, C.c_int, C.c_int, C.c_float, ull, C.c_uint, vp]),
    "step_layernorm96_f32": (C.c_int, [f32p, f32p, f32p, f32p, ll, vp]),
    "step_attn_bwd_f32": (C.c_int, [f32p, f32p, f32p, C.c_int, C.c_int, C.c_float, ull, C.c_uint, f32p, f32p, vp]),
    "step_add_layernorm96_fwd": (C.c_int, [f32p, f32p, f32p, f32p, ll, f32p, f32p, f32p, vp]),
    "step_add_layernorm96_bwd": (C.c_int, [f32p, f32p, f32p, f32p, ll, f32p, f32p, f32p, vp]),
    "step_dropout_f32": (C.c_int, [f32p, ll, C.c_float, ull, C.c_uint, f32p, vp]),
    "step_ts_encoder_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "step_ts_encoder_fwd": (C.c_int, [f32p, ll, ll, ll, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p,
                                      C.POINTER(TsLayerWeights), C.c_int, f32p, f32p, f32p, vp, C.c_size_t, C.c_int,
                                      C.c_float, ull, vp]),
    "step_ts_layers_fwd": (C.c_int, [f32p, C.c_int, C.c_int, C.POINTER(TsLayerWeights), C.c_int, f32p, f32p, vp, C.c_size_t,
                                     C.c_float, ull, vp]),
    "step_tc_pack_weight": (C.c_int, [f32p, C.c_int, C.c_int, vp, vp]),
    "step_tc_rows_to_image": (C.c_int, [f32p, ll, C.c_int, vp, vp]),
    "step_tc_image_to_rows": (C.c_int, [vp, ll, C.c_int, f32p, vp]),
    "step_tc_linear": (C.c_int, [vp, vp, f32p, ll, C.c_int, C.c_int, C.c_int, vp, f32p, f32p, vp, f32p, vp]),
    "step_tc_embed_fwd": (C.c_int, [f32p, ll, ll, ll, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p, vp, C.c_float, ull, vp]),
    "step_gwnet_dropout_probe": (C.c_int, [f32p, ll, C.c_float, ull, C.c_int, f32p, vp]),
    "step_tc_linear_drop": (C.c_int, [vp, vp, f32p, ll, C.c_int, C.c_int, C.c_int, vp, f32p, f32p, vp, f32p, C.c_float, ull, vp]),
    "step_tc_attn_image_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "step_tc_attn_drop_threshold": (C.c_uint, [C.c_float]),
    "step_tc_qkv": (C.c_int, [vp, vp, f32p, C.c_int, C.c_int, vp, vp, vp, f32p, vp]),
    "step_tc_attention": (C.c_int, [vp, vp, vp, vp, f32p, C.c_int, C.c_int, C.c_float, ull, vp]),
    "step_tc_attn_train_lse_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "step_tc_attn_train_pack": (C.c_int, [f32p, C.c_int, C.c_int, vp, vp, vp, f32p, vp]),
    "step_tc_attn_train_fwd": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_float, ull, f32p, f32p, vp]),
    "step_tc_attn_train_bwd": (C.c_int, [vp, vp, vp, f32p, f32p, f32p, C.c_int, C.c_int, C.c_float, ull, f32p, vp]),
    "step_tc_attn_train_keep_mask": (C.c_int, [C.c_int, C.c_int, C.c_float, ull, vp, vp]),
    "step_ts_encoder_bf16_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "step_ts_encoder_fwd_bf16": (C.c_int, [f32p, ll, ll, ll, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p,
                                           C.POINTER(TsLayerWeights), C.POINTER(TsLayerImages), C.c_int, f32p, f32p, f32p, vp, vp,
                                           C.c_size_t, C.c_float, ull, vp]),
    "step_tc_seq_image_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "step_tc_hidden_to_seq_image": (C.c_int, [f32p, C.c_int, C.c_int, C.c_int, vp, vp]),
    "step_tc_cosine_gram": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, f32p, f32p, vp]),
    "step_tc_gram_rows": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32p, vp]),
    "step_gram_normalize": (C.c_int, [f32p, C.c_int, C.c_int, f32p, vp]),
    "step_cosine_gram_f32": (C.c_int, [f32p, C.c_int, C.c_int, ll, f32p, f32p, vp]),
    "step_topk_mask_f32": (C.c_int, [f32p, C.c_int, C.c_int, C.c_int, f32p, vp]),
    "step_edge_logits_fwd": (C.c_int, [f32p, f32p, f32p, f32p, C.c_int, C.c_int, f32p, f32p, vp]),
    "step_edge_logits_bwd": (C.c_int, [f32p, f32p, f32p, f32p, C.c_int, C.c_int, f32p, f32p, f32p, f32p, vp]),
    "step_gumbel_sample_fwd": (C.c_int, [f32p, f32p, C.c_int, C.c_int, C.c_float, ull, f32p, f32p, vp]),
    "step_gumbel_sample_bwd": (C.c_int, [f32p, f32p, C.c_int, C.c_int, C.c_float, C.c_int, f32p, vp]),
    "step_loss_fwd_bwd": (C.c_int, [f32p, f32p, ll, C.c_float, C.c_float, C.c_float, C.c_int, f32p, f32p, C.c_int, C.c_int,
                                    C.c_float, f32p, f32p, f32p, vp, vp]),
    "step_dgl_conv_fwd": (C.c_int, [f32p, C.c_int, C.c_int] + [f32p] * 8 + [C.c_float, C.c_int, f32p, f32p, f32p, f32p, vp, vp]),
    "step_dgl_conv_bwd": (C.c_int, [f32p, f32p, C.c_int, C.c_int] + [f32p] * 5 + [C.c_float] + [f32p] * 12 + [vp, vp]),
    "step_dgl_fc_splits": (C.c_int, [C.c_int, ll, ll]),
    "step_dgl_fc_fwd": (C.c_int, [f32p, f32p, C.c_int, ll, ll, ll, f32p, f32p, vp]),
    "step_dgl_fc_bn_fwd": (C.c_int, [f32p, f32p, f32p, f32p, C.c_int, C.c_float, C.c_int, f32p, f32p, vp]),
    "step_dgl_fc_bn_bwd": (C.c_int, [f32p, f32p, f32p, f32p, C.c_int, f32p, f32p, f32p, f32p, vp]),
    "step_dgl_fc_bwd": (C.c_int, [f32p, f32p, f32p, C.c_int, ll, ll, ll, C.c_float, f32p, f32p, vp]),
    "step_gemm_f32": (C.c_int, [f32p, ll, C.c_int, f32p, ll, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, f32p, C.c_int, f32p, ll,
                                f32p, C.c_int, C.c_int, f32p, ll, vp]),
    "step_colsum_f32": (C.c_int, [f32p, ll, C.c_int, ll, f32p, vp]),
    "step_relu_bwd_f32": (C.c_int, [f32p, f32p, ll, f32p, vp]),
    "step_gw_start_fwd": (C.c_int, [f32p, C.c_int, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p, vp]),
    "step_gw_start_bwd": (C.c_int, [f32p, C.c_int, C.c_int, C.c_int, C.c_int, f32p, f32p, vp]),
    "step_gw_supports_fwd": (C.c_int, [f32p, C.c_int, C.c_int, f32p, f32p, f32p, vp]),
    "step_gw_supports_bwd": (C.c_int, [f32p, f32p, f32p, f32p, f32p, C.c_int, C.c_int, f32p, f32p, vp]),
    "step_gw_adp_fwd": (C.c_int, [f32p, f32p, C.c_int, C.c_int, f32p, vp]),
    "step_gw_adp_bwd": (C.c_int, [f32p, f32p, f32p, f32p, C.c_int, C.c_int, f32p, f32p, f32p, vp]),
    "step_opt_chunk_elems": (C.c_int, []),
    "step_clip_adam_step": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, vp, vp, f32p, f32p, vp, C.c_float, C.c_float, C.c_float,
                                      C.c_float, C.c_float, C.c_float, f32p, vp]),
    "step_metrics_accumulate": (C.c_int, [f32p, f32p, ll, C.c_float, C.c_float, C.c_float, C.c_int, vp, vp, vp]),
    "step_gwnet_stash_floats": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "step_gwnet_stack_fwd": (C.c_int, [f32p, f32p, f32p, f32p, C.POINTER(GwLayerParams), C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_float, ull, f32p, f32p, f32p, vp]),
    "step_gwnet_stack_bwd": (C.c_int, [f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, C.POINTER(GwLayerParams),
                                       C.POINTER(GwLayerGrads), C.c_int, C.c_int, C.c_int, C.c_float, ull, f32p, f32p,
                                       f32p, f32p, f32p, f32p, vp]),
}

ABI_VERSION = 3
_lib = None
_lock = threading.Lock()


class StepB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built - there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise StepB200Error(
                f"{LIB_PATH} is missing. Build it with `python -m step_b200.build` (needs nvcc). "
                "step_b200 has no CPU or PyTorch fallback path.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        got = lib.step_abi_version()
        if got != ABI_VERSION:
            raise StepB200Error(f"libstep_b200.so ABI version {got}, binding expects {ABI_VERSION}")
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().step_last_error_string().decode("utf-8", "replace")
        kind = "CUDA error" if rc > 0 else "bad argument"
        raise StepB200Error(f"{what} failed ({kind} {rc}): {msg}")
