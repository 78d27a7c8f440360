"""ctypes binding of libd2s_b200.so (C ABI declared in include/d2s.h).

The library is the product: if it cannot be loaded this module raises -- there is no CPU or PyTorch
fallback for any op in this package.
"""
import ctypes
import os
import threading

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libd2s_b200.so")

F32, BF16 = 0, 1
ORDER_INDEX_ASC, ORDER_SCORE_DESC = 0, 1
PROB_SOFTMAX, PROB_SIGMOID = 0, 1
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2

_p = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_i64 = ctypes.c_int64
_u64 = ctypes.c_uint64

# name -> argtypes; every entry point returns int (0 == ok).  Keep in sync with include/d2s.h.
SIGNATURES = {
    "d2s_select_topk_f32": [_p, _i, _i, _i, _i, _p, _p, _p],
    "d2s_threshold_select_f32": [_p, _i, _i, _f, _p, _p, _p, _p],
    "d2s_score_tail_a": [_p, _i, _i, _i, _i, _p, _p, _i, _p, _p, _p, _p, _p, _p, _i, _p, _p],
    "d2s_score_tail_b": [_p, _i, _i, _i, _i, _p, _p, _f, _p, _p, _i, _i, _p, _p, _p, _p, _p],
    "d2s_gumbel_decision_f32": [_p, _p, _p, _i64, _p, _p, _p],
    "d2s_gumbel_decision_bwd_f32": [_p, _p, _p, _p, _i64, _p, _p, _p],
    "d2s_gather_tokens": [_p, _i, _i, _i, _i, _p, _i, _i, _p, _p],
    "d2s_scatter_tokens_bwd": [_p, _i, _i, _i, _i, _p, _i, _i, _p, _p],
    "d2s_ptopk_fwd": [_p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_ptopk_fwd_rng": [_p, _u64, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_ptopk_bwd": [_p, _p, _i, _i, _i, _p, _p],
    "d2s_softmax_policy_fwd": [_p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_softmax_policy_bwd": [_p, _p, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_colsum_bf16": [_p, ctypes.c_longlong, _i, _p, _p],
    "d2s_gelu_bwd_colsum_bf16": [_p, _p, ctypes.c_longlong, _i, _p, _p, _p],
    "d2s_colsum_acc_bf16": [_p, ctypes.c_longlong, _i, _p, _p],
    "d2s_gelu_bwd_colsum_acc_bf16": [_p, _p, ctypes.c_longlong, _i, _p, _p, _p],
    "d2s_token_kl_fwd": [_p, _i, ctypes.c_longlong, _p, _i, ctypes.c_longlong, _i, _i, _i, _p, _p, _p],
    "d2s_adamw_flat_f32": [_p, _p, _p, _p, _p, ctypes.c_longlong, ctypes.c_longlong, _p, _p, _f, _f, _f, _f, _f, _p],
    "d2s_attn_policy_fwd": [_p, _p, _i, _i, _i, _i, _i, _f, _f, _p, _p, _p, _p],
    "d2s_attn_policy_bwd": [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_pool_act": [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p],
    "d2s_bias_act": [_p, _p, _i, ctypes.c_longlong, _i, _i, _i, _p],
    "d2s_pool_concat_inplace": [_p, _i, _i, _i, _i, _p],
    "d2s_predictor_a_tail_bf16": [_p, _i, ctypes.c_longlong, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p],
    "d2s_pool_strided_bf16": [_p, _p, _i, _i, _i, ctypes.c_longlong, _i, _p, _p],
    "d2s_pool_concat_fwd": [_p, _p, _i, _i, _i, _i, _p, _p, _p, _p],
    "d2s_pool_concat_bwd": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p],
    "d2s_assemble_tokens": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "d2s_patchify": [_p, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    "d2s_patchify_u8": [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p],
    "d2s_layernorm_fwd": [_p, _i, _p, _p, ctypes.c_longlong, _i, _f, _p, _i, _p, _p],
    "d2s_layernorm_bwd": [_p, _i, _p, _i, _p, _p, ctypes.c_longlong, _i, _p, _p, _p, _p],
    "d2s_layernorm_seg_fwd": [_p, _i, _p, _p, ctypes.c_longlong, _i, _i, _i, _f, _p, _i, _p, _p],
    "d2s_layernorm_seg_bwd": [_p, _i, _p, _i, _p, _p, ctypes.c_longlong, _i, _i, _i, _p, _p, _p, _p],
    "d2s_add_layernorm_fwd": [_p, _p, _i, _p, _p, ctypes.c_longlong, _i, _f, _p, _p, _i, _p, _p],
    "d2s_add_layernorm_bwd": [_p, _i, _p, _i, _p, _p, _p, ctypes.c_longlong, _i, _p, _p, _p, _p],
    "d2s_linear_act_pair_bf16": [_p, _p, _p, _i, _i, _i, _i, _p, _p, _p],
    "d2s_linear_lnin_act_pair_bf16": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p],
    "d2s_linear_residual_ln_bf16": [_p, _p, _p, _p, _p, _p, _f, _i, _i, _i, _p, _p, _p],
    "d2s_linear_residual_stats_bf16": [_p, _p, _p, _p, _f, _i, _i, _i, _p, _p, _p],
    "d2s_gather_layernorm": [_p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_assemble_layernorm": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_gather_layernorm_stats": [_p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_assemble_layernorm_stats": [_p, _p, _p, _i, _i, _i, _f, _p, _p, _p],
    "d2s_apply_layernorm_stats_bf16": [_p, _p, _p, _p, _i, _i, ctypes.c_longlong, ctypes.c_longlong, _p, _p],
    "d2s_mlp_residual_ln_bf16": [_p, _p, _p, _p, _p, _p, _p, _p, _f, _i, _i, _i, _i, _i, _p, _p, _p],
    "d2s_mlp_lnin_residual_ln_bf16": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _f, _i, _i, _i, _i, _i, _p, _p, _p, _p],
    "d2s_add_layernorm": [_p, _p, _p, _p, _i, _i, _i, _i, ctypes.c_longlong, ctypes.c_longlong, _f, _i, _p, _p, _p],
    "d2s_threshold_select_varlen_f32": [_p, _p, _i, _i, _f, _p, _p, _p, _p],
    "d2s_score_tail_b_varlen": [_p, _p, _i, _i, _i, _i, _p, _p, _f, _p, _p, _i, _p, _p, _p],
    "d2s_pool_concat_varlen_inplace": [_p, _p, _i, _i, _i, _i, _p],
    "d2s_attn_varlen_fwd": [_p, _p, _i, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_attn_long_fwd": [_p, _p, _p, _i, _i, _i, _i, _f, _f, _p, _p, _p],
    "d2s_attn_long_fwd_stats": [_p, _p, _i, _i, _i, _i, _f, _f, _p, _p, _p, _p],
    "d2s_attn_long_bwd": [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p, _p],
    "d2s_gather_layernorm_varlen": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p, _p, _p],
    "d2s_gather_layernorm_stats_varlen": [_p, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
}
INFO_SYMBOLS = ["d2s_last_error", "d2s_version", "d2s_launch_count"]
ALL_SYMBOLS = sorted(list(SIGNATURES) + INFO_SYMBOLS)

_lock = threading.Lock()
_lib = None


def load(build_if_missing=True):
    """Load (building in-tree with nvcc first if the .so is absent).  Raises RuntimeError on failure."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            if not build_if_missing:
                raise RuntimeError(f"{LIB_PATH} is missing: run `python dense2sparse-vit_b200/build.py`")
            import importlib.util
            spec = importlib.util.spec_from_file_location("_d2s_build", os.path.join(PKG_DIR, "build.py"))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            mod.build()
        try:
            lib = ctypes.CDLL(LIB_PATH)
        except OSError as e:  # no fallback: the CUDA extension IS the implementation
            raise RuntimeError(f"cannot load {LIB_PATH}: {e}") from e
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = ctypes.c_int
        lib.d2s_last_error.restype = ctypes.c_char_p
        lib.d2s_last_error.argtypes = []
        lib.d2s_version.restype = ctypes.c_int
        lib.d2s_launch_count.restype = ctypes.c_uint64
        _lib = lib
        return lib


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.d2s_last_error().decode(errors="replace")
        raise RuntimeError(f"{name} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().d2s_launch_count())
