"""ctypes binding of include/leaf_b200.h. There is no fallback: a missing library is an ImportError-grade
failure, and every entry point fails with LEAF_ERR_CUDA when no sm_100 device is present."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LEAF_B200_LIB") or os.path.join(HERE, "lib", "libleaf_b200.so")   # the override is for same-box A/B runs of two builds

c_int, c_void_p, c_float, c_i64 = ctypes.c_int32, ctypes.c_void_p, ctypes.c_float, ctypes.c_int64


class LeafCfg(ctypes.Structure):
    _fields_ = [("width", c_int), ("layers", c_int), ("heads", c_int), ("embed_dim", c_int), ("activation", c_int),
                ("ln_eps", c_float)]


class LeafLayerPtrs(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in (
        "ln1_w", "ln1_b", "in_proj_w", "in_proj_b", "q_w", "k_w", "v_w", "q_b", "k_b", "v_b", "out_w", "out_b",
        "ln2_w", "ln2_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


class LeafWeightPtrs(ctypes.Structure):
    _fields_ = [("token_embedding", c_void_p), ("positional_embedding", c_void_p), ("lnf_w", c_void_p),
                ("lnf_b", c_void_p), ("text_projection", c_void_p), ("projection_is_ew", c_int),
                ("layers", ctypes.POINTER(LeafLayerPtrs))]


# name -> (restype, argtypes); also the list tests check against the header
SIGNATURES = {
    "leaf_create": (c_int, [ctypes.POINTER(LeafCfg), ctypes.POINTER(c_void_p)]),
    "leaf_destroy": (c_int, [c_void_p]),
    "leaf_last_error": (ctypes.c_char_p, []),
    "leaf_version": (ctypes.c_char_p, []),
    "leaf_load_bpe": (c_int, [c_void_p, c_void_p, c_int]),
    "leaf_bind_weights": (c_int, [c_void_p, ctypes.POINTER(LeafWeightPtrs), c_void_p]),
    "leaf_refresh_weights": (c_int, [c_void_p, c_void_p]),
    "leaf_reserve": (c_int, [c_void_p, c_int]),
    "leaf_expand_tokenize": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "leaf_set_tokenizer_mode": (c_int, [c_void_p, c_int]),
    "leaf_set_max_caption_bytes": (c_int, [c_void_p, c_int]),
    "leaf_load_words": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int]),
    "leaf_constrain_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p]),
    "leaf_encode": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "leaf_score": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "leaf_topk": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "leaf_train_reserve": (c_int, [c_void_p, c_int]),
    "leaf_forward_train": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, ctypes.POINTER(c_i64), c_void_p]),
    "leaf_backward": (c_int, [c_void_p, c_i64, c_void_p, c_int, ctypes.POINTER(LeafWeightPtrs), c_void_p]),
    "leaf_set_backward_hook": (c_int, [c_void_p, c_void_p, c_void_p]),
    "leaf_set_sm_budget": (c_int, [c_void_p, c_int]),
    "leaf_set_deterministic": (c_int, [c_void_p, c_int]),
    "leaf_adamw": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_i64, ctypes.c_float, ctypes.c_float,
                           ctypes.c_float, ctypes.c_float, ctypes.c_float, c_int, ctypes.c_float, c_void_p]),
    "leaf_sumsq": (c_int, [c_void_p, c_void_p, c_i64, c_void_p, c_void_p]),
    "leaf_scale": (c_int, [c_void_p, c_void_p, c_i64, ctypes.c_float, c_void_p]),
    "leaf_gemm_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                               c_void_p, c_void_p]),
    "leaf_gemm_bf16_mn": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "leaf_test_layernorm": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "leaf_test_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "leaf_test_attention_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "leaf_set_prune_last": (c_int, [c_void_p, c_int]),
    "leaf_launch_count": (c_i64, [c_void_p, c_int]),
    "leaf_last_rows": (c_i64, [c_void_p]),
    "leaf_set_timing": (c_int, [c_void_p, c_int]),
    "leaf_timing_ms": (ctypes.c_double, [c_void_p, c_int, ctypes.POINTER(c_int)]),
}

BACKWARD_HOOK = ctypes.CFUNCTYPE(None, c_int, c_void_p)      # leaf_backward_hook_t

_lib = None


class LeafError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LeafError(f"{LIB_PATH} is missing: build it with `python -m leaf_b200.build` "
                            "(leaf_b200 has no CPU or PyTorch fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise LeafError(f"leaf_b200 error {rc}: {lib().leaf_last_error().decode('utf-8', 'replace')}")
