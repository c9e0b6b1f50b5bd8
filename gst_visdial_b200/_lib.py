"""ctypes binding of include/gstvd.h (the C ABI of libgstvd.so).

There is deliberately no fallback: if the shared library is missing or cannot be loaded the import of any
compute entry point raises, so a GPU box can never silently run a CPU / eager path.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libgstvd.so")

GSTVD_ABI_VERSION = 7
GSTVD_MAX_CONNECTIONS = 16
GSTVD_F32, GSTVD_BF16 = 0, 1
GSTVD_SELECT_SAMPLE, GSTVD_SELECT_BEAM, GSTVD_SELECT_BEAM_SAMPLE = 0, 1, 2
GSTVD_FLAG_NO_CUDA_GRAPH = 1
GSTVD_FLAG_DEBUG_SIMT_GEMM = 2
GSTVD_FLAG_GENERIC_ATTENTION = 4
GSTVD_FLAG_NO_PDL = 8
GSTVD_MAX_TOP_K = 16
# gstvd_gemm_kernel / gstvd_gemm_store
GEMM_KERNELS = {"simt": 0, "tc32": 1, "tc64": 2, "tc128": 3, "tc256": 4, "skinny32": 5, "skinny64": 6, "pair128": 7, "pair256": 8,
                "ln32": 9, "ln64": 10}
GEMM_STORES = {"generic": 0, "tma": 1, "direct": 2}

STATUS_NAMES = {0: "OK", -1: "INVALID", -2: "CUDA", -3: "UNSUPPORTED", -4: "STATE"}


class GstvdConfig(Structure):
    _fields_ = [
        ("abi_version", c_int32), ("compute_dtype", c_int32),
        ("vocab_size", c_int32), ("hidden_size", c_int32), ("num_hidden_layers", c_int32), ("num_attention_heads", c_int32),
        ("intermediate_size", c_int32), ("max_position_embeddings", c_int32), ("type_vocab_size", c_int32),
        ("v_feature_size", c_int32), ("v_hidden_size", c_int32), ("v_num_hidden_layers", c_int32),
        ("v_num_attention_heads", c_int32), ("v_intermediate_size", c_int32),
        ("bi_hidden_size", c_int32), ("bi_num_attention_heads", c_int32),
        ("num_connections", c_int32),
        ("v_biattention_id", c_int32 * GSTVD_MAX_CONNECTIONS), ("t_biattention_id", c_int32 * GSTVD_MAX_CONNECTIONS),
        ("dec_num_hidden_layers", c_int32), ("dec_num_attention_heads", c_int32), ("dec_intermediate_size", c_int32),
        ("max_batch", c_int32), ("max_text_len", c_int32), ("max_regions", c_int32), ("max_new_tokens", c_int32),
        ("max_beams", c_int32), ("max_dec_len", c_int32), ("flags", c_int32),
    ]


class GstvdGenParams(Structure):
    _fields_ = [
        ("mode", c_int32), ("num_beams", c_int32), ("max_new_tokens", c_int32), ("top_k", c_int32),
        ("temperature", c_float), ("top_p", c_float), ("ngram_blocking_size", c_int32), ("seed", c_uint64),
        ("row_offset", c_int64), ("num_return_sequences", c_int32), ("num_beam_groups", c_int32), ("diversity_penalty", c_float),
        ("repetition_penalty", c_float), ("no_repeat_ngram_size", c_int32), ("min_length", c_int32),
        ("length_penalty", c_float), ("early_stopping", c_int32), ("bad_words_ids", c_uint64), ("bad_words_len", c_int32),
    ]


class GstvdError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"gstvd error {STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


# every symbol include/gstvd.h declares: (name, restype, argtypes)
_P = c_void_p
SYMBOLS = [
    ("gstvd_abi_version", c_int, []),
    ("gstvd_create", c_int, [POINTER(GstvdConfig), c_int, POINTER(_P)]),
    ("gstvd_destroy", None, [_P]),
    ("gstvd_last_error", c_char_p, [_P]),
    ("gstvd_load_weight", c_int, [_P, c_char_p, _P, c_int64, _P]),
    ("gstvd_finalize_weights", c_int, [_P, _P]),
    ("gstvd_missing_weights", c_int, [_P]),
    ("gstvd_encode", c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    ("gstvd_prefill_cross", c_int, [_P, c_int, c_int, _P, _P, _P]),
    ("gstvd_generate", c_int, [_P, c_int, POINTER(GstvdGenParams), _P, c_int, _P, _P, c_int, _P, _P, _P]),
    ("gstvd_round", c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, POINTER(GstvdGenParams), _P, c_int, _P, _P, _P]),
    ("gstvd_score", c_int, [_P, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    ("gstvd_score_options", c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    ("gstvd_reorder_cache", c_int, [_P, c_int, c_int, c_int, _P, _P]),
    ("gstvd_splice", c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P, _P, c_int, c_int, _P, _P]),
    ("gstvd_op_linear", c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P, c_int64, c_int, POINTER(c_int32), c_int, c_int,
                                POINTER(c_int32), _P]),
    ("gstvd_op_linear_ln", c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, c_int, POINTER(c_int32),
                                   _P]),
    ("gstvd_op_add_layernorm", c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    ("gstvd_op_attention", c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, _P, c_float, c_int, _P, _P]),
    ("gstvd_op_deferred_ln_chain", c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    ("gstvd_op_dec_self_attn", c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    ("gstvd_op_dec_cross_attn", c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P, _P, _P]),
    ("gstvd_op_anc_update", c_int, [_P, c_int, c_int, c_int, c_int, _P, c_int, _P, _P, _P]),
    ("gstvd_debug_self_cache", c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    ("gstvd_debug_cross_cache", c_int, [_P, c_int, c_int, _P, _P]),
    ("gstvd_op_beam_begin", c_int, [_P, c_int, c_int, c_int, _P]),
    ("gstvd_op_beam_step", c_int, [_P, _P, c_int64, _P, _P, _P, _P]),
    ("gstvd_op_beam_end", c_int, [_P, _P, _P, _P]),
    ("gstvd_op_sample", c_int, [_P, c_int, _P, c_int64, POINTER(GstvdGenParams), _P, _P, c_int, _P, c_int, c_int, _P, _P]),
    ("gstvd_cross_key_counts", c_int, [_P, c_int, _P, _P]),
    ("gstvd_launch_count", c_int64, [_P]),
    ("gstvd_profile_gemm", c_int, [_P, c_int, c_int]),
    ("gstvd_profile_read", c_int, [_P, POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(c_int64)]),
]

_lib = None


def load():
    """Loads libgstvd.so (once) and declares the prototypes.  Raises if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"gst_visdial_b200: CUDA extension {LIB_PATH} is missing. Build it with `python -m gst_visdial_b200._build` "
            "(or __graft_entry__.build()); there is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)           # AttributeError here = header / library mismatch
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.gstvd_abi_version() != GSTVD_ABI_VERSION:
        raise RuntimeError("gst_visdial_b200: libgstvd.so ABI version mismatch; rebuild the extension")
    _lib = lib
    return lib


def check(ctx, rc: int) -> int:
    if rc < 0:
        msg = load().gstvd_last_error(ctx)
        raise GstvdError(rc, msg.decode() if msg else "")
    return rc
