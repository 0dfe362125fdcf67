"""ctypes binding of the C-ABI library (include/chimeralm_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, this module
raises.  Build the library with `python -c "import __graft_entry__ as g; g.build()"` or
`make -C chimeralm_b200/csrc`.
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

LIB_NAME = "libchimeralm_b200.so"
LIB_PATH = Path(__file__).resolve().parent / LIB_NAME

CLM_F32, CLM_BF16, CLM_U8, CLM_I32, CLM_I64 = 0, 1, 2, 3, 4
CLM_ERR_STATE, CLM_ERR_TOKEN_RANGE, CLM_ERR_FP16_RANGE = -3, -6, -7
EPI_BIAS_BF16, EPI_BIAS_GELU_TANH, EPI_BIAS_RES_F32, EPI_SCORE = 0, 1, 2, 3


class clm_config(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "d_model", "n_layer", "d_inner", "vocab_rows", "max_seq_len", "filter_order", "emb_dim",
        "short_filter_order", "num_inner_mlps", "head_hidden", "num_classes")] + [
        ("layer_norm_eps", C.c_float), ("filter_shift", C.c_float), ("pooling", C.c_int)]

POOLING = {"attention": 0, "mean": 1, "max": 2, "cls": 3}


class clm_head_train_cfg(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("dropout", C.c_double), ("seed", C.c_uint)]


class ChimeraLMNativeError(RuntimeError):
    def __init__(self, msg, status: int = 0):
        super().__init__(msg)
        self.status = status


class Fp16RangeError(ChimeraLMNativeError):
    """A batch left the range of the fp16 tensor-core convolution; its logits are invalid (rerun with tc_conv off)."""


# name -> (restype, argtypes); mirrors include/chimeralm_b200.h one to one
_SIGNATURES = {
    "clm_default_config": (None, [C.POINTER(clm_config)]),
    "clm_version": (C.c_char_p, []),
    "clm_create": (C.c_int, [C.POINTER(clm_config), C.c_int, C.POINTER(C.c_void_p)]),
    "clm_destroy": (None, [C.c_void_p]),
    "clm_last_error": (C.c_char_p, [C.c_void_p]),
    "clm_load_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.c_int]),
    "clm_finalize": (C.c_int, [C.c_void_p]),
    "clm_reserve": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "clm_reserve_tokens": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_longlong]),
    "clm_encode_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "clm_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "clm_predict_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_void_p, C.c_void_p]),
    "clm_predict_host_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "clm_predict_host_wait": (C.c_int, [C.c_void_p, C.c_int]),
    "clm_forward_seq": (C.c_longlong, [C.c_void_p]),
    "clm_forward_status": (C.c_int, [C.c_void_p, C.c_longlong]),
    "clm_tc_fallback_count": (C.c_longlong, [C.c_void_p]),
    "clm_launch_count": (C.c_longlong, [C.c_void_p]),
    "clm_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "clm_profile_reset": (C.c_int, [C.c_void_p]),
    "clm_profile_num": (C.c_int, []),
    "clm_profile_name": (C.c_char_p, [C.c_int]),
    "clm_profile_get": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "clm_gemm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "clm_block_in": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "clm_block_in_trace": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "clm_block_mlp": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "clm_block_mlp_cm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "clm_block_mlp_cm_trace": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p]),
    "clm_block_mlp_trace": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "clm_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "clm_longconv": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                               C.c_void_p]),
    "clm_longconv_tc": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p]),
    "clm_longconv_tc_auto": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p]),
    "clm_attention_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "clm_longconv_variant": (C.c_int, [C.c_void_p, C.c_int]),
    "clm_longconv_tc_trace": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p, C.c_void_p]),
    "clm_get_filter": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "clm_set_debug_stop": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "clm_debug_copy": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "clm_head_train_begin": (C.c_int, [C.c_void_p, C.POINTER(clm_head_train_cfg)]),
    "clm_head_train_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "clm_head_grad_copy": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p]),
    "clm_head_export": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p]),
    "clm_bam_open": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]),
    "clm_bam_close": (None, [C.c_void_p]),
    "clm_bam_error": (C.c_char_p, [C.c_void_p]),
    "clm_bam_records_seen": (C.c_longlong, [C.c_void_p]),
    "clm_bam_set_chunk_bytes": (C.c_int, [C.c_void_p, C.c_longlong]),
    "clm_bam_set_shard": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "clm_bam_next": (C.c_longlong, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong,
                                    C.c_void_p, C.c_void_p, C.c_int]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)
_lib = None


def load() -> C.CDLL:
    """Load the native library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ChimeraLMNativeError(
            f"{LIB_PATH} not found: the CUDA extension is not built and there is no CPU fallback. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'`.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(ctx, rc: int, what: str) -> None:
    if rc < 0:
        msg = load().clm_last_error(ctx)
        text = f"{what} failed (status {rc}): {msg.decode() if msg else '?'}"
        if rc == CLM_ERR_TOKEN_RANGE:
            raise IndexError(text)   # what the reference's nn.Embedding raises for an id outside the table
        raise (Fp16RangeError if rc == CLM_ERR_FP16_RANGE else ChimeraLMNativeError)(text, rc)
