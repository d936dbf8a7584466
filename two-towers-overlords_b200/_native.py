"""
ctypes binding of libtt_b200.so (the C ABI declared in include/tt_b200.h).

PyTorch is only the allocator and stream provider here: every call passes raw device pointers
(`tensor.data_ptr()`), sizes and the current CUDA stream.  There is no CPU fallback: if the library is
missing or the device is not sm_100 the import / first call raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtt_b200.so")

# enum tt_dtype / tt_precision (include/tt_b200.h)
TT_F32, TT_BF16, TT_I64, TT_I32, TT_U16, TT_U8 = range(6)
PREC_FP32, PREC_BF16X3, PREC_BF16 = range(3)
PRECISIONS = {"fp32": PREC_FP32, "bf16x3": PREC_BF16X3, "bf16": PREC_BF16}

_DTYPES = {
    torch.float32: TT_F32, torch.bfloat16: TT_BF16, torch.int64: TT_I64, torch.int32: TT_I32,
    torch.uint16: TT_U16, torch.uint8: TT_U8, torch.int16: TT_U16,
}


class NativeError(RuntimeError):
    pass


class PoolSeg(ctypes.Structure):
    _fields_ = [("table", c_void_p), ("ids", c_void_p), ("mask", c_void_p), ("B", c_int), ("L", c_int),
                ("row0", c_int), ("_pad", c_int)]


class TokenBankDesc(ctypes.Structure):
    _fields_ = [("flat", c_void_p), ("offsets", c_void_p), ("dtype", c_int), ("_pad", c_int)]


class MinedNegatives(ctypes.Structure):
    _fields_ = [("table", c_void_p), ("count", c_void_p), ("depth", c_int), ("n_rows", c_int), ("n_docs", c_int),
                ("ratio", c_float)]


class StepArgs(ctypes.Structure):
    _fields_ = [
        ("q_ids", c_void_p), ("q_mask", c_void_p), ("Lq", c_int),
        ("p_ids", c_void_p), ("p_mask", c_void_p),
        ("n_ids", c_void_p), ("n_mask", c_void_p), ("Ld", c_int),
        ("ids_dtype", c_int), ("mask_dtype", c_int),
        ("B", c_int),
        ("table_q", c_void_p), ("table_d", c_void_p), ("table_dtype", c_int), ("vocab", c_int), ("H", c_int),
        ("P", c_int),
        ("Wq1", c_void_p), ("bq1", c_void_p), ("Wq2", c_void_p), ("bq2", c_void_p),
        ("Wd1", c_void_p), ("bd1", c_void_p), ("Wd2", c_void_p), ("bd2", c_void_p),
        ("margin", c_float), ("inv_batch", c_float), ("grad_scale", c_float),
        ("loss", c_void_p),
        ("dWq1", c_void_p), ("dbq1", c_void_p), ("dWq2", c_void_p), ("dbq2", c_void_p),
        ("dWd1", c_void_p), ("dbd1", c_void_p), ("dWd2", c_void_p), ("dbd2", c_void_p),
        ("dtable_q", c_void_p), ("dtable_d", c_void_p),
        ("err_flag", c_void_p),
        ("precision", c_int),
        ("ws", c_void_p), ("ws_bytes", c_size_t),
        ("phases", c_int),
        ("adam_state", c_void_p),
        ("adam_param", c_void_p), ("adam_grad", c_void_p), ("adam_exp_avg", c_void_p), ("adam_exp_avg_sq", c_void_p),
        ("adam_n", c_size_t),
        ("adam_lr", c_float), ("adam_beta1", c_float), ("adam_beta2", c_float), ("adam_eps", c_float),
        ("chain", c_int),
        ("neg_index", c_void_p),
        ("pooled_q", c_void_p), ("pooled_q_rows", c_int64),
        ("pooled_d", c_void_p), ("pooled_d_rows", c_int64),
        ("pooled_index", c_void_p),
        ("grad_accumulate", c_int),
        ("table_param_q", c_void_p), ("table_param_d", c_void_p),
        ("table_exp_avg_q", c_void_p), ("table_exp_avg_sq_q", c_void_p),
        ("table_exp_avg_d", c_void_p), ("table_exp_avg_sq_d", c_void_p),
    ]


class EncoderLayer(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in ("wqkv_hi", "wqkv_lo", "bqkv", "wo_hi", "wo_lo", "bo", "ln1_g", "ln1_b", "w1_hi",
                                        "w1_lo", "b1", "w2_hi", "w2_lo", "b2", "ln2_g", "ln2_b")]


class EncoderWeights(ctypes.Structure):
    _fields_ = [("word_emb", c_void_p), ("pos_emb", c_void_p), ("type_emb", c_void_p), ("emb_ln_g", c_void_p),
                ("emb_ln_b", c_void_p), ("vocab", c_int), ("max_pos", c_int), ("hidden", c_int), ("heads", c_int),
                ("inter", c_int), ("n_layers", c_int), ("ln_eps", c_float), ("layers", POINTER(EncoderLayer))]


# name -> (restype, argtypes): exactly the symbols include/tt_b200.h declares
_SIGNATURES = {
    "tt_version": (c_int, []),
    "tt_last_error": (c_char_p, []),
    "tt_launch_count": (ctypes.c_ulonglong, []),
    "tt_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "tt_pool_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tt_pool_fwd_multi": (c_int, [POINTER(PoolSeg), c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p]),
    "tt_pool_bwd_ws_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "tt_pool_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                            c_int, c_int, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "tt_mlp_ws_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "tt_encode_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "tt_encode_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "tt_triplet_loss_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_void_p, c_void_p,
                                    c_void_p]),
    "tt_triplet_loss_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p,
                                    c_void_p, c_void_p, c_void_p]),
    "tt_step_ws_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "tt_triplet_step": (c_int, [POINTER(StepArgs), c_void_p]),
    "tt_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float,
                             c_int, c_float, c_void_p]),
    "tt_adam_step_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float,
                                 c_void_p, c_float, c_void_p]),
    "tt_l2_normalize_rows": (c_int, [c_void_p, c_int64, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "tt_scan_ws_bytes": (c_size_t, [c_int, c_int64, c_int, c_int, c_int]),
    "tt_scan_topk": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_int64, c_int,
                             c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tt_score_candidates": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int64, c_void_p,
                                    c_void_p, c_void_p, c_void_p]),
    "tt_topk_merge": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "tt_ndcg_at_k": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tt_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), c_void_p]),
    "tt_peer_open": (c_int, [c_void_p, POINTER(c_void_p)]),
    "tt_peer_close": (c_int, [c_void_p]),
    "tt_peer_free": (c_int, [c_void_p]),
    "tt_dp_segment_bytes": (c_size_t, [c_size_t, c_int]),
    "tt_dp_reduce_adam": (c_int, [POINTER(c_void_p), c_int, c_int, c_size_t, c_void_p, c_void_p, c_void_p, c_float,
                                  c_float, c_float, c_float, c_void_p, c_void_p, c_int, c_void_p]),
    "tt_assemble_triplets": (c_int, [POINTER(TokenBankDesc), POINTER(TokenBankDesc), c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_int, c_int, c_int, ctypes.c_uint64, c_int, c_int, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "tt_assemble_triplet_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, ctypes.c_uint64,
                                         c_void_p, c_void_p, c_void_p, c_void_p]),
    "tt_mine_negatives": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                  c_void_p]),
    "tt_assemble_triplets_mined": (c_int, [POINTER(TokenBankDesc), POINTER(TokenBankDesc), c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_int, c_int, c_int, ctypes.c_uint64, c_int, c_int,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                           c_void_p, c_void_p, POINTER(MinedNegatives), c_void_p]),
    "tt_assemble_triplet_rows_mined": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                               ctypes.c_uint64, c_void_p, c_void_p, c_void_p, POINTER(MinedNegatives),
                                               c_void_p]),
    "tt_encoder_ws_bytes": (c_size_t, [c_int, c_int, c_int]),
    "tt_encoder_fwd": (c_int, [POINTER(EncoderWeights), c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                               c_void_p, c_size_t, c_void_p]),
    "tt_split_bf16_terms": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "tt_debug_step_buffer": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_char_p,
                                     POINTER(c_void_p)]),
    "tt_ubench_l2_read": (c_int, [c_void_p, c_size_t, c_int, c_int, c_void_p, c_void_p]),
    "tt_selftest_mn_major": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "tt_peer_barrier": (c_int, [POINTER(c_void_p), c_int, c_int, c_void_p, c_void_p]),
    "tt_peer_topk_merge": (c_int, [POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load() -> ctypes.CDLL:
    """Loads libtt_b200.so (no compute, no GPU needed) and attaches the signatures."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the two-tower hot path)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return (load().tt_last_error() or b"").decode()


def check(rc: int, what: str):
    if rc != 0:
        raise NativeError(f"{what} failed (rc={rc}): {last_error()}")


def require_device(t: torch.Tensor | None = None):
    if not torch.cuda.is_available():
        raise NativeError("the two-tower hot path needs a CUDA (sm_100a) device; there is no CPU fallback")
    if t is not None and not t.is_cuda:
        raise NativeError("expected a CUDA tensor; there is no CPU fallback")


def ptr(t: torch.Tensor | None) -> int | None:
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "native calls need contiguous CUDA tensors"
    return t.data_ptr()


def dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise NativeError(f"unsupported dtype {t.dtype}") from None


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


_device_checked = False


def ensure_sm100():
    global _device_checked
    if _device_checked:
        return
    require_device()
    sms, major, minor = c_int(), c_int(), c_int()
    check(load().tt_device_info(ctypes.byref(sms), ctypes.byref(major), ctypes.byref(minor)), "tt_device_info")
    _device_checked = True


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
