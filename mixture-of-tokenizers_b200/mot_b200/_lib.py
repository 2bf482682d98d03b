"""ctypes binding of libmot_b200.so (the C ABI declared in include/mot_b200.h).

The library is the product: there is no CPU or PyTorch fallback.  If the shared
object is missing it is built in-tree with nvcc (mixture-of-tokenizers_b200/build.py);
if that is impossible the import fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmot_b200" + os.environ.get("MOT_LIB_SUFFIX", "") + ".so")  # suffix: experiment builds

ABI_VERSION = 7
# enums of include/mot_b200.h
OK, ERR_BAD_ARG, ERR_UNSUPPORTED, ERR_MISALIGNED, ERR_WORKSPACE, ERR_CUDA, ERR_NO_DEVICE = range(7)
BF16, F32 = 0, 1
TTB_I16, TTB_F32, TTB_BF16 = 0, 1, 2
ADD, CONCAT, TOK_ONLY, BYTES_ONLY, MEAN = range(5)
F_TOK_NORM, F_BYTE_NORM, F_OUT_NORM, F_BYTES_FIRST = 1, 2, 4, 8
F_SLOT_MAJOR, F_IDS_FROM_TTB, F_TTB_SCRAMBLE, F_IDS_I64, F_HAS_LAMBDAS = 16, 32, 64, 128, 256
F_TTB_PULL_LEFT, F_TTB_PULL_RIGHT, F_TTB_NEXT_TOK = 512, 1024, 2048
WS_PLAN_READY, WS_CLEAN, WS_PLAN_JOINED = 1, 2, 4
DP_NVLS, DP_P2P = 0, 1
DP_MAX_ROW_TABLES = 8


class MotDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("dtype", C.c_int32),
        ("n_tokens", C.c_int64), ("seq_len", C.c_int64),
        ("tok_vocab", C.c_int32), ("byte_vocab", C.c_int32), ("bpt", C.c_int32),
        ("tok_dim", C.c_int32), ("byte_dim", C.c_int32), ("out_dim", C.c_int32),
        ("combine", C.c_int32), ("flags", C.c_int32), ("ttb_dtype", C.c_int32),
        ("eps", C.c_float),
        ("row_stride", C.c_int64), ("col_offset", C.c_int32), ("dp_slabs", C.c_int32),
        ("pad_id", C.c_int32), ("eot_id", C.c_int32),
    ]


class MotRowTable(C.Structure):
    _fields_ = [("byte_offset", C.c_int64), ("row_bytes", C.c_int32), ("reserved", C.c_int32)]


_P = C.c_void_p
_SIGNATURES = {
    "mot_strerror": (C.c_char_p, [C.c_int]),
    "mot_abi_version": (C.c_int, []),
    "mot_last_cuda_error": (C.c_char_p, []),
    "mot_launch_count": (C.c_int64, []),
    "mot_launch_count_reset": (None, []),
    "mot_profile_events": (None, [_P, _P, _P, _P]),
    "mot_profile_trace": (None, [_P]),
    "mot_ttb_expand": (C.c_int, [_P, C.c_int64, _P, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
    "mot_ttb_build": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "mot_ttb_repad": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "mot_tokens_to_digits": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, _P, C.c_int32, _P]),
    "mot_embed_workspace_bytes": (C.c_size_t, [C.POINTER(MotDesc)]),
    "mot_embed_fwd": (C.c_int, [C.POINTER(MotDesc), _P, _P, _P, _P, _P, _P, _P, _P]),
    "mot_embed_workspace_init": (C.c_int, [C.POINTER(MotDesc), _P, C.c_size_t, _P]),
    "mot_embed_plan": (C.c_int, [C.POINTER(MotDesc), _P, _P, C.c_size_t, C.c_int32, _P]),
    "mot_embed_plan_async": (C.c_int, [C.POINTER(MotDesc), _P, _P, C.c_size_t, C.c_int32, _P, _P, _P, _P]),
    "mot_stream_wait_event": (C.c_int, [_P, _P]),
    "mot_embed_bwd": (C.c_int, [C.POINTER(MotDesc), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t,
                                C.c_int32, _P]),
    "mot_embed_fwd_ex": (C.c_int, [C.POINTER(MotDesc), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mot_embed_bwd_ex": (C.c_int, [C.POINTER(MotDesc), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                   C.c_size_t, C.c_int32, _P]),
    "mot_embed_bwd_slab": (C.c_int, [C.POINTER(MotDesc), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t,
                                     C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "mot_embed_slab_rows": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "mot_tokens_widen_u16": (C.c_int, [_P, C.c_int64, _P, _P]),
    "mot_embed_bwd_uses_saved": (C.c_int, [C.POINTER(MotDesc)]),
    "mot_byte_pair_fwd": (C.c_int, [C.POINTER(MotDesc), _P, _P, _P, _P, _P, _P, _P]),
    "mot_byte_pair_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "mot_byte_pair_bwd": (C.c_int, [C.POINTER(MotDesc), _P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "mot_dp_exchange": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_uint32, C.c_int32,
                                  C.c_int32, _P]),
    "mot_embed_touched_rows": (C.c_int, [C.POINTER(MotDesc), _P, C.c_size_t, _P, _P]),
    "mot_dp_exchange_rows": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64,
                                       C.c_int64, C.c_int32, C.c_uint32, C.c_int32, _P]),
    "mot_dp_exchange_rows_multi": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, C.POINTER(MotRowTable), C.c_int32, C.c_int32,
                                             C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_uint32, C.c_int32, _P]),
    "mot_dp_allreduce_avg": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_uint32, _P]),
    "mot_pull_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int32]),
    "mot_pull": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P,
                           C.c_size_t, _P]),
    "mot_mixout_copy_fwd": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P]),
    "mot_mixout_copy_bwd": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P]),
    "mot_linear_fwd": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "mot_linear_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
    "mot_linear_bwd_input": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, C.c_size_t, _P]),
    "mot_linear_bwd_weight": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, C.c_size_t, _P]),
    "mot_cast_f32_bf16": (C.c_int, [_P, _P, C.c_int64, _P]),
    "mot_colsum": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P]),
    "mot_rmsnorm_fwd": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_float, _P]),
    "mot_rmsnorm_bwd": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_float, _P]),
}

_lib = None


def _build_if_missing() -> None:
    if os.path.exists(LIB_PATH):
        return
    sys.path.insert(0, os.path.dirname(_HERE))
    try:
        import build as _build  # mixture-of-tokenizers_b200/build.py
        _build.build()
    finally:
        sys.path.pop(0)


def lib() -> C.CDLL:
    """The loaded library; raises if it cannot be found or built (no fallback)."""
    global _lib
    if _lib is None:
        _build_if_missing()
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"mot_b200: {LIB_PATH} is missing and could not be built; "
                               "this package has no CPU / PyTorch fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        if L.mot_abi_version() != ABI_VERSION:
            raise RuntimeError("mot_b200: libmot_b200.so ABI version mismatch; rebuild")
        _lib = L
    return _lib


def exported_symbols() -> list[str]:
    return sorted(_SIGNATURES)


def check(rc: int, what: str) -> None:
    if rc != OK:
        L = lib()
        msg = L.mot_strerror(rc).decode()
        if rc == ERR_CUDA:
            msg += ": " + L.mot_last_cuda_error().decode()
        if rc == ERR_UNSUPPORTED:
            raise NotImplementedError(f"{what}: {msg}")
        raise RuntimeError(f"{what}: {msg}")
