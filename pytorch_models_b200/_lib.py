"""ctypes binding of libb200enc.so (the C-ABI declared in include/b200enc.h).

There is no fallback: if the shared library has not been built (``python -c 'import __graft_entry__ as g; g.build()'``
or ``make -C pytorch_models_b200/csrc``) every kernel call raises. PyTorch only owns the buffers and the stream.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_longlong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200ENC_LIB: load another build of the same library instead (same-box A/B of compile-time variants:
# `make -C pytorch_models_b200/csrc variant NAME=ab_x DEFS=-D...` -> pytorch_models_b200/ab_x/libb200enc.so)
LIB_PATH = os.environ.get("B200ENC_LIB") or os.path.join(_HERE, "libb200enc.so")

LINEAR_GELU = 1
LINEAR_GELU_TANH = 2
LINEAR_RELU = 4
LINEAR_SILU = 8
ATTN_CAUSAL = 1
ATTN_GENERAL = 131072
LINEAR_FP8 = 16
DTYPE_BF16 = 0
DTYPE_F32 = 1

_lib = None


class LinearArgs(ctypes.Structure):
    """Mirror of ``b200enc_linear_args`` in include/b200enc.h."""

    _fields_ = [
        ("x", c_void_p), ("x_batch_stride", c_longlong), ("ldx", c_int),
        ("w", c_void_p), ("ldw", c_int),
        ("bias", c_void_p), ("colsum", c_void_p),
        ("rowstats", c_void_p), ("rowstats_parts", c_int), ("ln_eps", c_float),
        ("residual", c_void_p), ("res_batch_stride", c_longlong), ("ldr", c_int),
        ("out", c_void_p), ("out_batch_stride", c_longlong), ("ldo", c_int),
        ("stats_out", c_void_p),
        ("batches", c_int), ("M", c_int), ("N", c_int), ("K", c_int),
        ("flags", c_int),
        ("stats_rows_per_batch", c_int), ("stats_row_offset", c_int),
        ("acc_scale", c_void_p),
    ]


class Op(ctypes.Structure):
    """Mirror of ``b200enc_op`` in include/b200enc.h: one recorded launch of a plan (`plans.py`)."""

    _fields_ = [
        ("kind", c_int), ("reserved", c_int),
        ("linear", LinearArgs),
        ("p", c_void_p * 8), ("i", c_longlong * 16), ("f", c_float * 2),
    ]


# b200enc_op.kind per entry point (B200ENC_OP_* in include/b200enc.h)
OP_KINDS = {
    "b200enc_linear": 1, "b200enc_patch_embed16": 2, "b200enc_attention": 3, "b200enc_attention_bias": 4,
    "b200enc_layernorm": 5, "b200enc_row_stats": 6, "b200enc_mean_tokens": 7, "b200enc_patch_rows": 8,
    "b200enc_cls_rows": 9, "b200enc_embed_rows": 10, "b200enc_time_rows": 11,
}

_SIGNATURES = {
    "b200enc_version": (c_int, []),
    "b200enc_last_error": (ctypes.c_char_p, []),
    "b200enc_async_status": (ctypes.c_uint, [c_int]),
    "b200enc_tensor_map_cache_stats": (None, [ctypes.POINTER(ctypes.c_ulonglong), ctypes.POINTER(ctypes.c_ulonglong)]),
    "b200enc_linear": (c_int, [ctypes.POINTER(LinearArgs), c_void_p]),
    "b200enc_attention": (
        c_int,
        [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_longlong, c_int, c_void_p, c_longlong, c_int, c_int,
         c_int, c_int, c_int, c_int, c_float, c_int, c_void_p],
    ),
    "b200enc_attention_bias": (
        c_int,
        [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_longlong, c_int, c_void_p, c_longlong, c_int, c_int,
         c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_longlong, c_longlong, c_longlong, c_void_p],
    ),
    "b200enc_layernorm": (
        c_int,
        [c_void_p, c_longlong, c_void_p, c_void_p, c_float, c_int, c_int, c_void_p, c_longlong, c_void_p, c_void_p],
    ),
    "b200enc_row_stats": (c_int, [c_void_p, c_longlong, c_float, c_int, c_int, c_void_p, c_void_p]),
    "b200enc_mean_tokens": (
        c_int, [c_void_p, c_longlong, c_longlong, c_int, c_int, c_int, c_void_p, c_longlong, c_void_p]),
    "b200enc_patch_embed16": (c_int, [ctypes.POINTER(LinearArgs), c_int, c_int, c_void_p]),
    "b200enc_patch_rows": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "b200enc_cls_rows": (c_int, [c_void_p, c_int, c_int, c_void_p, c_longlong, c_void_p]),
    "b200enc_embed_rows": (
        c_int, [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "b200enc_whisper_logmel": (
        c_int, [c_void_p, c_longlong, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "b200enc_time_rows": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "b200enc_run_ops": (c_int, [ctypes.POINTER(Op), c_int, ctypes.POINTER(c_int), c_void_p]),
    "b200enc_attention_decode": (
        c_int,
        [c_void_p, c_longlong, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p,
         c_int, c_int, c_void_p, c_longlong, c_int, c_int, c_int, c_float, c_void_p, c_longlong, c_void_p],
    ),
    "b200enc_attention_decode_workspace_bytes": (c_longlong, [c_int, c_int, c_int, c_int]),
    "b200enc_embed_rows_at": (
        c_int,
        [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    ),
    "b200enc_decode_advance": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "b200enc_attention_extend": (
        c_int,
        [c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p, c_int, c_void_p,
         c_longlong, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p],
    ),
    "b200enc_kv_append": (
        c_int, [c_void_p, c_longlong, c_int, c_void_p, c_longlong, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int,
                c_void_p]),
    "b200enc_argmax_rows": (c_int, [c_void_p, c_longlong, c_int, c_int, c_void_p, c_longlong, c_void_p]),
    "b200enc_speculative_accept": (
        c_int, [c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p,
                c_longlong, c_int, c_int, c_void_p]),
    "b200enc_ngram_draft": (
        c_int, [c_void_p, c_longlong, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class B200EncError(RuntimeError):
    """A non-zero return from libb200enc (argument errors map to ValueError in `check`)."""


def load() -> ctypes.CDLL:
    """Load (once) and return the shared library; raise if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200EncError(
            f"{LIB_PATH} not found: the sm_100a extension is not built and there is no CPU/PyTorch fallback. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` from the repository root."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    msg = load().b200enc_last_error().decode("utf-8", "replace")
    if rc == -3:  # an earlier kernel gave up on a barrier wait: device-side fault, not a caller error
        raise B200EncError(f"{what}: {msg}")
    if rc < 0:
        raise ValueError(f"{what}: {msg}")
    raise B200EncError(f"{what}: CUDA error {rc}: {msg}")
