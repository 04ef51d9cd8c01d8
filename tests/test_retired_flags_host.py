"""Host-side checks (no GPU needed): the C-ABI refuses flag bits outside the documented set of each entry point, so a
caller that still passes a retired debug bit fails loudly instead of silently getting another code path."""
from __future__ import annotations

import ctypes

import pytest

from pytorch_models_b200 import _lib

FAKE = 0x10000


def _run(op):
    lib = _lib.load()
    failed = ctypes.c_int(-1)
    rc = lib.b200enc_run_ops((_lib.Op * 1)(op), 1, ctypes.byref(failed), None)
    return rc, lib.b200enc_last_error()


def _linear_op(flags, M=256):
    op = _lib.Op()
    op.kind = _lib.OP_KINDS["b200enc_linear"]
    a = op.linear
    a.x, a.w, a.out = FAKE, FAKE, FAKE
    a.ldx, a.ldw, a.ldo = 768, 768, 768
    a.batches, a.M, a.N, a.K = 1, M, 768, 768
    a.flags = flags
    return op


def _attention_op(kind, flags, B=2):
    op = _lib.Op()
    op.kind = _lib.OP_KINDS[kind]
    for j in range(5):
        op.p[j] = FAKE
    op.i[:15] = (197 * 2304, 2304, 197 * 2304, 2304, 197 * 768, 768, B, 12, 197, 197, 64, flags, 0, 0, 197)
    op.f[0] = 0.125
    return op


@pytest.mark.parametrize("flags", [256, 512, 1024, 1 << 16, 1 << 17, _lib.LINEAR_GELU | 256])
def test_linear_refuses_undocumented_flags(flags):
    rc, msg = _run(_linear_op(flags))
    assert rc == -1
    assert f"flags={flags} ".encode() in msg


@pytest.mark.parametrize("kind", ["b200enc_attention", "b200enc_attention_bias"])
@pytest.mark.parametrize("flags", [65536, _lib.ATTN_CAUSAL | 65536])
def test_attention_refuses_undocumented_flags(kind, flags):
    rc, msg = _run(_attention_op(kind, flags))
    assert rc == -1
    assert f"flags={flags} ".encode() in msg


def test_shape_errors_are_reported_before_the_flag_check():
    rc, msg = _run(_linear_op(256, M=0))
    assert rc == -1 and b"bad shape batches=1 M=0" in msg
    for kind in ("b200enc_attention", "b200enc_attention_bias"):
        rc, msg = _run(_attention_op(kind, 65536, B=0))
        assert rc == -1 and b"bad shape B=0 H=12" in msg
