"""Host-side checks of the head_dim support (no GPU needed): which head dims the modules and the C-ABI accept."""
from __future__ import annotations

import ctypes

import pytest
import torch

import pytorch_models_b200 as pm
from pytorch_models_b200 import _lib


@pytest.mark.parametrize("hd", [80, 96, 112, 128])
def test_wide_head_dims_pass_the_module_check(hd):
    """MHA with a wide head is accepted and only stops at the device check (there is no CPU fallback)."""
    x = torch.randn(1, 4, 256)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.MHA(256, head_dim=hd).eval()(x)


@pytest.mark.parametrize("hd", [16, 32, 48, 72, 144, 256])
def test_other_head_dims_stay_refused_by_the_module(hd):
    with pytest.raises(NotImplementedError, match=f"head_dim={hd}"):
        pm.MHA(512, head_dim=hd).eval()(torch.randn(1, 4, 512))


def _attention_op(head_dim, B):
    fake = 0x10000
    op = _lib.Op()
    op.kind = _lib.OP_KINDS["b200enc_attention"]
    for j in range(4):
        op.p[j] = fake
    op.i[:12] = (1000, 640, 1000, 640, 1000, 640, B, 5, 7, 8, head_dim, 0)   # ..., B, H, Lq, Lkv, head_dim, flags
    return op


@pytest.mark.parametrize("hd", [48, 72, 144, 256])
def test_c_abi_refuses_other_head_dims(hd):
    """The head_dim check comes first (before the shape check) and names the value."""
    lib = _lib.load()
    failed = ctypes.c_int(-1)
    ops = (_lib.Op * 1)(_attention_op(hd, 0))
    assert lib.b200enc_run_ops(ops, 1, ctypes.byref(failed), None) == -1
    assert f"head_dim={hd}".encode() in lib.b200enc_last_error()


@pytest.mark.parametrize("hd", [80, 128])
def test_c_abi_accepts_wide_head_dims(hd):
    """head_dim 80 / 128 get past the head_dim check and stop at the next one, the shape check (B = 0)."""
    lib = _lib.load()
    failed = ctypes.c_int(-1)
    ops = (_lib.Op * 1)(_attention_op(hd, 0))
    assert lib.b200enc_run_ops(ops, 1, ctypes.byref(failed), None) == -1
    assert b"B=0 H=5 Lq=7 Lkv=8" in lib.b200enc_last_error()
