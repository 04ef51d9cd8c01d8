"""Host-side checks of incremental decoding (no GPU needed): the argument checks of the new C-ABI entry points and the
refusals of the cached decode path, all raised before anything is enqueued."""
from __future__ import annotations

import ctypes

import pytest
import torch

import pytorch_models_b200 as pm
from pytorch_models_b200 import _lib

A = 0x10000  # a 16-byte aligned fake device address: every call below fails its checks before touching it


def _decode(**over):
    """b200enc_attention_decode in append mode with valid arguments except for ``over``; returns (rc, message)."""
    B, H, hd, cap = 2, 3, 64, 100
    W = H * hd
    lib = _lib.load()
    ws = lib.b200enc_attention_decode_workspace_bytes(B, H, hd, cap)
    a = dict(q=A, q_bs=3 * W, k_new=A, v_new=A, new_bs=3 * W, k_cache=A, v_cache=A, cache_bs=cap * 2 * W,
             ld_cache=2 * W, capacity=cap, len=A, Lkv=0, out=A, out_bs=W, B=B, H=H, head_dim=hd, scale=0.125,
             ws=A, ws_bytes=ws)
    a.update(over)
    rc = lib.b200enc_attention_decode(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


def test_workspace_size_is_positive_and_grows_with_capacity():
    lib = _lib.load()
    small = lib.b200enc_attention_decode_workspace_bytes(1, 12, 64, 1024)
    big = lib.b200enc_attention_decode_workspace_bytes(1, 12, 64, 32768)
    assert 0 < small <= big
    assert lib.b200enc_attention_decode_workspace_bytes(0, 12, 64, 1024) == 0


@pytest.mark.parametrize("over,needle", [
    (dict(q=None), "q=(nil)"),
    (dict(out=None), "out=(nil)"),
    (dict(ws=None), "workspace=(nil)"),
    (dict(k_new=None), "needs k_new and v_new"),
    (dict(len=None, Lkv=50), "takes no k_new"),
    (dict(head_dim=32), "head_dim=32"),
    (dict(head_dim=72), "head_dim=72"),
    (dict(B=0), "B=0"),
    (dict(capacity=0), "capacity=0"),
    (dict(len=None, k_new=None, v_new=None, Lkv=101), "Lkv=101"),
    (dict(ld_cache=100), "ld_cache=100"),
    (dict(cache_bs=1000), "cache_batch_stride=1000"),
    (dict(q_bs=8), "q_batch_stride=8"),
    (dict(out_bs=8), "out_batch_stride=8"),
    (dict(new_bs=8), "new_batch_stride=8"),
    (dict(q=A + 8), "16-byte aligned"),
    (dict(out_bs=196), "out 196"),
    (dict(ws_bytes=16), "workspace_bytes=16"),
])
def test_decode_argument_checks(over, needle):
    rc, msg = _decode(**over)
    assert rc == -1 and needle in msg, msg


def _embed_at(**over):
    lib = _lib.load()
    a = dict(ids=A, rows=4, L=1, tok=A, pos=A, n_pos=10, pos0=A, dtype=0, vocab=50, d=64, out=A)
    a.update(over)
    rc = lib.b200enc_embed_rows_at(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    (dict(pos0=None), "null pointer"),
    (dict(rows=3, L=2), "rows=3"),
    (dict(n_pos=0), "n_pos=0"),
    (dict(vocab=0), "vocab=0"),
    (dict(d=60), "d=60"),
    (dict(out=A + 4), "16-byte aligned"),
    (dict(dtype=7), "dtype 7"),
])
def test_embed_rows_at_argument_checks(over, needle):
    rc, msg = _embed_at(**over)
    assert rc == -1 and needle in msg, msg


def test_decode_advance_refuses_null():
    lib = _lib.load()
    assert lib.b200enc_decode_advance(None, 1, None) == -1
    assert b"null len" in lib.b200enc_last_error()


# ---------------------------------------------------------------------------------------------- Python refusals
def _gpt2():
    return pm.GPT2(1, 64).eval()


def test_capacity_beyond_position_table():
    with pytest.raises(ValueError, match="capacity 1025"):
        _gpt2().new_kv_cache(1, 1025)
    with pytest.raises(ValueError, match="capacity 513"):
        pm.GPT(1, 64).eval().new_kv_cache(1, 513)
    with pytest.raises(ValueError, match="capacity 449"):
        pm.WhisperDecoder(100, 1, 64).eval().new_kv_cache(torch.zeros(1, 10, 64), 449)


def test_step_on_a_full_cache():
    m = _gpt2()
    cache = m.new_kv_cache(2, 4)
    cache.n = 4  # what four appended tokens leave behind
    with pytest.raises(ValueError, match="full"):
        m.step(torch.zeros(2, dtype=torch.long), cache)


def test_prefill_into_a_non_empty_cache():
    m = _gpt2()
    cache = m.new_kv_cache(1, 8)
    cache.n = 3
    with pytest.raises(ValueError, match="empty cache"):
        m.prefill(torch.zeros(1, 2, dtype=torch.long), cache)
    cache.reset()
    assert cache.n == 0 and int(cache.length.item()) == 0
    with pytest.raises(ValueError, match="capacity 8"):
        m.prefill(torch.zeros(1, 9, dtype=torch.long), cache)


def test_batch_mismatch():
    m = _gpt2()
    cache = m.new_kv_cache(2, 8)
    with pytest.raises(ValueError, match="batch 3"):
        m.step(torch.zeros(3, dtype=torch.long), cache)
    with pytest.raises(ValueError, match="batch 1"):
        m.prefill(torch.zeros(1, 4, dtype=torch.long), cache)
    with pytest.raises(ValueError, match="one token per sequence"):
        m.step(torch.zeros(2, 2, dtype=torch.long), cache)


def test_memory_shape_mismatch():
    dec = pm.WhisperDecoder(100, 1, 64).eval()
    with pytest.raises(ValueError, match="does not match"):
        dec.new_kv_cache(torch.zeros(1, 10, 32), 8)
    with pytest.raises(ValueError, match="does not match"):
        dec.layers.new_kv_cache(2, 8, torch.zeros(1, 10, 64))
    with pytest.raises(ValueError, match=r"\(N, Lm, d\)"):
        dec.new_kv_cache(torch.zeros(10, 64), 8)


def test_cross_attention_without_memory():
    with pytest.raises(NotImplementedError, match="without memory"):
        pm.Decoder(1, 64, cross_attn=True).eval().new_kv_cache(1, 8)


def test_training_mode_dropout():
    m = pm.GPT2(1, 64, dropout=0.1)  # training mode
    with pytest.raises(NotImplementedError, match="dropout"):
        m.new_kv_cache(1, 8)
    cache = m.eval().new_kv_cache(1, 8)
    m.train()
    with pytest.raises(NotImplementedError, match="dropout"):
        m.step(torch.zeros(1, dtype=torch.long), cache)


def test_cpu_tensors_are_refused_after_the_checks():
    m = _gpt2()
    cache = m.new_kv_cache(1, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.step(torch.zeros(1, dtype=torch.long), cache)
    assert cache.n == 0
