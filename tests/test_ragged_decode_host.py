"""Host-side checks of ragged incremental decoding, sequences of different lengths in one batch (no GPU needed): the
argument checks of the per-sequence entry points, the refusals of a ragged prefill, and that a ragged decode step
issues the same launches as a shared-length one."""
from __future__ import annotations

import pytest
import torch

import pytorch_models_b200 as pm
from pytorch_models_b200 import _lib, ops
from pytorch_models_b200.transformer import KVCache

A = 0x10000  # a 16-byte aligned fake device address: every call below fails its checks before touching it


def _decode_ragged(**over):
    """b200enc_attention_decode_ragged with valid arguments except for ``over``; returns (rc, message)."""
    B, H, hd, cap = 2, 3, 64, 100
    W = H * hd
    lib = _lib.load()
    ws = lib.b200enc_attention_decode_workspace_bytes(B, H, hd, cap)
    a = dict(q=A, q_bs=3 * W, k_new=A, v_new=A, new_bs=3 * W, k_cache=A, v_cache=A, cache_bs=cap * 2 * W,
             ld_cache=2 * W, capacity=cap, lens=A, out=A, out_bs=W, B=B, H=H, head_dim=hd, scale=0.125,
             ws=A, ws_bytes=ws)
    a.update(over)
    rc = lib.b200enc_attention_decode_ragged(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    (dict(lens=None), "lens=(nil)"),
    (dict(q=None), "q=(nil)"),
    (dict(out=None), "out=(nil)"),
    (dict(ws=None), "workspace=(nil)"),
    (dict(k_new=None), "needs k_new and v_new"),
    (dict(head_dim=72), "head_dim=72"),
    (dict(B=0), "B=0"),
    (dict(capacity=0), "capacity=0"),
    (dict(ld_cache=100), "ld_cache=100"),
    (dict(cache_bs=1000), "cache_batch_stride=1000"),
    (dict(q_bs=8), "q_batch_stride=8"),
    (dict(new_bs=8), "new_batch_stride=8"),
    (dict(q=A + 8), "16-byte aligned"),
    (dict(out_bs=196), "out 196"),
    (dict(ws_bytes=16), "workspace_bytes=16"),
])
def test_decode_ragged_argument_checks(over, needle):
    rc, msg = _decode_ragged(**over)
    assert rc == -1 and needle in msg, msg
    assert msg.startswith("b200enc_attention_decode_ragged:"), msg


def _embed_at_ragged(**over):
    lib = _lib.load()
    a = dict(ids=A, rows=4, L=1, tok=A, pos=A, n_pos=10, pos0=A, dtype=0, vocab=50, d=64, out=A)
    a.update(over)
    rc = lib.b200enc_embed_rows_at_ragged(*a.values(), None)
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
def test_embed_rows_at_ragged_argument_checks(over, needle):
    rc, msg = _embed_at_ragged(**over)
    assert rc == -1 and needle in msg and msg.startswith("b200enc_embed_rows_at_ragged:"), msg


def test_decode_advance_ragged_checks():
    lib = _lib.load()
    assert lib.b200enc_decode_advance_ragged(None, 4, 1, None) == -1
    assert b"null len" in lib.b200enc_last_error()
    assert lib.b200enc_decode_advance_ragged(A, 0, 1, None) == -1
    assert b"n=0" in lib.b200enc_last_error()


def test_ops_refuse_a_length_of_the_wrong_size():
    cpu = torch.zeros(3, dtype=torch.int32)
    with pytest.raises(ValueError, match="1 or 2 elements"):
        ops._per_sequence(cpu, 2, "length")
    with pytest.raises(ValueError, match="1 or 3 elements"):
        ops._per_sequence(torch.zeros(3, 2, dtype=torch.int32)[:, 0], 3, "length")
    assert not ops._per_sequence(torch.zeros(1, dtype=torch.int32), 4, "length")
    assert ops._per_sequence(torch.zeros(4, dtype=torch.int32), 4, "length")


# ---------------------------------------------------------------------------------------------- Python refusals
def _gpt2():
    return pm.GPT2(1, 64).eval()


@pytest.mark.parametrize("lengths,match", [
    ([3], "1 entries for a batch of 2"),
    ([3, 4, 1], "3 entries for a batch of 2"),
    ([0, 4], r"length 0 is outside \[1, 4\]"),
    ([2, 5], r"length 5 is outside \[1, 4\]"),
])
def test_prefill_refuses_bad_lengths(lengths, match):
    m = _gpt2()
    cache = m.new_kv_cache(2, 8)
    with pytest.raises(ValueError, match=match):
        m.prefill(torch.zeros(2, 4, dtype=torch.long), cache, lengths=lengths)
    assert cache.n == 0 and not cache.ragged


def test_prefill_refuses_cuda_lengths():
    class FakeCuda(torch.Tensor):  # a tensor that reports a CUDA device, so no GPU is needed to see the refusal
        @property
        def is_cuda(self):
            return True

    m = _gpt2()
    cache = m.new_kv_cache(2, 8)
    lengths = torch.tensor([1, 2]).as_subclass(FakeCuda)
    with pytest.raises(ValueError, match="not a CUDA tensor"):
        m.prefill(torch.zeros(2, 4, dtype=torch.long), cache, lengths=lengths)
    assert cache.n == 0


def test_uniform_refusals_come_first():
    m = _gpt2()
    cache = m.new_kv_cache(2, 8)
    with pytest.raises(ValueError, match="batch 3"):
        m.prefill(torch.zeros(3, 4, dtype=torch.long), cache, lengths=[1, 2, 3])
    with pytest.raises(ValueError, match="capacity 8"):
        m.prefill(torch.zeros(2, 9, dtype=torch.long), cache, lengths=[1, 9])
    cache.n = 2
    with pytest.raises(ValueError, match="empty cache"):
        m.prefill(torch.zeros(2, 4, dtype=torch.long), cache, lengths=[1, 4])


def test_cpu_ids_are_refused_after_the_checks():
    m = _gpt2()
    cache = m.new_kv_cache(2, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.prefill(torch.zeros(2, 4, dtype=torch.long), cache, lengths=[1, 4])
    assert cache.n == 0 and not cache.ragged


def _ragged_cache(dec, B=2, capacity=8, P=5, lengths=(2, 5)):
    cache = KVCache(dec, B, capacity, None)
    dec.prefill(torch.zeros(B, P, dec.d_model, dtype=torch.bfloat16), cache, lengths=list(lengths))
    return cache


def test_host_mirror_of_a_ragged_fill(monkeypatch):
    for name in ("linear", "attention", "row_stats", "layernorm"):
        monkeypatch.setattr(ops, name, lambda *a, **k: None)
    dec = pm.Decoder(1, 64).eval()
    cache = _ragged_cache(dec)
    assert cache.ragged and cache.n == 5 and cache.pad == [3, 0]
    assert cache.seq_lengths == [2, 5]
    assert cache.length is cache.seq_length and cache.length.tolist() == [2, 5]
    seq_length = cache.seq_length
    cache.n += 3  # what three steps leave behind
    assert cache.seq_lengths == [5, 8]
    with pytest.raises(ValueError, match="full"):  # the longest sequence is full
        cache.check_step(2)
    cache.reset()
    assert not cache.ragged and cache.length is cache.shared_length and cache.seq_lengths == [0, 0]
    dec.prefill(torch.zeros(2, 4, 64, dtype=torch.bfloat16), cache, lengths=torch.tensor([4, 1]))
    assert cache.seq_length is seq_length, "the per-sequence length tensor must outlive a prefill (graph capture)"
    assert cache.seq_lengths == [4, 1] and cache.length.tolist() == [4, 1]


# ---------------------------------------------------------------------------------------------- launch lists
CASES = {f"{norm}_{attn}": dict(pre_norm=norm == "pre", cross=attn == "cross")
         for norm in ("pre", "post") for attn in ("self", "cross")}


def _step_launches(case, ragged, monkeypatch):
    from test_decoder_launches_host import RECORDED, Recorder

    rec = Recorder()
    for name, ret in RECORDED.items():
        monkeypatch.setattr(ops, name, rec.entry(name, ret))
    torch.manual_seed(0)
    B, P, d = 3, 5, 128
    dec = pm.Decoder(2, d, head_dim=64, cross_attn=case["cross"], pre_norm=case["pre_norm"]).eval()
    m3 = torch.zeros(B, 7, d, dtype=torch.bfloat16) if case["cross"] else None
    cache = KVCache(dec, B, 16, m3)
    dec.prefill(torch.zeros(B, P, d, dtype=torch.bfloat16), cache, lengths=[2, 5, 1] if ragged else None)
    n = len(rec.calls)
    x1 = torch.zeros(B, 1, d, dtype=torch.bfloat16)
    dec.step(x1, cache)
    dec.step(x1, cache)
    return rec.calls[n:], cache


@pytest.mark.parametrize("name", list(CASES))
def test_ragged_step_issues_the_uniform_launches(name, monkeypatch):
    """Same entry points, same arguments; only the length tensor is (B,) instead of (1,)."""
    import json

    uniform, cu = _step_launches(CASES[name], False, monkeypatch)
    monkeypatch.undo()
    ragged, cr = _step_launches(CASES[name], True, monkeypatch)
    assert cu.length.shape == (1,) and cr.length.shape == (3,)
    want = json.loads(json.dumps(uniform).replace(" (1) (1) int32", " (3) (1) int32"))
    got = json.loads(json.dumps(ragged))
    assert len(got) == len(want)
    assert sum(" (3) (1) int32" in json.dumps(c) for c in got) > 0, "no launch reads the per-sequence lengths"
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, f"launch {i} differs:\n got  {g}\n want {w}"
