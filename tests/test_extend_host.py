"""Host-side checks of extending a filled KV cache by several tokens per sequence (no GPU needed): the argument checks
of b200enc_attention_extend and b200enc_kv_append, the refusals of `extend`, the cache's host mirror afterwards, and
that an extend issues the launches of a prefill with the self-attention replaced by kv_append + attention_extend."""
from __future__ import annotations

import json
import re

import pytest
import torch

import pytorch_models_b200 as pm
from pytorch_models_b200 import _lib, ops
from pytorch_models_b200.transformer import KVCache

A = 0x10000  # a 16-byte aligned fake device address: every call below fails its checks before touching it


def _extend(**over):
    """b200enc_attention_extend with valid arguments except for ``over``; returns (rc, message)."""
    B, H, hd, cap, P = 2, 3, 64, 100, 7
    W = H * hd
    lib = _lib.load()
    a = dict(q=A, q_bs=P * 3 * W, ldq=3 * W, k=A, v=A + 2 * W, cache_bs=cap * 2 * W, ld_cache=2 * W, capacity=cap,
             lens=A, len_stride=1, out=A, out_bs=P * W, ldo=W, B=B, H=H, P=P, head_dim=hd, scale=0.125)
    a.update(over)
    rc = lib.b200enc_attention_extend(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    (dict(lens=None), "lens=(nil)"),
    (dict(q=None), "null tensor pointer"),
    (dict(k=None), "null tensor pointer"),
    (dict(out=None), "null tensor pointer"),
    (dict(head_dim=72), "head_dim=72"),
    (dict(head_dim=144), "head_dim=144"),
    (dict(len_stride=2), "len_stride=2"),
    (dict(len_stride=-1), "len_stride=-1"),
    (dict(P=101), "P=101 new rows do not fit a cache of capacity=100"),
    (dict(P=0), "P=0"),
    (dict(B=0), "B=0"),
    (dict(cache_bs=1000), "cache_batch_stride=1000"),
    (dict(ld_cache=100), "16-byte aligned"),
    (dict(ldq=580), "16-byte aligned"),
    (dict(q=A + 8), "16-byte aligned"),
    (dict(v=A + 2), "16-byte aligned"),
    (dict(out=A + 8), "output rows must be 16-byte aligned"),
    (dict(ldo=100), "leading dimension"),
])
def test_attention_extend_argument_checks(over, needle):
    rc, msg = _extend(**over)
    assert rc == -1 and needle in msg, msg
    assert msg.startswith("b200enc_attention_extend:"), msg


def _append(**over):
    B, P, W, cap = 2, 7, 384, 100
    lib = _lib.load()
    a = dict(src=A, src_bs=P * 576, ld_src=576, cache=A, cache_bs=cap * W, ld_cache=W, capacity=cap, lens=A,
             len_stride=0, B=B, P=P, width=W)
    a.update(over)
    rc = lib.b200enc_kv_append(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    (dict(src=None), "null pointer"),
    (dict(cache=None), "null pointer"),
    (dict(lens=None), "null pointer"),
    (dict(len_stride=3), "len_stride=3"),
    (dict(width=60), "width=60"),
    (dict(P=0), "P=0"),
    (dict(P=101), "P=101 new rows do not fit a cache of capacity=100"),
    (dict(ld_cache=200), "ld_cache=200"),
    (dict(cache_bs=1000), "cache_batch_stride=1000"),
    (dict(src=A + 8), "16-byte aligned"),
    (dict(ld_src=580), "16-byte aligned"),
])
def test_kv_append_argument_checks(over, needle):
    rc, msg = _append(**over)
    assert rc == -1 and needle in msg and msg.startswith("b200enc_kv_append:"), msg


def test_ops_refuse_mismatched_cache_views():
    cache = torch.zeros(2, 16, 128, dtype=torch.bfloat16)
    length = torch.zeros(1, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):  # shapes fine: only the device is wrong
        ops.kv_append(torch.zeros(2, 3, 128, dtype=torch.bfloat16), cache, length)
    ops_dev = ops._need_cuda
    try:
        ops._need_cuda = lambda *ts: torch.device("cpu")
        with pytest.raises(ValueError, match=r"\(B=2, capacity, 128\)"):
            ops.kv_append(torch.zeros(2, 3, 128, dtype=torch.bfloat16), cache[:, :, :64], length)
        with pytest.raises(ValueError, match="1 or 2 elements"):
            ops.kv_append(torch.zeros(2, 3, 128, dtype=torch.bfloat16), cache, torch.zeros(3, dtype=torch.int32))
        q = torch.zeros(2, 3, 64, dtype=torch.bfloat16)
        with pytest.raises(ValueError, match="share shape and strides"):
            ops.attention_extend(q, cache[:, :, :64], cache[:, :8, 64:], q.clone(), 1, 0.125, length)
    finally:
        ops._need_cuda = ops_dev


# ---------------------------------------------------------------------------------------------- Python refusals
ENTRY_POINTS = ("linear", "attention", "attention_decode", "row_stats", "layernorm", "decode_advance", "kv_append",
                "attention_extend", "embed_rows", "embed_rows_at")


@pytest.fixture
def launches(monkeypatch):
    """Every `ops` entry point the decoders call, replaced by a recorder that launches nothing."""
    calls = []
    for name in ENTRY_POINTS:
        monkeypatch.setattr(ops, name, lambda *a, _n=name, **k: calls.append(_n))
    return calls


def _gpt2():
    return pm.GPT2(1, 64).eval()


class FakeCuda(torch.Tensor):  # a tensor that reports a CUDA device, so no GPU is needed to see the refusal
    @property
    def is_cuda(self):
        return True


@pytest.mark.parametrize("make_call,exc,match", [
    (lambda m, c: m.extend(torch.zeros(3, 4, dtype=torch.long), c), ValueError, "batch 3"),
    (lambda m, c: m.extend(torch.zeros(2, 9, dtype=torch.long), c), ValueError, "capacity 8"),
    (lambda m, c: m.extend(torch.zeros(2, 4, dtype=torch.long), c, lengths=[3]), ValueError, "1 entries"),
    (lambda m, c: m.extend(torch.zeros(2, 4, dtype=torch.long), c, lengths=[0, 4]), ValueError, r"length 0"),
    (lambda m, c: m.extend(torch.zeros(2, 4, dtype=torch.long), c, lengths=[2, 5]), ValueError, r"length 5"),
    (lambda m, c: m.extend(torch.zeros(2, 4, dtype=torch.long), c,
                           lengths=torch.tensor([1, 2]).as_subclass(FakeCuda)), ValueError, "not a CUDA tensor"),
    (lambda m, c: m.train().extend(torch.zeros(2, 4, dtype=torch.long), c), NotImplementedError, "dropout"),
])
def test_extend_refusals_come_before_any_launch(make_call, exc, match, launches):
    m = pm.GPT2(1, 64, dropout=0.1).eval()
    cache = m.new_kv_cache(2, 8)
    with pytest.raises(exc, match=match):
        make_call(m, cache)
    assert launches == [] and cache.n == 0 and not cache.ragged


def test_extend_refuses_to_overflow_a_filled_cache(launches):
    dec = pm.Decoder(1, 64).eval()
    cache = KVCache(dec, 2, 8, None)
    dec.extend(torch.zeros(2, 5, 64, dtype=torch.bfloat16), cache, lengths=[5, 2])
    n = len(launches)
    with pytest.raises(ValueError, match="extend of 4 tokens onto 5 held tokens overflows a cache of capacity 8"):
        dec.extend(torch.zeros(2, 4, 64, dtype=torch.bfloat16), cache)
    with pytest.raises(ValueError, match="batch 3"):
        dec.extend(torch.zeros(3, 1, 64, dtype=torch.bfloat16), cache)
    assert len(launches) == n and cache.seq_lengths == [5, 2]
    dec.extend(torch.zeros(2, 3, 64, dtype=torch.bfloat16), cache)  # exactly full
    assert cache.seq_lengths == [8, 5]


def test_cpu_ids_are_refused_after_the_checks():
    m = _gpt2()
    cache = m.new_kv_cache(2, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.extend(torch.zeros(2, 4, dtype=torch.long), cache, lengths=[1, 4])
    assert cache.n == 0 and not cache.ragged


# ---------------------------------------------------------------------------------------------- host mirror
def test_host_mirror_after_extends(launches):
    dec = pm.Decoder(1, 64).eval()
    cache = KVCache(dec, 2, 32, None)
    x = lambda P: torch.zeros(2, P, 64, dtype=torch.bfloat16)  # noqa: E731
    dec.extend(x(4), cache)  # on an empty cache
    assert not cache.ragged and cache.n == 4 and cache.length is cache.shared_length and cache.length.tolist() == [4]
    dec.extend(x(5), cache, lengths=[3, 3])  # equal lengths keep one shared length
    assert not cache.ragged and cache.n == 7 and cache.length.tolist() == [7]
    dec.extend(x(5), cache, lengths=[5, 2])  # unequal lengths: the shared-length cache becomes ragged
    assert cache.ragged and cache.length is cache.seq_length
    assert cache.seq_lengths == [12, 9] and cache.length.tolist() == [12, 9] and cache.n == 12 and cache.pad == [0, 3]
    dec.extend(x(2), cache)  # a ragged cache stays ragged
    assert cache.ragged and cache.seq_lengths == [14, 11] and cache.length.tolist() == [14, 11]
    dec.extend(x(6), cache, lengths=[1, 6])
    assert cache.seq_lengths == [15, 17] and cache.length.tolist() == [15, 17] and cache.pad == [2, 0]
    assert launches.count("kv_append") == 5 and launches.count("attention_extend") == 5
    assert "decode_advance" not in launches  # the lengths come from the host mirror, as after a prefill

    cache.reset()
    dec.prefill(x(5), cache, lengths=[2, 5])
    dec.extend(x(3), cache)
    assert cache.ragged and cache.seq_lengths == [5, 8] and cache.length.tolist() == [5, 8]


# ---------------------------------------------------------------------------------------------- launch lists
CASES = {f"{norm}_{attn}": dict(pre_norm=norm == "pre", cross=attn == "cross")
         for norm in ("pre", "post") for attn in ("self", "cross")}
B, L, LM, CAPACITY, D = 2, 5, 7, 16, 128


def _unlabel(call):
    """A recorded call without the storage numbers (the extend's cache and workspace are other allocations)."""
    return json.loads(re.sub(r'"s\d+\+', '"s+', json.dumps(call)))


def _record(case, fill, monkeypatch):
    from test_decoder_launches_host import RECORDED, Recorder

    rec = Recorder()
    for name, ret in dict(RECORDED, kv_append=1, attention_extend=3).items():
        monkeypatch.setattr(ops, name, rec.entry(name, ret))
    torch.manual_seed(0)
    dec = pm.Decoder(2, D, head_dim=64, cross_attn=case["cross"], pre_norm=case["pre_norm"]).eval()
    m3 = torch.zeros(B, LM, D, dtype=torch.bfloat16) if case["cross"] else None
    cache = KVCache(dec, B, CAPACITY, m3)
    n = len(rec.calls)
    getattr(dec, fill)(torch.zeros(B, L, D, dtype=torch.bfloat16), cache)
    return rec.calls[n:]


@pytest.mark.parametrize("name", list(CASES))
def test_extend_issues_the_prefill_launches(name, monkeypatch):
    """The prefill's launches, the causal self-attention of each layer replaced by kv_append + attention_extend over
    the cache, and the memory's [k; v] projection (done once, when the cache was made) left out."""
    case = CASES[name]
    prefill = [_unlabel(c) for c in _record(case, "prefill", monkeypatch)]
    monkeypatch.undo()
    got = [_unlabel(c) for c in _record(case, "extend", monkeypatch)]
    inner = D
    qkv = f"({B},{L},{inner}) ({L * 3 * inner},{3 * inner},1) bfloat16"
    cache = f"({B},{CAPACITY},{inner}) ({CAPACITY * 2 * inner},{2 * inner},1) bfloat16"
    length = "s+0 (1) (1) int32"
    want, n_self = [], 0
    for c in prefill:
        if c[0] == "attention" and len(c[1]) > 6 and c[1][6] is True:  # the causal self-attention
            n_self += 1
            want.append(["kv_append", [f"s+{inner} ({B},{L},{2 * inner}) ({L * 3 * inner},{3 * inner},1) bfloat16",
                                       f"s+0 ({B},{CAPACITY},{2 * inner}) ({CAPACITY * 2 * inner},{2 * inner},1) "
                                       "bfloat16", length], {}])
            want.append(["attention_extend", [f"s+0 {qkv}", f"s+0 {cache}", f"s+{inner} {cache}", c[1][3], 2, 0.125,
                                              length], {}])
        elif c[0] == "linear" and c[1][0].startswith(f"s+0 ({B * LM},{D})"):  # the memory's [k; v] projection
            continue
        else:
            want.append(c)
    assert n_self == 2 and sum(c[0] == "attention" for c in want) == (2 if case["cross"] else 0)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, f"launch {i} differs:\n got  {g}\n want {w}"
