"""Host-side checks of greedy speculative decoding (no GPU needed): the argument checks of b200enc_argmax_rows and
b200enc_speculative_accept, the refusals of a round and of the generator (each before any launch), the host mirror
after `KVCache.truncate`, and the launches of one eager round."""
from __future__ import annotations

import pytest
import torch

import pytorch_models_b200 as pm
from pytorch_models_b200 import _lib, ops, speculative
from pytorch_models_b200.text import DecoderGenerator
from pytorch_models_b200.transformer import KVCache

A = 0x10000  # a 16-byte aligned fake device address: every call below fails its checks before touching it


def _argmax(**over):
    lib = _lib.load()
    a = dict(logits=A, ld=50264, rows=5, V=50257, out=A, out_stride=5)
    a.update(over)
    rc = lib.b200enc_argmax_rows(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    (dict(logits=None), "null pointer"),
    (dict(out=None), "null pointer"),
    (dict(rows=0), "rows=0"),
    (dict(V=0), "V=0"),
    (dict(ld=50256), "ld=50256 is smaller than V=50257"),
    (dict(ld=50265), "ld=50265"),
    (dict(logits=A + 8), "16-byte aligned"),
    (dict(out_stride=0), "out_stride=0"),
    (dict(out=A + 4), "8-byte aligned"),
])
def test_argmax_rows_argument_checks(over, needle):
    rc, msg = _argmax(**over)
    assert rc == -1 and needle in msg and msg.startswith("b200enc_argmax_rows:"), msg


def _accept(**over):
    lib = _lib.load()
    a = dict(picks=A, ids=A, budget=A, eos=-1, len_t=A, st=1, len_d=A, sd=1, emitted=A, n_emitted=A, out_stride=6,
             B=3, k=4)
    a.update(over)
    rc = lib.b200enc_speculative_accept(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    (dict(picks=None), "null pointer"),
    (dict(ids=None), "null pointer"),
    (dict(budget=None), "null pointer"),
    (dict(len_t=None), "null pointer"),
    (dict(len_d=None), "null pointer"),
    (dict(emitted=None), "null pointer"),
    (dict(n_emitted=None), "null pointer"),
    (dict(B=0), "B=0"),
    (dict(k=0), "k=0"),
    (dict(k=16), "k=16"),
    (dict(st=0), "target_len_stride=0"),
    (dict(sd=2), "draft_len_stride=2"),
    (dict(out_stride=4), "out_stride=4 is smaller than k+1=5"),
    (dict(eos=-2), "eos=-2"),
])
def test_speculative_accept_argument_checks(over, needle):
    rc, msg = _accept(**over)
    assert rc == -1 and needle in msg and msg.startswith("b200enc_speculative_accept:"), msg


def test_shared_length_is_accepted_with_one_sequence():
    rc, msg = _accept(B=1, st=0, sd=0, out_stride=0, k=16)  # fails on k only: the strides of B = 1 are fine
    assert rc == -1 and "k=16" in msg, msg


def test_ops_refuse_bad_views():
    ops_dev = ops._need_cuda
    try:
        ops._need_cuda = lambda *ts: torch.device("cpu")
        logits = torch.zeros(3, 16, dtype=torch.bfloat16)
        with pytest.raises(TypeError, match="logits must be torch.bfloat16"):
            ops.argmax_rows(logits.float(), torch.zeros(3, dtype=torch.long))
        with pytest.raises(ValueError, match="unit inner stride"):
            ops.argmax_rows(logits.t(), torch.zeros(16, dtype=torch.long))
        with pytest.raises(ValueError, match=r"out must be a \(3,\) view"):
            ops.argmax_rows(logits, torch.zeros(4, dtype=torch.long))
        ids = torch.zeros(2, 5, dtype=torch.long)
        res = torch.zeros(2, 6, dtype=torch.long)
        one = torch.zeros(1, dtype=torch.int32)
        with pytest.raises(ValueError, match=r"budget must be a contiguous \(2,\)"):
            ops.speculative_accept(ids, ids, torch.zeros(3, dtype=torch.int32), -1, one, one, res[:, :5], res[:, 5])
        with pytest.raises(ValueError, match="same row stride"):
            ops.speculative_accept(ids, ids, torch.zeros(2, dtype=torch.int32), -1, one, one, res[:, :5],
                                   torch.zeros(2, dtype=torch.long))
        with pytest.raises(ValueError, match="1 or 2 elements"):
            ops.speculative_accept(ids, ids, torch.zeros(2, dtype=torch.int32), -1, torch.zeros(3, dtype=torch.int32),
                                   one, res[:, :5], res[:, 5])
    finally:
        ops._need_cuda = ops_dev


# ---------------------------------------------------------------------------------------------- refusals
ENTRY_POINTS = ("linear", "attention", "attention_decode", "row_stats", "layernorm", "decode_advance", "kv_append",
                "attention_extend", "embed_rows", "embed_rows_at", "argmax_rows", "speculative_accept")


@pytest.fixture
def launches(monkeypatch):
    calls = []
    for name in ENTRY_POINTS:
        monkeypatch.setattr(ops, name, lambda *a, _n=name, **k: calls.append(_n))
    return calls


class FakeCuda(torch.Tensor):  # a tensor that reports a CUDA device, so no GPU is needed to see the refusal
    @property
    def is_cuda(self):
        return True


def _lm(vocab=96, layers=1, cls=pm.GPT2, **kw):
    return type("SmallLM", (cls,), dict(vocab_size=vocab))(layers, 64, **kw).eval()


def _pair(B=2, cap=16, ragged=True, **target_kw):
    target, draft = _lm(**target_kw), _lm()
    tc, dc = target.new_kv_cache(B, cap), draft.new_kv_cache(B, cap)
    if ragged:
        for c in (tc, dc):
            c.store_lengths([3, 5][:B] if B == 2 else [4] * B)
    return target, tc, draft, dc


def _ids(B, k):
    return torch.zeros(B, k + 1, dtype=torch.long).as_subclass(FakeCuda)


def _budget(B):
    return torch.zeros(B, dtype=torch.int32)


@pytest.mark.parametrize("make,match", [
    (lambda t, tc, d, dc: speculative.speculative_round(t, tc, _lm(vocab=97), dc, _ids(2, 4), _budget(2)),
     "vocabulary of 97 tokens differs from the target's 96"),
    (lambda t, tc, d, dc: speculative.speculative_round(t, tc, d, d.new_kv_cache(3, 16), _ids(2, 4), _budget(2)),
     "target cache holds 2 sequences, the draft cache 3"),
    (lambda t, tc, d, dc: speculative.speculative_round(t, tc, d, dc, _ids(2, 0), _budget(2)), "k=0"),
    (lambda t, tc, d, dc: speculative.speculative_round(t, tc, d, dc, _ids(2, 16), _budget(2)), "k=16"),
    (lambda t, tc, d, dc: speculative.speculative_round(t, t.new_kv_cache(2, 16), d, dc, _ids(2, 4), _budget(2)),
     "target cache holds one shared length for a batch of 2"),
    (lambda t, tc, d, dc: speculative.speculative_round(t, tc, d, dc, _ids(2, 11), _budget(2)),
     "k=11 draft tokens writes 12 rows past the 5 tokens the target cache holds, more than its capacity of 16"),
    (lambda t, tc, d, dc: speculative.speculative_round(t.train(), tc, d, dc, _ids(2, 4), _budget(2)), "dropout"),
    (lambda t, tc, d, dc: speculative.speculative_round(t, tc, d, dc, _ids(3, 4), _budget(3)), "ids hold 3"),
    (lambda t, tc, d, dc: pm.SpeculativeRound(t, tc, d, dc, 16), "k=16"),
    (lambda t, tc, d, dc: pm.SpeculativeRound(t, tc, _lm(vocab=97), dc, 4), "vocabulary"),
])
def test_round_refusals_come_before_any_launch(make, match, launches):
    target, tc, draft, dc = _pair(dropout=0.1)
    exc = NotImplementedError if match == "dropout" else ValueError
    with pytest.raises(exc, match=match):
        make(target, tc, draft, dc)
    assert launches == [] and tc.seq_lengths == [3, 5] and dc.seq_lengths == [3, 5]


def test_one_sequence_may_hold_a_shared_length(launches):
    target, tc, draft, dc = _pair(B=1, cap=8, ragged=False)
    tc.store_lengths([3]), dc.store_lengths([3])
    speculative.check_round(target, tc, draft, dc, 4)
    with pytest.raises(ValueError, match="draft cache holds 3 of|the 3 tokens the target cache holds"):
        speculative.check_round(target, tc, draft, dc, 5)
    assert launches == [] and not tc.ragged


class _Tok:
    eos_token_id = None

    def encode(self, s):
        return [int(t) for t in s.split()]

    def decode(self, ids):
        return " ".join(map(str, ids))


@pytest.mark.parametrize("call,exc,match", [
    (lambda g, d: g.generate("1 2", 4, topk=3, use_cache=True, draft=d), NotImplementedError, "topk=3"),
    (lambda g, d: g.generate("1 2", 4, draft=d), ValueError, "use_cache=True"),
    (lambda g, d: g.generate_batch(["1 2"], 4, topk=2, draft=d), NotImplementedError, "topk=2"),
    (lambda g, d: g.generate("1 2", 4, use_cache=True, draft=_lm(vocab=97)), ValueError, "vocabulary"),
    (lambda g, d: g.generate_batch(["1 2", "3"], 4, draft=d, draft_tokens=0), ValueError, "k=0"),
])
def test_generator_refusals_come_before_any_launch(call, exc, match, launches):
    gen = DecoderGenerator(_lm(), _Tok())
    with pytest.raises(exc, match=match):
        call(gen, _lm())
    assert launches == []


# ---------------------------------------------------------------------------------------------- truncate
def test_truncate_host_mirror(launches):
    dec = pm.Decoder(1, 64).eval()
    cache = KVCache(dec, 3, 32, None)
    dec.extend(torch.zeros(3, 6, 64, dtype=torch.bfloat16), cache)
    cache.truncate([4, 4, 4])  # equal lengths keep one shared length
    assert not cache.ragged and cache.length is cache.shared_length and cache.length.tolist() == [4] and cache.n == 4
    cache.truncate(torch.tensor([4, 1, 0]))  # unequal lengths: per-sequence
    assert cache.ragged and cache.length is cache.seq_length and cache.length.tolist() == [4, 1, 0]
    assert cache.seq_lengths == [4, 1, 0] and cache.n == 4 and cache.pad == [0, 3, 4]
    cache.truncate([2, 1, 0])  # a ragged cache stays ragged
    assert cache.ragged and cache.seq_lengths == [2, 1, 0] and cache.pad == [0, 1, 2]
    dec.extend(torch.zeros(3, 2, 64, dtype=torch.bfloat16), cache)
    assert cache.seq_lengths == [4, 3, 2] and cache.length.tolist() == [4, 3, 2]
    assert "decode_advance" not in launches  # the lengths come from the host, as after an extend


@pytest.mark.parametrize("lengths,match", [
    ([5, 3], r"length 5 of sequence 0 is outside \[0, 4\]"),
    ([4, 7], r"length 7 of sequence 1 is outside \[0, 6\]"),
    ([-1, 0], r"length -1 of sequence 0"),
    ([1], "1 entries for a batch of 2"),
    (torch.tensor([1, 1]).as_subclass(FakeCuda), "not a CUDA tensor"),
])
def test_truncate_refusals(lengths, match):
    dec = pm.Decoder(1, 64).eval()
    cache = KVCache(dec, 2, 32, None)
    cache.store_lengths([4, 6])
    with pytest.raises(ValueError, match=match):
        cache.truncate(lengths)
    assert cache.seq_lengths == [4, 6] and cache.length.tolist() == [4, 6]


# ---------------------------------------------------------------------------------------------- launch list
@pytest.mark.parametrize("k", [1, 4])
@pytest.mark.parametrize("cls", [pm.GPT2, pm.GPT])
def test_round_launches(k, cls, monkeypatch):
    """k + 1 draft steps (each a `step`'s launches; all but the last followed by the logits GEMM and argmax_rows into
    column j + 1 of the ids), the launches of the target's `extend` with decode_advance by k + 1 after its layers,
    argmax_rows over the B·(k+1) verify rows, speculative_accept."""
    from test_decoder_launches_host import RECORDED, Recorder

    B, V = 2, 90  # the logits rows are 96 columns apart
    target, draft = _lm(V, 2, cls), _lm(V, cls=cls)
    rec = Recorder()
    extra = dict(kv_append=1, attention_extend=3, embed_rows_at=4, argmax_rows=1, speculative_accept=6)
    for name, ret in dict(RECORDED, **extra).items():
        monkeypatch.setattr(ops, name, rec.entry(name, ret))
    names = lambda calls: [c[0] for c in calls]  # noqa: E731

    ref_cache = draft.new_kv_cache(B, 32)
    ref_cache.store_lengths([3, 5])
    n = len(rec.calls)
    draft.step(torch.zeros(B, dtype=torch.long).as_subclass(FakeCuda), ref_cache)
    step = names(rec.calls[n:])
    tref = target.new_kv_cache(B, 32)
    tref.store_lengths([3, 5])
    n = len(rec.calls)
    target.extend(_ids(B, k), tref)
    extend = names(rec.calls[n:])

    t, tc, d, dc = target, target.new_kv_cache(B, 32), draft, draft.new_kv_cache(B, 32)
    tc.store_lengths([3, 5]), dc.store_lengths([3, 5])
    n = len(rec.calls)
    speculative.speculative_round(t, tc, d, dc, _ids(B, k), _budget(B), eos=7)
    got = rec.calls[n:]
    assert tc.seq_lengths == [3, 5] and dc.seq_lengths == [3, 5]  # the mirrors wait for finish_round

    layers = len(extend) - 2  # extend = embed_rows_at, the layers' launches, the logits GEMM
    want = (step + ["argmax_rows"]) * k + step[:-1] + extend[:1 + layers] + ["decode_advance"] + extend[-1:] + \
        ["argmax_rows", "speculative_accept"]
    assert names(got) == want
    assert step[-1] == "linear" and extend[-1] == "linear"
    picks = [c for c in got if c[0] == "argmax_rows"]
    for j, c in enumerate(picks[:-1]):
        assert c[1][0].endswith(f"({B},{V}) ({((V + 7) // 8) * 8},1) bfloat16"), c  # the bf16 rows, padded stride
        assert c[1][1].endswith(f"+{j + 1} ({B}) ({k + 1}) int64"), c  # column j + 1 of the ids
    assert picks[-1][1][0].endswith(f"({B * (k + 1)},{V}) ({((V + 7) // 8) * 8},1) bfloat16")
    adv = [c for c in got if c[0] == "decode_advance"]
    assert len(adv) == k + 2 and all(len(c[1]) == 1 for c in adv[:-1]) and adv[-1][1][1] == k + 1
    assert adv[-1][1][0] != adv[0][1][0]  # the verify advances the target's lengths, the steps the draft's
    acc = got[-1][1]
    assert acc[3] == 7 and acc[4].endswith(f"({B}) (1) int32") and acc[6] == f"{acc[6][:acc[6].index('+')]}+0 " \
        f"({B},{k + 1}) ({k + 2},1) int64" and acc[7].split(" ")[0].endswith(f"+{k + 1}")
