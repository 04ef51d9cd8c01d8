"""Host-side checks of draft-free speculative decoding (no GPU needed): the argument checks of b200enc_ngram_draft, the
range refusals of `NGramDraft`, the refusals of a round and of the generator (each before any launch), the token
history's host mirror, the launches of one n-gram round, and the Python restatement of the drafting rule that
test_gpu_ngram.py holds the kernel to."""
from __future__ import annotations

import pytest
import torch

import pytorch_models_b200 as pm
from pytorch_models_b200 import _lib, ops, speculative
from pytorch_models_b200.speculative import NGramDraft, TokenHistory
from pytorch_models_b200.text import DecoderGenerator
from test_speculative_host import A, _budget, _ids, _lm, _Tok


def ngram_ref(row, n, last, k, max_ngram, min_ngram, capacity):
    """The drafts of one sequence, restated from the rule: (drafts, whether the history is written)."""
    if not 0 <= n <= capacity - k - 1:
        return [last] * k, False
    s = list(row[:n]) + [last]
    for g in range(max_ngram, min_ngram - 1, -1):
        if g > n:
            continue
        suffix = s[n - g + 1:]
        e = next((e for e in range(n - 1, g - 2, -1) if s[e - g + 1:e + 1] == suffix), None)
        if e is not None:
            for i in range(1, k + 1):  # the overlapping copy: s' is s followed by the drafts
                s.append(s[e + i])
            return s[n + 1:], True
    return [last] * k, True


@pytest.mark.parametrize("row,last,k,mx,mn,want", [
    ([1, 2, 3, 9, 1, 2], 3, 3, 3, 1, [9, 1, 2]),  # 1 2 3 occurs at the start: what followed it
    ([5, 6, 7, 5, 6, 7, 5, 6], 7, 7, 3, 1, [5, 6, 7, 5, 6, 7, 5]),  # period 3 continues past the history
    ([4, 4, 4], 4, 4, 2, 1, [4, 4, 4, 4]),  # period 1
    ([1, 2, 3], 8, 2, 3, 1, [8, 8]),  # no match: last repeated
    ([7, 1, 7, 2, 7], 3, 2, 3, 1, [3, 3]),  # 3 never occurred
    ([7, 1, 7, 2, 9, 7], 7, 2, 3, 1, [7, 7]),  # the latest earlier "7" ends right before last: period 1
    ([7, 1, 7, 2, 9, 7], 2, 2, 3, 1, [9, 7]),  # "7 2" occurred once
    ([1, 2, 9, 2], 5, 2, 3, 2, [5, 5]),  # min_ngram 2: "2 5" never occurred
    ([1, 2, 9, 1, 2], 9, 3, 2, 1, [1, 2, 9]),  # "2 9" beats the later "9"
    ([], 4, 3, 3, 1, [4, 4, 4]),  # an empty history
])
def test_reference_rule_on_hand_made_rows(row, last, k, mx, mn, want):
    got, written = ngram_ref(row, len(row), last, k, mx, mn, 64)
    assert got == want and written


def test_reference_refuses_bad_lengths():
    assert ngram_ref([1] * 10, 7, 3, 4, 3, 1, 11) == ([3] * 4, False)  # 7 > capacity - k - 1 = 6
    assert ngram_ref([1] * 10, 6, 3, 4, 3, 1, 11)[1]
    assert ngram_ref([1] * 10, -1, 3, 4, 3, 1, 11) == ([3] * 4, False)


# ---------------------------------------------------------------------------------------------- argument checks
def _draft(**over):
    lib = _lib.load()
    a = dict(hist=A, ld=64, capacity=64, len=A, len_stride=1, ids=A, B=3, k=4, max_ngram=3, min_ngram=1)
    a.update(over)
    rc = lib.b200enc_ngram_draft(*a.values(), None)
    return rc, lib.b200enc_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    (dict(hist=None), "null pointer"),
    (dict(len=None), "null pointer"),
    (dict(ids=None), "null pointer"),
    (dict(B=0), "B=0"),
    (dict(k=0), "k=0"),
    (dict(k=16), "k=16"),
    (dict(min_ngram=0), "min_ngram=0"),
    (dict(min_ngram=4), "min_ngram=4 and max_ngram=3"),
    (dict(max_ngram=9), "max_ngram=9"),
    (dict(len_stride=0), "len_stride=0"),
    (dict(len_stride=2), "len_stride=2"),
    (dict(capacity=4), "capacity=4 cannot hold the k+1=5 rows"),
    (dict(ld=63), "hist_stride=63 is smaller than capacity=64"),
    (dict(hist=A + 4), "8-byte aligned"),
    (dict(ids=A + 2), "8-byte aligned"),
])
def test_ngram_draft_argument_checks(over, needle):
    rc, msg = _draft(**over)
    assert rc == -1 and needle in msg and msg.startswith("b200enc_ngram_draft:"), msg


def test_shared_length_is_accepted_with_one_sequence():
    rc, msg = _draft(B=1, len_stride=0, ld=0, k=16)  # fails on k only: stride 0 and a zero row stride are fine at B 1
    assert rc == -1 and "k=16" in msg, msg


def test_ops_refuses_bad_views():
    ops_dev = ops._need_cuda
    try:
        ops._need_cuda = lambda *ts: torch.device("cpu")
        hist = torch.zeros(2, 32, dtype=torch.long)
        ids = torch.zeros(2, 5, dtype=torch.long)
        two = torch.zeros(2, dtype=torch.int32)
        with pytest.raises(TypeError, match="hist must be torch.int64"):
            ops.ngram_draft(hist.int(), two, ids, 4, 3, 1)
        with pytest.raises(TypeError, match="length must be torch.int32"):
            ops.ngram_draft(hist, two.long(), ids, 4, 3, 1)
        with pytest.raises(ValueError, match="unit inner stride"):
            ops.ngram_draft(hist.t(), two, ids, 4, 3, 1)
        with pytest.raises(ValueError, match=r"ids must be a contiguous \(2, 5\)"):
            ops.ngram_draft(hist, two, ids[:, :4], 4, 3, 1)
        with pytest.raises(ValueError, match="1 or 2 elements"):
            ops.ngram_draft(hist, torch.zeros(3, dtype=torch.int32), ids, 4, 3, 1)
    finally:
        ops._need_cuda = ops_dev


@pytest.mark.parametrize("mx,mn", [(3, 0), (2, 3), (9, 1), (0, 0)])
def test_ngram_draft_range_refusals(mx, mn):
    with pytest.raises(ValueError, match=f"min_ngram={mn} and max_ngram={mx} must satisfy"):
        NGramDraft(max_ngram=mx, min_ngram=mn)


def test_defaults_and_extremes():
    d = NGramDraft()
    assert (d.max_ngram, d.min_ngram) == (3, 1)
    assert (NGramDraft(8, 8).max_ngram, NGramDraft(1, 1).min_ngram) == (8, 1)
    with pytest.raises(ValueError, match="batch=0"):
        d.new_kv_cache(0, 8, device="cpu")


# ---------------------------------------------------------------------------------------------- history mirror
def test_history_host_mirror():
    d = NGramDraft()
    h = d.new_kv_cache(3, 32, device="cpu")
    assert isinstance(h, TokenHistory) and h.n == 0 and not h.ragged and h.tokens.shape == (3, 32)
    d.prefill(torch.tensor([[1, 2, 3, 4], [5, 6, 0, 0], [7, 0, 0, 0]]), h, lengths=[4, 2, 1])
    assert h.ragged and h.length is h.seq_length and h.length.tolist() == [4, 2, 1]
    assert h.seq_lengths == [4, 2, 1] and h.n == 4 and h.pad == [0, 2, 3]
    assert h.tokens[0, :4].tolist() == [1, 2, 3, 4] and h.tokens[1, :2].tolist() == [5, 6] and h.tokens[2, 0] == 7
    with pytest.raises(ValueError, match="prefill needs an empty cache"):
        d.prefill(torch.tensor([[1], [2], [3]]), h)
    h.truncate([2, 2, 1])
    assert h.seq_lengths == [2, 2, 1] and h.length.tolist() == [2, 2, 1] and h.n == 2 and h.pad == [0, 0, 1]
    h.store_lengths([7, 5, 2], device=False)  # as after a round: the accept kernel already wrote the device lengths
    assert h.seq_lengths == [7, 5, 2] and h.n == 7 and h.pad == [0, 2, 5] and h.length.tolist() == [2, 2, 1]
    with pytest.raises(ValueError, match=r"length 8 of sequence 0 is outside \[0, 7\]"):
        h.truncate([8, 0, 0])
    h.reset()
    assert h.n == 0 and not h.ragged and h.length is h.shared_length and h.length.tolist() == [0]

    one = d.new_kv_cache(1, 8, device="cpu")
    d.prefill(torch.tensor([9, 8, 7]), one)  # one prompt, (P,) ids: a shared length
    assert not one.ragged and one.length.tolist() == [3] and one.n == 3 and one.tokens[0, :3].tolist() == [9, 8, 7]
    one.truncate([1])
    assert not one.ragged and one.length.tolist() == [1] and one.seq_lengths == [1]
    with pytest.raises(ValueError, match=r"length 4 is outside \[1, 3\]"):
        d.prefill(torch.tensor([[1, 2, 3]] * 3), d.new_kv_cache(3, 8, device="cpu"), lengths=[1, 4, 2])
    with pytest.raises(ValueError, match="prefill of 9 tokens into a cache of capacity 8"):
        d.prefill(torch.zeros(9, dtype=torch.long), d.new_kv_cache(1, 8, device="cpu"))


# ---------------------------------------------------------------------------------------------- refusals
ENTRY_POINTS = ("linear", "attention", "attention_decode", "row_stats", "layernorm", "decode_advance", "kv_append",
                "attention_extend", "embed_rows", "embed_rows_at", "argmax_rows", "speculative_accept", "ngram_draft")


@pytest.fixture
def launches(monkeypatch):
    calls = []
    for name in ENTRY_POINTS:
        monkeypatch.setattr(ops, name, lambda *a, _n=name, **k: calls.append(_n))
    return calls


def _filled(B=2, cap=16, hcap=16, ragged=True, **target_kw):
    target = _lm(**target_kw)
    tc, hist = target.new_kv_cache(B, cap), NGramDraft().new_kv_cache(B, hcap, device="cpu")
    if ragged:
        for c in (tc, hist):
            c.store_lengths([3, 5][:B] if B == 2 else [4] * B)
    return target, tc, hist


N = NGramDraft()
R = speculative.speculative_round


@pytest.mark.parametrize("make,match", [
    (lambda t, tc, h: R(t, tc, N, h, _ids(2, 0), _budget(2)), "k=0"),
    (lambda t, tc, h: R(t, tc, N, h, _ids(2, 16), _budget(2)), "k=16"),
    (lambda t, tc, h: R(t, t.new_kv_cache(2, 16), N, h, _ids(2, 4), _budget(2)),
     "target cache holds one shared length for a batch of 2"),
    (lambda t, tc, h: R(t, tc, N, N.new_kv_cache(2, 16, device="cpu"), _ids(2, 4), _budget(2)),
     "draft cache holds one shared length for a batch of 2"),
    (lambda t, tc, h: R(t, tc, N, N.new_kv_cache(3, 16, device="cpu"), _ids(2, 4), _budget(2)),
     "target cache holds 2 sequences, the draft cache 3"),
    (lambda t, tc, h: R(t, tc, N, h, _ids(2, 11), _budget(2)),
     "k=11 draft tokens writes 12 rows past the 5 tokens the target cache holds, more than its capacity of 16"),
    (lambda t, tc, h: R(t.train(), tc, N, h, _ids(2, 4), _budget(2)), "dropout"),
    (lambda t, tc, h: R(t, tc, N, h, _ids(3, 4), _budget(3)), "ids hold 3"),
    (lambda t, tc, h: R(t, tc, N, t.new_kv_cache(2, 16), _ids(2, 4), _budget(2)),
     "NGramDraft with a KVCache"),
    (lambda t, tc, h: R(t, tc, _lm(), h, _ids(2, 4), _budget(2)), "with a TokenHistory"),
    (lambda t, tc, h: pm.SpeculativeRound(t, tc, N, h, 16), "k=16"),
    (lambda t, tc, h: pm.SpeculativeRound(t.train(), tc, N, h, 4), "dropout"),
])
def test_round_refusals_come_before_any_launch(make, match, launches):
    target, tc, hist = _filled(dropout=0.1)
    exc = NotImplementedError if match == "dropout" else ValueError
    with pytest.raises(exc, match=match):
        make(target, tc, hist)
    assert launches == [] and tc.seq_lengths == [3, 5] and hist.seq_lengths == [3, 5]


def test_history_without_room_is_refused(launches):
    target, tc, hist = _filled(hcap=9)
    with pytest.raises(ValueError, match="writes 5 rows past the 5 tokens the draft cache holds, more than its "
                                         "capacity of 9"):
        R(target, tc, N, hist, _ids(2, 4), _budget(2))
    speculative.check_round(target, tc, N, hist, 3)  # 5 + 4 rows fit
    assert launches == []


@pytest.mark.parametrize("call,exc,match", [
    (lambda g: g.generate("1 2", 4, topk=3, use_cache=True, draft=N), NotImplementedError, "topk=3"),
    (lambda g: g.generate("1 2", 4, draft=N), ValueError, "use_cache=True"),
    (lambda g: g.generate_batch(["1 2"], 4, topk=2, draft=N), NotImplementedError, "topk=2"),
    (lambda g: g.generate_batch(["1 2", "3"], 4, draft=N, draft_tokens=0), ValueError, "k=0"),
    (lambda g: g.generate("1 2", 4, use_cache=True, draft=N, draft_tokens=16), ValueError, "k=16"),
])
def test_generator_refusals_come_before_any_launch(call, exc, match, launches):
    gen = DecoderGenerator(_lm(), _Tok())
    with pytest.raises(exc, match=match):
        call(gen)
    assert launches == []


def test_generator_refuses_a_model_that_cannot_decode(launches):
    gen = DecoderGenerator(_lm(dropout=0.1).train(), _Tok())
    with pytest.raises(NotImplementedError, match="dropout"):
        gen.generate("1 2", 4, use_cache=True, draft=N)
    assert launches == []


# ---------------------------------------------------------------------------------------------- launch list
@pytest.mark.parametrize("k", [1, 4])
@pytest.mark.parametrize("cls", [pm.GPT2, pm.GPT])
def test_round_launches(k, cls, monkeypatch):
    """One ngram_draft launch, the launches of the target's `extend` with decode_advance by k + 1 after its layers,
    argmax_rows over the B·(k+1) verify rows, and speculative_accept with the history's length as the draft length.
    No draft-model launch."""
    from test_decoder_launches_host import RECORDED, Recorder

    B, V = 2, 90  # the logits rows are 96 columns apart
    target = _lm(V, 2, cls)
    rec = Recorder()
    extra = dict(kv_append=1, attention_extend=3, embed_rows_at=4, argmax_rows=1, speculative_accept=6, ngram_draft=2)
    for name, ret in dict(RECORDED, **extra).items():
        monkeypatch.setattr(ops, name, rec.entry(name, ret))
    names = lambda calls: [c[0] for c in calls]  # noqa: E731

    tref = target.new_kv_cache(B, 32)
    tref.store_lengths([3, 5])
    n = len(rec.calls)
    target.extend(_ids(B, k), tref)
    extend = names(rec.calls[n:])

    draft = NGramDraft(4, 2)
    tc, hist = target.new_kv_cache(B, 32), draft.new_kv_cache(B, 24, device="cpu")
    tc.store_lengths([3, 5]), hist.store_lengths([3, 5])
    ids = _ids(B, k)
    n = len(rec.calls)
    speculative.speculative_round(target, tc, draft, hist, ids, _budget(B), eos=7)
    got = rec.calls[n:]
    assert tc.seq_lengths == [3, 5] and hist.seq_lengths == [3, 5]  # the mirrors wait for finish_round

    layers = len(extend) - 2  # extend = embed_rows_at, the layers' launches, the logits GEMM
    want = ["ngram_draft"] + extend[:1 + layers] + ["decode_advance"] + extend[-1:] + ["argmax_rows",
                                                                                        "speculative_accept"]
    assert names(got) == want
    hist_len, ids_arg = rec._arg(hist.length), rec._arg(ids)
    assert got[0][1] == [rec._arg(hist.tokens), hist_len, ids_arg, k, 4, 2]
    assert hist_len.endswith(f"({B}) (1) int32") and rec._arg(hist.tokens).endswith(f"({B},24) (24,1) int64")
    adv = [c for c in got if c[0] == "decode_advance"]
    assert len(adv) == 1 and adv[0][1] == [rec._arg(tc.length), k + 1]
    assert got[-2][1][0].endswith(f"({B * (k + 1)},{V}) ({((V + 7) // 8) * 8},1) bfloat16")
    acc = got[-1][1]
    assert acc[1] == ids_arg and acc[3] == 7 and acc[4] == rec._arg(tc.length) and acc[5] == hist_len
