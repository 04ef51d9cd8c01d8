"""Draft-free speculative decoding on the GPU: `ops.ngram_draft` against the Python restatement of the rule (bit-exact),
a graphed n-gram round against the eager one, the generator with `NGramDraft` against the model's own greedy decoding
(GPT-2, post-norm GPT, Whisper decoder), and every round's emitted count against the count the rule predicts."""
from __future__ import annotations

import random

import numpy as np
import pytest
import torch

from conftest import build_model
from test_gpu_ragged_decode import _agree, _padded, _Tok
from test_gpu_speculative import PROMPTS, _agree_rows, _greedy_steps, _random_lm
from test_ngram_host import ngram_ref

import pytorch_models_b200 as pm
from pytorch_models_b200 import ops, speculative
from pytorch_models_b200.text import DecoderGenerator

pytestmark = pytest.mark.gpu

GARBAGE = -987654321


# ---------------------------------------------------------------------------------------------- the kernel
def _history(rng, n, kind, vocab):
    """n tokens of one kind of history, and the last token."""
    if kind == "periodic":  # the overlapping copy continues the period past the history
        p = rng.randrange(1, 6)
        unit = [rng.randrange(vocab) for _ in range(p)]
        seq = [unit[i % p] for i in range(n + 1)]
    elif kind == "planted":  # a passage repeated later, cut off inside the repeat
        seq = [rng.randrange(vocab) for _ in range(n + 1)]
        if n >= 8:
            a, span = rng.randrange(0, n // 2), rng.randrange(3, max(4, n // 3))
            at = rng.randrange(a + 1, n + 1)
            for i in range(min(span, n + 1 - at)):
                seq[at + i] = seq[a + i]
    elif kind == "nomatch":  # every token distinct
        seq = rng.sample(range(vocab, vocab + 100000), n + 1)
    else:  # a small vocabulary: matches of every length
        seq = [rng.randrange(3) for _ in range(n + 1)]
    return seq[:n], seq[n]


@pytest.mark.parametrize("B", [1, 3, 64])
@pytest.mark.parametrize("k", [1, 4, 15])
@pytest.mark.parametrize("mx,mn", [(1, 1), (3, 1), (8, 2)])
def test_ngram_draft_matches_restatement(B, k, mx, mn):
    rng = random.Random(B * 1000 + k * 10 + mx)
    cap, ld = 96, 104  # a row stride past the capacity
    kinds = ["periodic", "planted", "nomatch", "small"]
    for trial in range(4):
        if B == 1:
            lengths = [[0, 1, cap - k - 1, rng.randrange(2, cap - k)][trial]]
        else:
            lengths = [rng.choice([0, 1, cap - k - 1, rng.randrange(2, cap - k)]) for _ in range(B)]
            lengths[0], lengths[1] = 0, cap - k - 1
            if B == 64:
                lengths[2], lengths[3] = cap - k, -1  # out of range: drafts of last, no history write
        buf = torch.randint(-3, 3, (B, ld), dtype=torch.long)  # garbage past each length, tokens among them
        buf[:, cap:] = GARBAGE
        lasts = []
        for b, n in enumerate(lengths):
            row, last = _history(rng, max(n, 0), kinds[(b + trial) % 4], 1000)
            buf[b, :len(row)] = torch.tensor(row, dtype=torch.long)
            lasts.append(last)
        ids = torch.full((B, k + 1), GARBAGE, dtype=torch.long)
        ids[:, 0] = torch.tensor(lasts)
        hist, d_ids = buf.cuda(), ids.cuda()
        length = torch.tensor(lengths, dtype=torch.int32, device="cuda")
        ops.ngram_draft(hist[:, :cap], length, d_ids, k, mx, mn)
        want_hist = buf.clone()
        for b, n in enumerate(lengths):
            drafts, written = ngram_ref(buf[b].tolist(), n, lasts[b], k, mx, mn, cap)
            assert d_ids[b].tolist() == [lasts[b]] + drafts, (trial, b, n)
            if written:
                want_hist[b, n:n + k + 1] = torch.tensor([lasts[b]] + drafts)
        assert torch.equal(hist.cpu(), want_hist), trial  # nothing else written, the stride padding untouched
        assert length.tolist() == [n + k + 1 for n in lengths]


def test_ngram_draft_long_histories():
    """Capacities of 1024 and 4096: the search strides over many rows per thread; the latest occurrence wins."""
    rng = random.Random(5)
    for cap in (1024, 4096):
        B, k = 5, 8
        lengths = [cap - k - 1, cap // 2, 300, 2, 0]
        buf = torch.randint(0, 50, (B, cap), dtype=torch.long)
        lasts = [rng.randrange(50) for _ in range(B)]
        buf[0, 10:13] = torch.tensor(buf[0, lengths[0] - 2:lengths[0]].tolist() + [lasts[0]])  # an early 3-gram too
        ids = torch.zeros(B, k + 1, dtype=torch.long)
        ids[:, 0] = torch.tensor(lasts)
        hist, d_ids = buf.cuda(), ids.cuda()
        length = torch.tensor(lengths, dtype=torch.int32, device="cuda")
        ops.ngram_draft(hist, length, d_ids, k, 3, 1)
        for b, n in enumerate(lengths):
            drafts, _ = ngram_ref(buf[b].tolist(), n, lasts[b], k, 3, 1, cap)
            assert d_ids[b, 1:].tolist() == drafts, (cap, b)


# ---------------------------------------------------------------------------------------------- rounds
def _filled(target, draft, ids, lengths, cap):
    tc, hist = target.new_kv_cache(len(lengths), cap), draft.new_kv_cache(len(lengths), cap)
    x = _padded(ids, lengths)
    logits = target.prefill(x, tc, lengths=lengths)
    draft.prefill(x, hist, lengths=lengths)
    last = logits[torch.arange(len(lengths), device="cuda"), torch.tensor(lengths, device="cuda") - 1].argmax(-1)
    return tc, hist, last


def test_graphed_round_is_bit_identical_to_eager(golden):
    g = golden("gpt2")
    target = build_model(g).cuda()
    draft = pm.NGramDraft(4, 1)
    ids = torch.from_numpy(np.array(g.input)).cuda()
    ids = torch.cat([ids, ids[:1]])
    ids[2, 8:16] = ids[2, :8]  # a repeat to find
    lengths, k, budget = [5, 13, 16], 4, [30, 7, 30]
    with torch.no_grad():
        tc, th, last = _filled(target, draft, ids, lengths, 96)
        eids = torch.zeros(3, k + 1, device="cuda", dtype=torch.long)
        eids[:, 0] = last
        ebud = torch.tensor(budget, device="cuda", dtype=torch.int32)
        gt, gh, glast = _filled(target, draft, ids, lengths, 96)
        rnd = pm.SpeculativeRound(target, gt, draft, gh, k, eos=11)
        assert gt.length.tolist() == lengths and gh.length.tolist() == lengths
        rnd.start(glast, budget)
        for r in range(6):
            want = speculative.finish_round(tc, th, speculative.speculative_round(target, tc, draft, th, eids, ebud, 11))
            got = rnd()
            assert got == want, f"round {r}"
            for a, b in ((tc, gt), (th, gh)):
                assert a.seq_lengths == b.seq_lengths and a.n == b.n and a.pad == b.pad
                assert a.length.tolist() == b.length.tolist() == a.seq_lengths
            assert tc.seq_lengths == th.seq_lengths
            for s, n in enumerate(th.seq_lengths):
                assert torch.equal(th.tokens[s, :n], gh.tokens[s, :n]), f"round {r}: history of sequence {s}"
                for ka, kb in zip(tc.kv, gt.kv):
                    assert torch.equal(ka[s, :n], kb[s, :n]), f"round {r}: cache rows of sequence {s}"
            assert torch.equal(eids[:, 0], rnd.ids[:, 0]) and torch.equal(ebud, rnd.budget)
        # the history holds the prompt and every emitted token but the newest
        for s, n in enumerate(gh.seq_lengths):
            assert gh.tokens[s, :lengths[s]].tolist() == ids[s, :lengths[s]].tolist()
        # truncate both back to the prompts: a step equals one on a fresh prefill
        gt.truncate(lengths), gh.truncate(lengths)
        fresh, _, _ = _filled(target, draft, ids, lengths, 96)
        nxt = torch.stack([ids[b, n - 1] for b, n in enumerate(lengths)])
        gt.truncate([n - 1 for n in lengths]), fresh.truncate([n - 1 for n in lengths])
        assert torch.equal(target.step(nxt, gt), target.step(nxt, fresh))
        gt.reset()
        target.prefill(ids[:, :4], gt)
        with pytest.raises(ValueError, match="capture a new SpeculativeRound"):
            rnd()


def _acceptance(monkeypatch):
    rounds = []
    call = pm.graphs.SpeculativeRound.__call__

    def rec(self):
        out = call(self)
        rounds.append(out)
        return out

    monkeypatch.setattr(pm.graphs.SpeculativeRound, "__call__", rec)
    return rounds


def _predicted_counts(seq, P, k, mx, mn, eos):
    """Per round, the emitted count the drafting rule predicts for the generator's own output ``seq`` of a prompt of
    P tokens: a round that starts with history seq[:t] and last seq[t] drafts by the rule, keeps the leading drafts
    that equal the next output tokens plus the target's own token, and stops at EOS and at the end of the output."""
    counts, t = [], P
    while t + 1 < len(seq) and seq[t] != eos:
        drafts, _ = ngram_ref(seq[:t], t, seq[t], k, mx, mn, 1 << 30)
        a = 0
        while a < k and t + 1 + a < len(seq) and drafts[a] == seq[t + 1 + a] and seq[t + a] != eos:
            a += 1
        m = min(a + 1, len(seq) - 1 - t)
        counts.append(m)
        t += m
    return counts


@pytest.mark.parametrize("name", ["gpt2", "gpt"])
def test_generate_with_ngram_draft_is_greedy_and_accepts_by_the_rule(golden, name, monkeypatch):
    target = build_model(golden(name)).cuda()
    rounds = _acceptance(monkeypatch)
    gen = DecoderGenerator(target, _Tok())
    prompts = PROMPTS + ["1 2 3 4 5 1 2 3 4 5 1 2 3"]
    for k, draft in ((4, pm.NGramDraft()), (2, pm.NGramDraft(8, 2)), (8, pm.NGramDraft(1, 1))):
        for p in prompts:
            rounds.clear()
            plain = [int(t) for t in gen.generate(p, max_tokens=40, use_cache=True).split()]
            got = [int(t) for t in gen.generate(p, max_tokens=40, use_cache=True, draft=draft,
                                                draft_tokens=k).split()]
            assert len(got) == len(plain) == len(p.split()) + 40
            _agree(target, plain, got)
            pred = _predicted_counts(got, len(p.split()), k, draft.max_ngram, draft.min_ngram, -1)
            assert [len(r[0]) for r in rounds] == pred, (k, p)
        rounds.clear()
        batch = gen.generate_batch(prompts, max_tokens=40, draft=draft, draft_tokens=k)
        plain = gen.generate_batch(prompts, max_tokens=40)
        for b, (p, a, s) in enumerate(zip(prompts, plain, batch)):
            a, s = [int(t) for t in a.split()], [int(t) for t in s.split()]
            assert len(a) == len(s) == len(p.split()) + 40
            _agree(target, a, s)
            pred = _predicted_counts(s, len(p.split()), k, draft.max_ngram, draft.min_ngram, -1)
            assert [len(r[b]) for r in rounds if r[b]] == pred, (k, p)
    acc = sum(len(r[0]) for r in rounds) / max(1, len(rounds))
    print(f"{name}: mean tokens per round {acc:.2f}")


def test_ngram_draft_stops_each_sequence_at_its_eos(golden, monkeypatch):
    target = build_model(golden("gpt2")).cuda()
    prompts = PROMPTS[:3] + ["4 4 4 4 4 4"]
    free = [[int(t) for t in s.split()] for s in DecoderGenerator(target, _Tok()).generate_batch(prompts, 12)]
    eos = free[0][len(prompts[0].split()) + 3]
    gen = DecoderGenerator(target, _Tok(eos))
    rounds = _acceptance(monkeypatch)
    for k in (1, 4):
        rounds.clear()
        draft = pm.NGramDraft()
        got = [[int(t) for t in s.split()] for s in gen.generate_batch(prompts, 12, draft=draft, draft_tokens=k)]
        for b, (p, f, g_) in enumerate(zip(prompts, free, got)):
            n = len(p.split())
            new = f[n:]
            want = f[:n + new.index(eos) + 1] if eos in new else f
            assert g_ == want, (k, p, f, g_)
            assert [len(r[b]) for r in rounds if r[b]] == _predicted_counts(g_, n, k, 3, 1, eos), (k, p)
    draft = pm.NGramDraft()
    one = gen.generate_batch(prompts, max_tokens=1, draft=draft)
    assert [len(s.split()) for s in one] == [len(p.split()) + 1 for p in prompts]
    assert gen.generate_batch(prompts, max_tokens=0, draft=draft) == prompts
    assert gen.generate(prompts[0], max_tokens=0, use_cache=True, draft=draft) == prompts[0]
    assert len(gen.generate(prompts[1], max_tokens=1, use_cache=True, draft=draft).split()) == 2


def test_tail_runs_into_the_position_table():
    """max_seq_len 64: prompts of 3..20 tokens plus 45 new ones reach the last position, so the rounds stop and the
    target's plain steps finish."""
    target = _random_lm(pm.GPT2, 777, 2, 64, 7, max_seq_len=64)
    gen = DecoderGenerator(target, _Tok())
    prompts = [" ".join(str(3 + i % 7) for i in range(20)), "7 8 9"]
    plain = gen.generate_batch(prompts, max_tokens=45)
    for k in (4, 8):
        got = gen.generate_batch(prompts, max_tokens=45, draft=pm.NGramDraft(), draft_tokens=k)
        for a, b in zip(plain, got):
            _agree(target, [int(t) for t in a.split()], [int(t) for t in b.split()])
        one = gen.generate(prompts[0], max_tokens=45, use_cache=True, draft=pm.NGramDraft(), draft_tokens=k)
        _agree(target, [int(t) for t in plain[0].split()], [int(t) for t in one.split()])


def _rounds(target, tc, draft, hist, last, k, n):
    rnd = pm.SpeculativeRound(target, tc, draft, hist, k)
    rnd.start(last, [n] * tc.batch)
    out = [[t] for t in last.tolist()]
    while any(len(o) < n + 1 for o in out):
        for b, toks in enumerate(rnd()):
            out[b] += toks
    return out


def test_whisper_decoder_round(golden):
    g = golden("whisper_full")
    m = build_model(g).cuda()
    target = m.decoder
    x = torch.from_numpy(np.array(g.input)).cuda()
    prompt = torch.from_numpy(np.array(g.extra["targets"])).cuda()[:, :6]
    prompt[1, 3:6] = prompt[1, :3]
    n, lengths = 20, [4, 6]
    draft = pm.NGramDraft()
    with torch.no_grad():
        memory = m.encoder(x)
        caches = []
        for _ in range(2):
            tc, hist = target.new_kv_cache(memory, 64), draft.new_kv_cache(2, 64)
            xp = _padded(prompt, lengths)
            logits = target.prefill(xp, tc, lengths=lengths)
            draft.prefill(xp, hist, lengths=lengths)
            caches.append((tc, hist, logits[torch.arange(2, device="cuda"), torch.tensor(lengths, device="cuda") - 1]
                           .argmax(-1)))
        tc, hist, last = caches[0]
        got = _rounds(target, tc, draft, hist, last, 4, n)
        pc, _, plast = caches[1]
        toks, rows = _greedy_steps(target, pc, plast, n)
    for b in range(2):
        plain = [t[b] for t in toks] + [int(rows[-1][b].argmax())]
        _agree_rows(plain[1:], [r[b] for r in rows], got[b][1:n + 1], f"Whisper sequence {b}")
