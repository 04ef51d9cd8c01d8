"""Greedy speculative decoding on the GPU: `ops.argmax_rows` against torch.argmax, `ops.speculative_accept` against a
Python restatement of the acceptance, `KVCache.truncate`, a graphed round against the eager one, and the generator
with a draft against the model's own greedy decoding (GPT-2, post-norm GPT, Whisper decoder)."""
from __future__ import annotations

import copy
import random

import numpy as np
import pytest
import torch

from conftest import build_model
from oracle import oracle_torch
from test_gpu_kv_cache import MAX_ABS_12, _assert_logits
from test_gpu_ragged_decode import _agree, _padded, _Tok

import pytorch_models_b200 as pm
from pytorch_models_b200 import ops, speculative
from pytorch_models_b200.text import DecoderGenerator

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- argmax_rows
def _rows(n, V=50257, ld=50264, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf = torch.randn(n, ld, device="cuda", generator=g).to(torch.bfloat16)
    buf[:, V:] = float("inf")  # the padding columns: never a candidate
    x = buf[:, :V]
    rng = random.Random(seed)
    for r in range(n):
        kind = r % 7
        if kind == 1:  # ties of the maximum at several indices
            for j in sorted(rng.sample(range(V), 4)):
                x[r, j] = 8.0
        elif kind == 2:
            x[r] = 0.5  # all equal
        elif kind == 3:
            x[r] = float("-inf")
        elif kind == 4:  # NaNs: the first wins
            for j in rng.sample(range(V), 3):
                x[r, j] = float("nan")
        elif kind == 5:  # the maximum in the last column, next to the padding
            x[r, V - 1] = 9.0
        elif kind == 6:  # a tie across the -0 / +0 pair and a coarse bf16 grid
            x[r] = torch.randint(-3, 1, (V,), device="cuda", generator=g).to(torch.bfloat16)
    return x


@pytest.mark.parametrize("n", [1, 5, 7, 40, 320, 640])
def test_argmax_rows_matches_torch(n):
    x = _rows(n, seed=n)
    out = torch.full((n,), -5, device="cuda", dtype=torch.long)
    ops.argmax_rows(x, out)
    want = torch.argmax(x, dim=-1)
    assert torch.equal(out, want), (out - want).nonzero()
    assert int(out.max()) < x.shape[1]


def test_argmax_rows_strided_output_and_small_vocab():
    x = _rows(12, V=90, ld=96)
    ids = torch.full((4, 6), -5, device="cuda", dtype=torch.long)
    ops.argmax_rows(x[:4], ids[:, 2])  # a column of a (B, k+1) buffer
    assert torch.equal(ids[:, 2], torch.argmax(x[:4], dim=-1)) and bool((ids[:, [0, 1, 3, 4, 5]] == -5).all())
    out = torch.empty(12, device="cuda", dtype=torch.long)
    assert torch.equal(ops.argmax_rows(x, out), torch.argmax(x, dim=-1))


# ---------------------------------------------------------------------------------------------- speculative_accept
def _accept_ref(picks, ids, budget, eos, k):
    """Step 4 of a round, restated per sequence."""
    em, cnt, bud, back, last = [], [], [], [], []
    for t, row, left in zip(picks, ids, budget):
        a = 0
        while a < k and t[a] == row[a + 1]:
            a += 1
        cand, kept = row[1:a + 1] + [t[a]], []
        for tok in cand:
            if len(kept) >= left:
                break
            kept.append(tok)
            if tok == eos:
                break
        m = len(kept)
        em.append(kept + [-1] * (k + 1 - m))
        cnt.append(m)
        bud.append(0 if (kept and kept[-1] == eos) else max(left - m, 0))
        back.append(k + 1 - m)
        last.append(kept[-1] if m else row[0])
    return em, cnt, bud, back, last


@pytest.mark.parametrize("B", [1, 3, 64])
@pytest.mark.parametrize("k", [1, 4, 15])
@pytest.mark.parametrize("shared", [False, True])
def test_speculative_accept_matches_restatement(B, k, shared):
    if shared and B > 1:
        pytest.skip("a shared length needs B = 1")
    rng = random.Random(B * 100 + k)
    for trial in range(8):
        eos = -1 if trial % 3 == 0 else 2
        picks = [[rng.randrange(6) for _ in range(k + 1)] for _ in range(B)]
        ids = []
        for t in picks:  # drafts that agree with the picks for a random prefix, then at random
            a = rng.randrange(k + 1)
            ids.append([rng.randrange(6)] + [t[i] if i < a else rng.randrange(6) for i in range(k)])
        budget = [rng.choice([0, 1, 2, k, k + 1, 100]) for _ in range(B)]
        lt = [rng.randrange(20, 40) for _ in range(B)]
        ld = [rng.randrange(20, 40) for _ in range(B)]
        dev = lambda v, dt=torch.long: torch.tensor(v, device="cuda", dtype=dt)  # noqa: E731
        d_picks, d_ids, d_budget = dev(picks), dev(ids), dev(budget, torch.int32)
        d_lt, d_ld = dev(lt[:1] if shared else lt, torch.int32), dev(ld[:1] if shared else ld, torch.int32)
        res = torch.full((B, k + 2), -7, device="cuda", dtype=torch.long)
        ops.speculative_accept(d_picks, d_ids, d_budget, eos, d_lt, d_ld, res[:, :k + 1], res[:, k + 1])
        em, cnt, bud, back, last = _accept_ref(picks, ids, budget, eos, k)
        assert res[:, :k + 1].tolist() == em and res[:, k + 1].tolist() == cnt
        assert d_budget.tolist() == bud
        assert d_lt.tolist() == [n - b for n, b in zip(lt, back)][:d_lt.numel()]
        assert d_ld.tolist() == [n - b for n, b in zip(ld, back)][:d_ld.numel()]
        assert d_ids[:, 0].tolist() == last and d_ids[:, 1:].tolist() == [r[1:] for r in ids]
        assert torch.equal(d_picks, dev(picks))


# ---------------------------------------------------------------------------------------------- truncate
def test_truncate_then_step_is_bit_identical(golden):
    g = golden("gpt2")
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    with torch.no_grad():
        a, b = m.new_kv_cache(2, 64), m.new_kv_cache(2, 64)
        m.prefill(ids[:, :10], a)
        m.prefill(ids[:, :10], b)
        m.extend(ids[:, 10:17], b)
        b.truncate([10, 10])
        assert not b.ragged and b.length.tolist() == [10]
        for t in range(10, 14):
            assert torch.equal(m.step(ids[:, t], a), m.step(ids[:, t], b)), f"step at position {t}"


def test_truncate_ragged_to_unequal_lengths(golden):
    g = golden("gpt2")
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    keep = [4, 7]
    with torch.no_grad():
        cache = m.new_kv_cache(2, 64)
        m.prefill(_padded(ids, [9, 12]), cache, lengths=[9, 12])
        cache.truncate(keep)
        assert cache.length.tolist() == keep and cache.seq_lengths == keep
        got = m.step(torch.stack([ids[b, n] for b, n in enumerate(keep)]), cache).float()
        for b, n in enumerate(keep):
            own = m.new_kv_cache(1, 64)
            m.prefill(ids[b, :n], own)
            want = m.step(ids[b, n:n + 1], own).float()
            _assert_logits(got[b:b + 1].cpu().numpy(), want.cpu().numpy(), f"sequence {b} truncated to {n}")


# ---------------------------------------------------------------------------------------------- rounds
def _random_lm(base, vocab, layers, d, seed, **attrs):
    torch.manual_seed(seed)
    m = type(f"{base.__name__}R", (base,), dict(vocab_size=vocab, **attrs))(layers, d).eval()
    oracle_torch.randomize_(m.state_dict(), seed)
    return m.cuda()


def _filled_pair(target, draft, ids, lengths, cap):
    tc, dc = target.new_kv_cache(len(lengths), cap), draft.new_kv_cache(len(lengths), cap)
    x = _padded(ids, lengths)
    logits = target.prefill(x, tc, lengths=lengths)
    draft.prefill(x, dc, lengths=lengths)
    last = logits[torch.arange(len(lengths), device="cuda"), torch.tensor(lengths, device="cuda") - 1].argmax(-1)
    return tc, dc, last


def test_graphed_round_is_bit_identical_to_eager(golden):
    g = golden("gpt2")
    target = build_model(g).cuda()
    draft = _random_lm(pm.GPT2, 777, 1, 64, 3)
    ids = torch.from_numpy(np.array(g.input)).cuda()
    ids = torch.cat([ids, ids[:1]])
    lengths, k, budget = [5, 13, 9], 4, [30, 7, 30]
    with torch.no_grad():
        tc, dc, last = _filled_pair(target, draft, ids, lengths, 64)
        eids = torch.zeros(3, k + 1, device="cuda", dtype=torch.long)
        eids[:, 0] = last
        ebud = torch.tensor(budget, device="cuda", dtype=torch.int32)
        gt, gd, glast = _filled_pair(target, draft, ids, lengths, 64)
        rnd = pm.SpeculativeRound(target, gt, draft, gd, k, eos=11)
        assert gt.seq_lengths == lengths and gt.length.tolist() == lengths and gd.length.tolist() == lengths
        rnd.start(glast, budget)
        for r in range(5):
            want = speculative.finish_round(tc, dc, speculative.speculative_round(target, tc, draft, dc, eids, ebud, 11))
            got = rnd()
            assert got == want, f"round {r}"
            for a, b in ((tc, gt), (dc, gd)):
                assert a.seq_lengths == b.seq_lengths and a.n == b.n and a.pad == b.pad
                assert a.length.tolist() == b.length.tolist() == a.seq_lengths
                for ka, kb in zip(a.kv, b.kv):
                    for s, n in enumerate(a.seq_lengths):
                        assert torch.equal(ka[s, :n], kb[s, :n]), f"round {r}: cache rows of sequence {s}"
            assert torch.equal(eids[:, 0], rnd.ids[:, 0]) and torch.equal(ebud, rnd.budget)
        gt.reset()
        target.prefill(ids[:, :4], gt)
        with pytest.raises(ValueError, match="capture a new SpeculativeRound"):
            rnd()


PROMPTS = ["5 17 300 2 41", "9", "1 2 3 4 5 6 7 8 9 10 11 12", "40 41"]


def _acceptance(monkeypatch, k):
    """Record every round's tokens; returns a function giving the mean accepted fraction of the drafts, over the rounds
    that no budget cut (every sequence's last round is left out)."""
    rounds = []
    call = pm.graphs.SpeculativeRound.__call__

    def rec(self):
        out = call(self)
        rounds.append(out)
        return out

    monkeypatch.setattr(pm.graphs.SpeculativeRound, "__call__", rec)

    def mean():
        fr = []
        for b in range(len(rounds[0]) if rounds else 0):
            seq = [r[b] for r in rounds if r[b]]
            fr += [(len(t) - 1) / k for t in seq[:-1]]
        return sum(fr) / max(1, len(fr)), len(fr)

    return mean


@pytest.mark.parametrize("which", ["different", "copy"])
def test_generate_with_draft_is_greedy(golden, which, monkeypatch):
    target = build_model(golden("gpt2")).cuda()
    draft = _random_lm(pm.GPT2, 777, 2, 64, 5) if which == "different" else copy.deepcopy(target)
    acc = _acceptance(monkeypatch, 4)
    gen = DecoderGenerator(target, _Tok())
    for p in PROMPTS:
        plain = [int(t) for t in gen.generate(p, max_tokens=40, use_cache=True).split()]
        got = [int(t) for t in gen.generate(p, max_tokens=40, use_cache=True, draft=draft).split()]
        assert len(got) == len(plain) == len(p.split()) + 40
        _agree(target, plain, got)
    batch = gen.generate_batch(PROMPTS, max_tokens=40, draft=draft, draft_tokens=4)
    plain = gen.generate_batch(PROMPTS, max_tokens=40)
    for p, a, b in zip(PROMPTS, plain, batch):
        a, b = [int(t) for t in a.split()], [int(t) for t in b.split()]
        assert len(a) == len(b) == len(p.split()) + 40
        _agree(target, a, b)
    rate, n = acc()
    print(f"{which} draft: mean acceptance {rate:.3f} over {n} rounds")
    if which == "copy":
        assert rate >= 0.9, rate


def test_draft_stops_each_sequence_at_its_eos(golden):
    target = build_model(golden("gpt2")).cuda()
    draft = _random_lm(pm.GPT2, 777, 2, 64, 5)
    prompts = PROMPTS[:3]
    free = [[int(t) for t in s.split()] for s in DecoderGenerator(target, _Tok()).generate_batch(prompts, 12)]
    eos = free[0][len(prompts[0].split()) + 3]
    gen = DecoderGenerator(target, _Tok(eos))
    for k in (1, 4):
        got = [[int(t) for t in s.split()] for s in gen.generate_batch(prompts, 12, draft=draft, draft_tokens=k)]
        for p, f, g_ in zip(prompts, free, got):
            n = len(p.split())
            new = f[n:]
            want = f[:n + new.index(eos) + 1] if eos in new else f
            assert g_ == want, (k, p, f, g_)
    one = gen.generate_batch(prompts, max_tokens=1, draft=draft)
    assert [len(s.split()) for s in one] == [len(p.split()) + 1 for p in prompts]
    assert gen.generate_batch(prompts, max_tokens=0, draft=draft) == prompts
    assert gen.generate(prompts[0], max_tokens=0, use_cache=True, draft=draft) == prompts[0]
    assert len(gen.generate(prompts[1], max_tokens=1, use_cache=True, draft=draft).split()) == 2


def test_tail_runs_into_the_position_table():
    """max_seq_len 64: prompts of 3..20 tokens plus 45 new ones reach the last position, so the rounds stop and the
    target's plain steps finish (the longest prompt ends exactly at position 63)."""
    target = _random_lm(pm.GPT2, 777, 2, 64, 7, max_seq_len=64)
    draft = copy.deepcopy(target)
    gen = DecoderGenerator(target, _Tok())
    prompts = [" ".join(str(3 + i) for i in range(20)), "7 8 9"]
    plain = gen.generate_batch(prompts, max_tokens=45)
    for k in (4, 8):
        got = gen.generate_batch(prompts, max_tokens=45, draft=draft, draft_tokens=k)
        for a, b in zip(plain, got):
            _agree(target, [int(t) for t in a.split()], [int(t) for t in b.split()])
        one = gen.generate(prompts[0], max_tokens=45, use_cache=True, draft=draft, draft_tokens=k)
        _agree(target, [int(t) for t in plain[0].split()], [int(t) for t in one.split()])


def _agree_rows(plain, rows, got, what):
    """``got`` equals the greedy tokens ``plain`` or first differs where the two best of that position's logits
    (``rows[i]``) lie within the logits bound."""
    if got == plain:
        return
    i = next(i for i, (a, b) in enumerate(zip(plain, got)) if a != b)
    top2 = rows[i].topk(2).values
    scale = max(1.0, float(rows[i].abs().max()) / 4.0)
    assert float(top2[0] - top2[1]) < MAX_ABS_12 * scale, (what, i, plain, got)


def _greedy_steps(m, cache, last, n):
    toks, rows = [], []
    cur = last
    for _ in range(n):
        toks.append(cur.tolist())
        lg = m.step(cur, cache).float()
        rows.append(lg)
        cur = lg.argmax(-1)
    return toks, rows


def _rounds(target, tc, draft, dc, last, k, n):
    rnd = pm.SpeculativeRound(target, tc, draft, dc, k)
    rnd.start(last, [n] * tc.batch)
    out = [[t] for t in last.tolist()]
    while any(len(o) < n + 1 for o in out):
        for b, toks in enumerate(rnd()):
            out[b] += toks
    return out


def test_post_norm_gpt_pair(golden):
    g = golden("gpt")
    target = build_model(g).cuda()
    draft = _random_lm(pm.GPT, 777, 1, 64, 9)
    ids = torch.from_numpy(np.array(g.input)).cuda()
    lengths, n = [6, 11], 24
    with torch.no_grad():
        tc, dc, last = _filled_pair(target, draft, ids, lengths, 64)
        got = _rounds(target, tc, draft, dc, last, 3, n)
        pc, _, plast = _filled_pair(target, draft, ids, lengths, 64)
        toks, rows = _greedy_steps(target, pc, plast, n)
    for b in range(2):
        plain = [t[b] for t in toks] + [int(rows[-1][b].argmax())]
        _agree_rows(plain[1:], [r[b] for r in rows], got[b][1:n + 1], f"GPT sequence {b}")


def test_whisper_decoder_pair(golden):
    g = golden("whisper_full")
    m = build_model(g).cuda()
    target = m.decoder
    torch.manual_seed(11)
    draft = type(target)(1001, 1, 128).eval()
    oracle_torch.randomize_(draft.state_dict(), 11)
    draft = draft.cuda()
    x = torch.from_numpy(np.array(g.input)).cuda()
    prompt = torch.from_numpy(np.array(g.extra["targets"])).cuda()[:, :4]
    n = 20
    with torch.no_grad():
        memory = m.encoder(x)
        caches = []
        for _ in range(2):
            tc, dc = target.new_kv_cache(memory, 64), draft.new_kv_cache(memory, 64)
            logits = target.prefill(prompt, tc, lengths=[4, 4])
            draft.prefill(prompt, dc, lengths=[4, 4])
            caches.append((tc, dc, logits[:, -1].argmax(-1)))
        tc, dc, last = caches[0]
        got = _rounds(target, tc, draft, dc, last, 4, n)
        pc, _, plast = caches[1]
        toks, rows = _greedy_steps(target, pc, plast, n)
    for b in range(2):
        plain = [t[b] for t in toks] + [int(rows[-1][b].argmax())]
        _agree_rows(plain[1:], [r[b] for r in rows], got[b][1:n + 1], f"Whisper sequence {b}")
