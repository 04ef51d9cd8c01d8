"""The inputs of test_gpu_attention_exact.py on the CPU: the exact expectations equal fp64 SDPA where that is cheap to
compute, and every mistake a kernel could make on each GPU case (tests/attention_inputs.py) breaks the bound that case
applies, in every sequence it applies to. The rejected mutants of each case are printed (pytest -s)."""
from __future__ import annotations

import math

import pytest
import torch
import torch.nn.functional as F

import attention_inputs as ai


def _check_rejects(case, exact):
    want = case.expected()
    rejected, missed = [], []
    for m in case.mutants():
        got = case.expected(m)
        if exact:
            got = ai.bf16_round(got)  # what a kernel that computes the mutant exactly would write
        checked = [b for b in range(case.B) if case.applies(m, b)]
        assert checked, f"mutant {m} applies to no sequence"
        for b in checked:
            try:
                if exact:
                    ai.assert_exact(got[b], want[b], case.zero_tol)
                else:
                    ai.assert_close(got[b], want[b])
                missed.append((m, b))
            except AssertionError:
                pass
        rejected.append(f"{m} (sequences {checked})" if len(checked) < case.B else m)
    assert not missed, f"mutants that pass the bound (mutant, sequence): {missed}"
    return rejected


def _required(case):
    """The mutants a case must list: every one that its shape lets a kernel make."""
    req = {"drop_first_unit"}
    if isinstance(case, ai.AttnExact):
        if case.n_seen == case.Lkv:
            req |= {"kv_plus_1"} | ({"kv_minus_1"} if case.Lkv > 1 else set())
        if case.causal:
            req |= {"diag_minus_1"} | ({"diag_plus_1"} if min(case.Lq, case.Lkv) > 1 else set())
            req |= {"bottom_right"} if case.Lq != case.Lkv else set()
        if case.use_bias:
            req.add("mask_leak")
    elif isinstance(case, ai.ExtendExact):
        req |= {"off_plus_1"} | ({"off_minus_1", "top_left"} if max(case.offsets) >= 1 else set())
        if len(set(case.offsets)) > 1:
            req |= {"other_len_prev", "other_len_next"}
    else:
        ns = [case._n(b) for b in range(case.B) if case._valid(case._n(b))]
        if case.append:
            req |= {"len_plus_1", "stale_for_new"} | ({"len_minus_1"} if max(ns) >= 1 else set())
            if not case.shared:
                req |= {"other_len_prev", "other_len_next"}
        else:
            req |= ({"len_plus_1"} if case.Lkv < case.capacity else set()) | ({"len_minus_1"} if case.Lkv > 1 else set())
    keys = _keys(case)
    if max(keys) > case.u:
        req |= {"drop_middle_unit", "drop_last_full_unit", "dup_middle_unit"}
    if any(n % case.u for n in keys):
        req.add("drop_tail_unit")
    return req


@pytest.mark.parametrize("name", sorted(ai.EXACT_CASES))
def test_exact_case_rejects_every_mutant(name):
    case = ai.EXACT_CASES[name]()
    want = case.expected()
    # the exact output itself passes, and so does its bf16 rounding
    ai.assert_exact(ai.bf16_round(want), want, case.zero_tol)
    ms = set(case.mutants())
    assert _required(case) <= ms, (name, _required(case) - ms)
    print(f"{name}: rejects {', '.join(_check_rejects(case, exact=True))}")


@pytest.mark.parametrize("name", sorted(ai.PLANTED_CASES))
def test_planted_case_rejects_a_mis_scaled_partial(name):
    case = ai.PLANTED_CASES[name]()
    assert set(case.mutants()) == {"planted_unit_x2", "planted_unit_x0.5"}
    print(f"{name}: rejects {', '.join(_check_rejects(case, exact=False))}")


def _keys(case):
    if isinstance(case, ai.AttnExact):
        return [case.n_seen]
    if isinstance(case, ai.ExtendExact):
        return [o + case.P for o in case.offsets]
    return [case._n(b) + case.append for b in range(case.B) if case._valid(case._n(b))]


# ------------------------------------------------------------------------------------------------- vs fp64 SDPA
def _sdpa64(q, k, v, H, mask=None):
    """q (Lq, W), k / v (Lkv, W) -> (Lq, W) float64."""
    heads = lambda t: t.double().view(t.shape[0], H, -1).transpose(0, 1)  # noqa: E731
    out = F.scaled_dot_product_attention(heads(q), heads(k), heads(v), attn_mask=mask)
    return out.transpose(0, 1).reshape(q.shape[0], -1)


@pytest.mark.parametrize("causal,Lq,Lkv", [(False, 130, 193), (True, 129, 129), (True, 5, 300), (True, 300, 5)])
@pytest.mark.parametrize("hd", [64, 80])
def test_attention_expectation_is_sdpa(causal, Lq, Lkv, hd):
    c = ai.AttnExact(2, 3, hd, Lq, Lkv, causal=causal)
    want = c.expected()
    W = c.W
    mask = torch.ones(Lq, Lkv).tril().bool() if causal else None
    for b in range(2):
        ref = _sdpa64(c.q[b], c.kv[b, :Lkv, :W], c.kv[b, :Lkv, W:], 3, mask)
        torch.testing.assert_close(want[b], ref, rtol=1e-12, atol=1e-12, equal_nan=True)


def test_bias_expectation_is_sdpa():
    c = ai.AttnExact(2, 3, 64, 130, 300, bias=True, seed=1)
    want = c.expected()
    W = c.W
    for b in range(2):
        heads = lambda t: t.double().view(t.shape[0], 3, -1).transpose(0, 1)  # noqa: E731
        ref = F.scaled_dot_product_attention(heads(c.q[b]), heads(c.kv[b, :300, :W]), heads(c.kv[b, :300, W:]),
                                             attn_mask=c.bias[b].double())
        torch.testing.assert_close(want[b], ref.transpose(0, 1).reshape(130, W), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("shared", [False, True])
def test_extend_expectation_is_sdpa(shared):
    P, cap = 7, 300
    offs = [129, 129] if shared else [0, 1, 128, cap - P]
    c = ai.ExtendExact(len(offs), 2, 64, P, offs, cap, shared=shared)
    want = c.expected()
    W = c.W
    for b, o in enumerate(offs):
        k = torch.cat([c.kv[b, :o, :W], c.qkv[b, :, W:2 * W]])
        v = torch.cat([c.kv[b, :o, W:], c.qkv[b, :, 2 * W:]])
        mask = torch.arange(o + P)[None, :] <= o + torch.arange(P)[:, None]
        torch.testing.assert_close(want[b], _sdpa64(c.qkv[b, :, :W], k, v, 2, mask), rtol=1e-12, atol=1e-12)
        # the stale rows a rollback left inside the last 128-key block carry the STALE flag, and nothing reads them
        end = min(-(-(o + P) // 128) * 128, cap)
        assert bool((c.kv[b, o + P:end, W:].float().view(-1, 2, 64)[:, :, ai.STALE] == 1).all())
        assert bool(c.kv[b, end:].float().isnan().all())
        assert bool((want[b].view(P, 2, 64)[:, :, ai.STALE] == 0).all())


def test_decode_expectation_is_sdpa():
    cap = 300
    lengths = [0, 1, 63, 64, 65, cap - 1, -1, cap]
    c = ai.DecodeExact(len(lengths), 3, 64, cap, lengths)
    want = c.expected()
    W = c.W
    for b, n in enumerate(lengths):
        if not 0 <= n < cap:
            assert bool(want[b].isnan().all())
            continue
        k = torch.cat([c.kv[b, :n, :W], c.qkv[b:b + 1, W:2 * W]])
        v = torch.cat([c.kv[b, :n, W:], c.qkv[b:b + 1, 2 * W:]])
        torch.testing.assert_close(want[b:b + 1], _sdpa64(c.qkv[b:b + 1, :W], k, v, 3), rtol=1e-12, atol=1e-12)
        cols = want[b].view(3, 64)
        assert bool((cols[:, ai.NEW] == 1 / (n + 1)).all()) and bool((cols[:, ai.STALE] == 0).all())
        assert bool((cols[:, ai.ONES] == 1).all())
        assert [int(x) for x in cols[0, ai.B_BITS:ai.B_BITS + 8]] == [(b >> i) & 1 for i in range(8)]
        assert [int(x) for x in cols[2, ai.H_BITS:ai.H_BITS + 6]] == [(2 >> i) & 1 for i in range(6)]
    c = ai.DecodeExact(2, 3, 64, cap, Lkv=200)
    want = c.expected()
    for b in range(2):
        ref = _sdpa64(c.qkv[b:b + 1, :W], c.kv[b, :200, :W], c.kv[b, :200, W:], 3)
        torch.testing.assert_close(want[b:b + 1], ref, rtol=1e-12, atol=1e-12)


def test_planted_reference_is_sdpa_and_the_planted_key_dominates():
    for kind, lengths in (("decode", [299, 299]), ("stream", [300]), ("extend", [300, 200])):
        c = ai.Planted(kind, 2, 3, 64, lengths, "last", seed=5)
        want = c.expected()
        for b in range(2):
            n = c.keys[b]
            k, v = c.k[b, :n].reshape(n, -1), c.v[b, :n].reshape(n, -1)
            q = c.q[b].reshape(c.Q, -1)
            mask = None
            if kind == "extend":
                mask = torch.arange(n)[None, :] <= n - c.Q + torch.arange(c.Q)[:, None]
            ref = _sdpa64(q, k, v, 3, mask)
            torch.testing.assert_close(want[b].reshape(c.Q, -1), ref, rtol=1e-12, atol=1e-12)
            s = torch.einsum("qhd,rhd->hqr", c.q[b], c.k[b, :n]) * c.scale
            if mask is not None:
                s = s.masked_fill(~mask, -math.inf)
            p = c.p[b]
            others = torch.cat([s[..., :p], s[..., p + 1:]], -1).max(-1).values
            margin = s[..., p] - others
            assert float(margin.min()) > ai.PLANT_MARGIN - 0.1, (kind, b, float(margin.min()))


def test_decode_chunk_rule():
    """decode_chunk in csrc/api_decode.cu: ~4096 work items, a multiple of 64 in [64, 4096]."""
    assert ai.decode_chunk(2, 3, 32776) == 64
    assert ai.decode_chunk(40, 4, 2056) == 128
    assert ai.decode_chunk(64, 64, 100000) == 4096
    assert ai.decode_chunk(1, 1, 1) == 64
    for B, H, keys in ((3, 5, 2048), (16, 12, 5000), (64, 4, 4104)):
        kc = ai.decode_chunk(B, H, keys)
        assert kc % 64 == 0 and -(-keys // kc) * B * H <= 4096 + B * H
