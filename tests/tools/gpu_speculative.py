#!/usr/bin/env python
"""Greedy speculative decoding on the B200 (not product code), in one process on one GPU, timed with CUDA events after
warm-up, medians of `--rounds` interleaved rounds, random weights in bf16:

1. `ops.argmax_rows` against torch.argmax on the same bf16 rows of 50257 logits (row stride 50264): 5, 40, 320 rows.
2. One graphed verify (the layers of `extend` for P tokens, the device-side length advance and the logits GEMM)
   against one graphed target step, GPT-2 xl (48 layers, d 1600), B 1 and 8, 256 and 768 cached tokens, P 2, 5, 9.
3. A GPT-2 small -> GPT-2 xl round at k 2, 4, 8, graphed as one round and as its three parts (k + 1 draft steps with
   their k picks; the verify; the pick of the verify rows + the accept), and the break-even acceptance rate alpha* from
   (1 - a^(k+1)) / (1 - a) = t_round / t_step(xl).
4. Tokens/s of `DecoderGenerator.generate_batch` on GPT-2 xl with and without the GPT-2 small draft (B 1 and 8, 64-token
   prompts, 128 new tokens), with the acceptance measured on these random weights; and a GPT-2 small target with a
   copy of itself as the draft (acceptance ~1): a round against k + 1 plain graphed steps.

Every graph below restores the cache lengths it advances (a negative `decode_advance` inside the graph, or a round with
a budget of 0, which rolls back all k + 1 rows), so repeated replays see one cache state. The device name, power
limit and SM clocks are queried (nothing is changed) and stored beside the numbers.

    python tests/tools/gpu_speculative.py --out profiles/r07/speculative.json
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
import pytorch_models_b200 as pm  # noqa: E402
from pytorch_models_b200 import ops  # noqa: E402
from pytorch_models_b200.text import DecoderGenerator  # noqa: E402
from pytorch_models_b200.transformer import embed_tokens_at  # noqa: E402
from gpu_attention_head_dim import device_info, summary, timeit  # noqa: E402


def _model(layers, d):
    with torch.device("cuda"):
        torch.manual_seed(layers * 7 + d)
        m = pm.GPT2(layers, d).eval()
        with torch.no_grad():
            m.pos_embs.normal_(0, 0.02)
    return m.bfloat16()


def _graph(fn, caches):
    """Capture fn() once (after one warm-up call on a side stream); the caches' lengths and mirrors are restored."""
    saved = [(c.length.clone(), c.n) for c in caches]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    for c, (length, n) in zip(caches, saved):
        c.length.copy_(length)
        c.n = n
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    for c, (length, n) in zip(caches, saved):
        c.length.copy_(length)
        c.n = n
    return g


def _interleaved(fns, rounds):
    out = {name: [] for name in fns}
    for _ in range(rounds):
        for name, fn in fns.items():
            out[name].append(timeit(fn, target_ms=100.0))
    return {name: summary(v) for name, v in out.items()}


def _filled(m, B, n, cap):
    cache = m.new_kv_cache(B, cap)
    ids = torch.randint(0, m.vocab_size, (B, n), device="cuda", generator=torch.Generator("cuda").manual_seed(n))
    m.prefill(ids, cache, lengths=[n] * B)
    return cache


def step_graph(m, cache):
    ids = torch.zeros(cache.batch, device="cuda", dtype=torch.long)

    def fn():
        m.step(ids, cache)
        ops.decode_advance(cache.length, -1)
    return _graph(fn, [cache])


def verify_graph(m, cache, P):
    ids = torch.zeros(cache.batch, P, device="cuda", dtype=torch.long)

    def fn():
        h, stats = m.layers.extend_launches(embed_tokens_at(ids, m.token_embs, m.pos_embs, cache), cache)
        ops.decode_advance(cache.length, P)
        m.logits_bf16(h, stats)
        ops.decode_advance(cache.length, -P)
    return _graph(fn, [cache])


@torch.no_grad()
def argmax_table(rounds):
    table = {}
    for rows in (5, 40, 320):
        buf = torch.randn(rows, 50264, device="cuda").to(torch.bfloat16)
        x = buf[:, :50257]
        out = torch.empty(rows, device="cuda", dtype=torch.long)
        assert torch.equal(ops.argmax_rows(x, out), torch.argmax(x, dim=-1))
        r = _interleaved({"argmax_rows": lambda: ops.argmax_rows(x, out),
                          "torch_argmax": lambda: torch.argmax(x, dim=-1)}, rounds)
        r["ratio_ours_over_torch"] = r["argmax_rows"]["ms"] / r["torch_argmax"]["ms"]
        table[f"rows{rows}"] = r
    return table


@torch.no_grad()
def verify_table(xl, rounds):
    table = {}
    for B in (1, 8):
        for n in (256, 768):
            cache = _filled(xl, B, n, n + 32)
            fns = {"step": step_graph(xl, cache)}
            for P in (2, 5, 9):
                fns[f"verify_p{P}"] = verify_graph(xl, cache, P)
            r = _interleaved({k: g.replay for k, g in fns.items()}, rounds)
            for P in (2, 5, 9):
                r[f"ratio_verify_p{P}_over_step"] = r[f"verify_p{P}"]["ms"] / r["step"]["ms"]
            table[f"b{B}_cached{n}"] = r
            del cache, fns
    return table


def _alpha_star(ratio, k):
    """The acceptance rate a at which a round of k drafts emits ratio tokens on average: (1 - a^(k+1)) / (1 - a)."""
    lo, hi = 0.0, 1.0
    if ratio > k + 1:
        return None
    for _ in range(60):
        a = (lo + hi) / 2
        if sum(a ** i for i in range(k + 1)) < ratio:
            lo = a
        else:
            hi = a
    return (lo + hi) / 2


@torch.no_grad()
def round_table(small, xl, rounds):
    table = {}
    B, n = 1, 256
    for k in (2, 4, 8):
        tc, dc = _filled(xl, B, n, n + 32), _filled(small, B, n, n + 32)
        ids = torch.zeros(B, k + 1, device="cuda", dtype=torch.long)
        budget = torch.zeros(B, device="cuda", dtype=torch.int32)  # 0: every round rolls all k + 1 rows back
        P = k + 1

        def draft_part():
            for j in range(P):
                h, stats = small.layers.step(embed_tokens_at(ids[:, j], small.token_embs, small.pos_embs, dc), dc)
                if j < k:
                    ops.argmax_rows(small.logits_bf16(h, stats)[:, 0], ids[:, j + 1])
            ops.decode_advance(dc.length, -P)

        logits = []

        def verify_part():
            h, stats = xl.layers.extend_launches(embed_tokens_at(ids, xl.token_embs, xl.pos_embs, tc), tc)
            ops.decode_advance(tc.length, P)
            logits[:] = [xl.logits_bf16(h, stats)]
            ops.decode_advance(tc.length, -P)

        verify = _graph(verify_part, [tc])
        lg = logits[0]
        picks = torch.empty(B, P, device="cuda", dtype=torch.long)
        res = torch.empty(B, P + 1, device="cuda", dtype=torch.long)

        def accept_part():
            ops.argmax_rows(lg.reshape(B * P, lg.shape[-1]), picks.view(-1))
            ops.speculative_accept(picks, ids, budget, -1, tc.length, dc.length, res[:, :P], res[:, P])
            ops.decode_advance(tc.length, P)  # the accept rolled both caches back by k + 1 (budget 0)
            ops.decode_advance(dc.length, P)

        rnd = pm.SpeculativeRound(xl, tc, small, dc, k)
        fns = {"round": rnd.graph.replay, "draft_steps": _graph(draft_part, [dc]).replay, "verify": verify.replay,
               "accept_pick": _graph(accept_part, [tc, dc]).replay, "xl_step": step_graph(xl, tc).replay}
        r = _interleaved(fns, rounds)
        t_round, t_step = r["round"]["ms"], r["xl_step"]["ms"]
        r["accept_pick_share_of_round"] = r["accept_pick"]["ms"] / t_round
        r["round_over_xl_step"] = t_round / t_step
        r["alpha_star"] = _alpha_star(t_round / t_step, k)
        table[f"k{k}"] = r
        del tc, dc, rnd, fns
    return table


class _Tok:
    eos_token_id = None

    def encode(self, s):
        return [int(t) for t in s.split()]

    def decode(self, ids):
        return " ".join(map(str, ids))


def _generate_timed(gen, prompts, max_tokens, **kw):
    gen.generate_batch(prompts, max_tokens=8, **kw)  # warm-up: packs, allocator, module loads
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = gen.generate_batch(prompts, max_tokens=max_tokens, **kw)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


@torch.no_grad()
def generate_table(small, xl, reps):
    table = {}
    g = torch.Generator().manual_seed(3)
    rounds_log = []
    call = pm.graphs.SpeculativeRound.__call__

    def rec(self):
        out = call(self)
        rounds_log.append((self.k, out))
        return out

    pm.graphs.SpeculativeRound.__call__ = rec
    try:
        for B in (1, 8):
            prompts = [" ".join(str(int(t)) for t in torch.randint(0, 50257, (64,), generator=g)) for _ in range(B)]
            gen = DecoderGenerator(xl, _Tok())
            row = {}
            for name, kw in (("plain", {}), ("draft_k2", dict(draft=small, draft_tokens=2)),
                             ("draft_k4", dict(draft=small, draft_tokens=4))):
                ts = []
                for _ in range(reps):
                    rounds_log.clear()
                    t, out = _generate_timed(gen, prompts, 128, **kw)
                    ts.append(t)
                acc = [(len(toks) - 1) / k for k, rr in rounds_log for toks in rr if toks]
                row[name] = dict(s=statistics.median(ts), tokens_per_s=B * 128 / statistics.median(ts),
                                 mean_acceptance=(sum(acc) / len(acc)) if acc else None)
            table[f"xl_b{B}"] = row
        # machinery: GPT-2 small with a copy of itself, one round against k + 1 plain steps
        import copy
        twin = copy.deepcopy(small)
        mach = {}
        for k in (2, 4, 8):
            tc, dc = _filled(small, 1, 256, 300), _filled(twin, 1, 256, 300)
            rnd = pm.SpeculativeRound(small, tc, twin, dc, k)
            st = step_graph(small, tc)
            r = _interleaved({"round": rnd.graph.replay, "step": st.replay}, 5)
            r["round_over_k_plus_1_steps"] = r["round"]["ms"] / ((k + 1) * r["step"]["ms"])
            mach[f"k{k}"] = r
        table["small_with_copy_draft"] = mach
    finally:
        pm.graphs.SpeculativeRound.__call__ = call
    return table


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this tool measures on the GPU only")
    res = dict(device=device_info(), torch=torch.__version__)
    res["argmax_rows"] = argmax_table(args.rounds)
    small, xl = _model(12, 768), _model(48, 1600)
    res["verify_vs_step_gpt2_xl"] = verify_table(xl, args.rounds)
    res["round_small_to_xl_b1_cached256"] = round_table(small, xl, args.rounds)
    res["generate"] = generate_table(small, xl, 3)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
