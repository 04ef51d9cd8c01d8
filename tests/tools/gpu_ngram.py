#!/usr/bin/env python
"""Draft-free (n-gram) speculative decoding on the B200 (not product code), in one process on one GPU, timed with CUDA
events after warm-up, medians of `--rounds` interleaved rounds, random weights in bf16:

1. `ops.ngram_draft` alone, B 1 and 64, capacity 1024 and 4096, k 4, every history nearly full (the search reads
   every row): a graph of one length reset and 20 launches, whose lengths run from capacity - 105 to capacity - 5.
2. One graphed n-gram round (`SpeculativeRound` with `NGramDraft`) over one graphed step of the same model, GPT-2 small
   (12 x 768) and xl (48 x 1600), B 1, 8 and 64, 256 cached tokens, k 2, 4 and 8. The round's budget is 0, so it rolls
   all k + 1 rows back and every replay sees one state; the round does the same work whatever it accepts.
3. Tokens/s of `generate` (B 1) and `generate_batch` (B 8) on GPT-2 xl, 64-token random prompts, 128 new tokens, with
   and without `NGramDraft` (k 4), and the acceptance measured on these random weights.
4. Two cases with a known outcome on GPT-2 xl at B 1: a prompt holding a 96-token passage and then its first 48
   tokens again, and no acceptance at all, where every round emits one token and costs the ratio of (2).

The device name, power limit and SM clocks are queried (nothing is changed) and stored beside the numbers.

    python tests/tools/gpu_ngram.py --out profiles/r08
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
from gpu_attention_head_dim import device_info  # noqa: E402
from gpu_speculative import _Tok, _filled, _interleaved, _model, step_graph  # noqa: E402


@torch.no_grad()
def kernel_table(rounds):
    table, k, calls = {}, 4, 20
    for B in (1, 64):
        for cap in (1024, 4096):
            g = torch.Generator(device="cuda").manual_seed(B + cap)
            hist = torch.randint(0, 50257, (B, cap), device="cuda", generator=g)
            ids = torch.randint(0, 50257, (B, k + 1), device="cuda", generator=g)
            start = torch.full((B,), cap - calls * (k + 1) - 5, device="cuda", dtype=torch.int32)
            length = start.clone() if B > 1 else start[:1].clone()

            def fn():
                length.copy_(start[:length.numel()])
                for _ in range(calls):
                    ops.ngram_draft(hist, length, ids, k, 3, 1)
            fn()
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                fn()
            r = _interleaved({"graph_of_20": graph.replay}, rounds)
            r["us_per_launch"] = r["graph_of_20"]["ms"] * 1000 / calls
            table[f"b{B}_cap{cap}"] = r
    return table


@torch.no_grad()
def round_table(models, rounds):
    table = {}
    for name, m in models.items():
        for B in (1, 8, 64):
            n = 256
            tc = _filled(m, B, n, n + 32)
            fns = {"step": step_graph(m, tc).replay}
            keep = []
            for k in (2, 4, 8):
                draft = pm.NGramDraft()
                hist = draft.new_kv_cache(B, n + 32)
                draft.prefill(torch.randint(0, m.vocab_size, (B, n), device="cuda"), hist, lengths=[n] * B)
                rnd = pm.SpeculativeRound(m, tc, draft, hist, k)  # budget 0: all k + 1 rows roll back
                keep.append(rnd)
                fns[f"round_k{k}"] = rnd.graph.replay
            r = _interleaved(fns, rounds)
            for k in (2, 4, 8):
                r[f"ratio_round_k{k}_over_step"] = r[f"round_k{k}"]["ms"] / r["step"]["ms"]
            table[f"{name}_b{B}"] = r
            del tc, fns, keep
    return table


def _recording():
    log = []
    call = pm.graphs.SpeculativeRound.__call__

    def rec(self):
        out = call(self)
        log.append((self.k, out))
        return out

    pm.graphs.SpeculativeRound.__call__ = rec
    return log, lambda: setattr(pm.graphs.SpeculativeRound, "__call__", call)


def _acceptance(log):
    """Mean accepted fraction of the drafts over the rounds that no budget cut (each sequence's last round left out)."""
    fr = []
    for b in range(len(log[0][1]) if log else 0):
        seq = [(k, r[b]) for k, r in log if r[b]]
        fr += [(len(t) - 1) / k for k, t in seq[:-1]]
    return (sum(fr) / len(fr)) if fr else None


def _timed(fn, reps):
    fn()  # warm-up: packs, allocator, module loads
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), out


@torch.no_grad()
def generate_table(xl, reps):
    table = {}
    g = torch.Generator().manual_seed(3)
    log, restore = _recording()
    gen = DecoderGenerator(xl, _Tok())
    rand = lambda L: [int(t) for t in torch.randint(0, 50257, (L,), generator=g)]  # noqa: E731
    try:
        cases = {"generate_b1": [rand(64)], "generate_batch_b8": [rand(64) for _ in range(8)]}
        passage = rand(96)
        cases["repeated_passage_b1"] = [rand(32) + passage + passage[:48]]
        for case, toks in cases.items():
            prompts = [" ".join(map(str, t)) for t in toks]
            row = {}
            for name, kw in (("plain", {}), ("ngram_k4", dict(draft=pm.NGramDraft(), draft_tokens=4))):
                if len(prompts) == 1:
                    fn = lambda: [gen.generate(prompts[0], max_tokens=128, use_cache=True, **kw)]  # noqa: E731
                else:
                    fn = lambda: gen.generate_batch(prompts, max_tokens=128, **kw)  # noqa: E731
                log.clear()
                t, out = _timed(fn, reps)
                row[name] = dict(s=t, tokens_per_s=len(prompts) * 128 / t, mean_acceptance=_acceptance(log),
                                 rounds_per_call=len(log) / (reps + 1))
            table[case] = row
    finally:
        restore()
    return table


def _write_readme(res, path):
    dev = res["device"]
    lines = ["# r08: draft-free (n-gram) speculative decoding", "",
             f"`ngram.json` was written by `python tests/tools/gpu_ngram.py --out profiles/r08` on one "
             f"{dev.get('name')} ({dev.get('power.limit')} power limit, {dev.get('clocks.max.sm')} max SM clock, read "
             "in the same run). All models have random weights in bf16. Times are medians of interleaved CUDA-event "
             "windows of about 100 ms each; generator times are wall-clock seconds of one call after a warm-up call, "
             "CUDA-graph captures included.", "", "## `ngram_draft` alone (k 4, nearly full histories)", "",
             "| | µs per launch |", "|---|---|"]
    for key, r in res["ngram_draft"].items():
        lines.append(f"| {key} | {r['us_per_launch']:.2f} |")
    lines += ["", "## n-gram round over one graphed step (256 cached tokens)", "",
              "| | step ms | k 2 | k 4 | k 8 |", "|---|---|---|---|---|"]
    for key, r in res["round_over_step"].items():
        lines.append(f"| {key} | {r['step']['ms']:.3f} | " + " | ".join(
            f"{r[f'ratio_round_k{k}_over_step']:.3f}" for k in (2, 4, 8)) + " |")
    lines += ["", "## Generator on GPT-2 xl, 128 new tokens", "",
              "| | plain tokens/s | n-gram k 4 tokens/s | speed-up | acceptance |", "|---|---|---|---|---|"]
    for key, r in res["generate_xl"].items():
        a, b = r["plain"], r["ngram_k4"]
        acc = "–" if b["mean_acceptance"] is None else f"{b['mean_acceptance']:.3f}"
        lines.append(f"| {key} | {a['tokens_per_s']:.1f} | {b['tokens_per_s']:.1f} | "
                     f"{b['tokens_per_s'] / a['tokens_per_s']:.2f} | {acc} |")
    na = res["no_acceptance_xl_b1_k4"]
    lines += ["", f"No acceptance (xl, B 1, k 4): every round emits one token and costs {na['round_ms']:.3f} ms "
              f"against {na['step_ms']:.3f} ms for a step, so tokens/s fall to {na['ratio']:.3f}⁻¹ of plain steps.",
              "", "Random-weight models fall into loops that an n-gram lookup predicts, so the acceptance above is not "
              "a trained model's. The repeated-passage prompt gives the same acceptance and round count as the random "
              "prompts: on these weights the output is the model's own loop, so this case does not show a passage "
              "being copied; a trained model that quotes its prompt is what it stands for. Generator "
              "times include one graph capture per call, and they vary more between calls than the graph replays do.",
              ""]
    with open(path, "w") as f:
        f.write("\n".join(lines))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for ngram.json and README.md (default: stdout only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this tool measures on the GPU only")
    res = dict(device=device_info(), torch=torch.__version__)
    res["ngram_draft"] = kernel_table(args.rounds)
    small, xl = _model(12, 768), _model(48, 1600)
    res["round_over_step"] = round_table({"small": small, "xl": xl}, args.rounds)
    r = res["round_over_step"]["xl_b1"]
    res["no_acceptance_xl_b1_k4"] = dict(round_ms=r["round_k4"]["ms"], step_ms=r["step"]["ms"],
                                         ratio=r["ratio_round_k4_over_step"])
    res["generate_xl"] = generate_table(xl, 2)
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "ngram.json"), "w") as f:
            json.dump(res, f, indent=1)
        _write_readme(res, os.path.join(args.out, "README.md"))


if __name__ == "__main__":
    main()
