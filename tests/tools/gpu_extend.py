#!/usr/bin/env python
"""Extending a filled KV cache on the B200 (not product code), in one process on one GPU, timed with CUDA events after
warm-up, median of `--rounds` interleaved rounds:

1. b200enc_attention_extend (P new query rows per sequence, causal from each sequence's cache length, every key read
   from the cache) against F.scaled_dot_product_attention's cuDNN, flash and mem-efficient backends with
   ``causal_lower_right`` on the same views: P = 128 and 512 against 1024 and 4096 cached keys at B x H = 768, the
   Whisper-large-v3 decoder self-attention, and one ragged batch (against our own uniform launch at the mean length,
   which SDPA cannot express, and SDPA at the longest). Algorithmic TFLOP/s count the visible (query, key) pairs.
2. The causal b200enc_attention of this build against another build of the library (``--parent``, e.g. the parent
   commit's), alternating in the same process on the same buffers: B 8, H 20, L 1500 and ViT-B/16 (B 128, H 12,
   L 197); the time ratio and whether the outputs are bit-identical.
3. GPT-2 small (random weights, bf16, B = 1): a 4-turn conversation of 64-token user turns plus 64 generated tokens
   each (graphed steps), ingesting each turn with `extend` against `reset()` + `prefill` of the whole history; and a
   1024-token prompt as one prefill against 8 extends of 128.

The device name, power limit and SM clocks are queried (nothing is changed) and stored beside the numbers.

    python tests/tools/gpu_extend.py --parent path/to/parent/libb200enc.so --out profiles/r06/extend.json
"""
import argparse
import ctypes
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
import pytorch_models_b200 as pm  # noqa: E402
from pytorch_models_b200 import _lib, ops  # noqa: E402
from gpu_attention_head_dim import device_info, summary, timeit  # noqa: E402

L2_BYTES = 126e6
# name: (B, H, head_dim, cached keys per sequence (int, or a list for a ragged batch), P)
SHAPES = {
    "b64_h12_hd64_cached1024_p128": (64, 12, 64, 1024, 128),
    "b64_h12_hd64_cached1024_p512": (64, 12, 64, 1024, 512),
    "b64_h12_hd64_cached4096_p128": (64, 12, 64, 4096, 128),
    "b64_h12_hd64_cached4096_p512": (64, 12, 64, 4096, 512),
    "b24_h32_hd128_cached4096_p512": (24, 32, 128, 4096, 512),
    # Whisper-large-v3 decoder self-attention (20 heads of 64, 448 positions): the last 128 of a full context
    "whisper_large_v3_b64_h20_hd64_cached320_p128": (64, 20, 64, 320, 128),
}
RAGGED = ("ragged_b64_h12_hd64_p128", 64, 12, 64, 128)  # cached keys drawn from [0, 4096 - 128]


def _pairs(offsets, P):
    """Visible (query, key) pairs: query i of a sequence at offset o sees o + i + 1 keys."""
    return sum(P * o + P * (P + 1) // 2 for o in offsets)


@torch.no_grad()
def extend_table(rounds):
    from torch.nn.attention import SDPBackend, sdpa_kernel
    from torch.nn.attention.bias import causal_lower_right

    backends = {"cudnn": SDPBackend.CUDNN_ATTENTION, "flash": SDPBackend.FLASH_ATTENTION,
                "efficient": SDPBackend.EFFICIENT_ATTENTION}
    table = {}
    cases = dict(SHAPES)
    g0 = torch.Generator().manual_seed(6)
    name, B, H, hd, P = RAGGED
    cases[name] = (B, H, hd, torch.randint(0, 4096 - P + 1, (B,), generator=g0).tolist(), P)
    for name, (B, H, hd, cached, P) in cases.items():
        ragged = isinstance(cached, list)
        offsets = cached if ragged else [cached] * B
        cap = max(offsets) + P
        W = H * hd
        g = torch.Generator(device="cuda").manual_seed(cap + P)
        kv = torch.randn(B, cap, 2 * W, device="cuda", dtype=torch.bfloat16, generator=g)
        qkv = torch.randn(B, P, 3 * W, device="cuda", dtype=torch.bfloat16, generator=g)
        out = torch.empty(B, P, W, device="cuda", dtype=torch.bfloat16)
        length = torch.tensor(offsets if ragged else offsets[:1], device="cuda", dtype=torch.int32)
        ops.kv_append(qkv[:, :, W:], kv, length)
        scale = hd ** -0.5
        ours = lambda: ops.attention_extend(qkv[:, :, :W], kv[:, :, :W], kv[:, :, W:], out, H, scale, length)  # noqa
        fns = {"b200enc": ours}
        pairs = _pairs(offsets, P) * H
        kv_bytes = 2 * sum(o + P for o in offsets) * W * 2
        row = dict(B=B, H=H, head_dim=hd, P=P, cached=cached if not ragged else dict(
            mean=statistics.mean(offsets), min=min(offsets), max=max(offsets)), kv_bytes=kv_bytes,
            exceeds_l2=kv_bytes > L2_BYTES, flop=4 * hd * pairs)
        if ragged:
            mean = round(statistics.mean(offsets))
            kv_u = torch.randn(B, mean + P, 2 * W, device="cuda", dtype=torch.bfloat16, generator=g)
            len_u = torch.full((1,), mean, device="cuda", dtype=torch.int32)
            out_u = torch.empty_like(out)
            fns["b200enc_uniform_at_mean"] = lambda: ops.attention_extend(  # noqa: E731
                qkv[:, :, :W], kv_u[:, :, :W], kv_u[:, :, W:], out_u, H, scale, len_u)
            row["flop_uniform_at_mean"] = 4 * hd * _pairs([mean] * B, P) * H
        # SDPA on the same cache views (the longest sequence for a ragged batch)
        L = max(offsets) + P
        qh = qkv[:, :, :W].unflatten(-1, (H, hd)).transpose(1, 2)
        kh = kv[:, :L, :W].unflatten(-1, (H, hd)).transpose(1, 2)
        vh = kv[:, :L, W:].unflatten(-1, (H, hd)).transpose(1, 2)
        mask = causal_lower_right(P, L)
        ours()
        for bname, be in backends.items():
            def fn(be=be):
                with sdpa_kernel(be):
                    return F.scaled_dot_product_attention(qh, kh, vh, attn_mask=mask, scale=scale)
            try:
                y = fn().transpose(1, 2).reshape(B, P, W)
                if not ragged:
                    row[f"max_abs_diff_vs_{bname}"] = float((y.float() - out.float()).abs().max())
                fns[bname] = fn
            except RuntimeError as e:
                row[bname] = dict(unsupported=f"{type(e).__name__}: {str(e)[:160]}")
        samples = {k: [] for k in fns}
        for _ in range(rounds):
            for k, fn in fns.items():
                samples[k].append(timeit(fn))
        for k, s in samples.items():
            flop = row["flop_uniform_at_mean"] if k == "b200enc_uniform_at_mean" else row["flop"]
            if k in backends and ragged:
                flop = 4 * hd * _pairs([max(offsets)] * B, P) * H
            row[k] = dict(summary(s), tflop_s=flop / statistics.median(s) * 1e-9)
        for k in samples:
            if k != "b200enc":
                row[f"time_ratio_vs_{k}"] = row["b200enc"]["ms"] / row[k]["ms"]
        table[name] = row
        print("extend", name, json.dumps(row), flush=True)
        del kv, qkv, out
        torch.cuda.empty_cache()
    return table


def _load_other(path):
    lib = ctypes.CDLL(path)
    fn = lib.b200enc_attention
    fn.restype, fn.argtypes = _lib._SIGNATURES["b200enc_attention"]
    return lib


@torch.no_grad()
def causal_regression(rounds, parent_path):
    """Causal b200enc_attention of this build and of `parent_path`, alternating on the same buffers."""
    libs = {"this": _lib.load(), "parent": _load_other(parent_path)}
    table = {}
    for name, (B, H, L) in {"b8_h20_l1500_hd64": (8, 20, 1500), "vit_b16_b128_h12_l197_hd64": (128, 12, 197)}.items():
        W = H * 64
        g = torch.Generator(device="cuda").manual_seed(L)
        qkv = torch.randn(B, L, 3 * W, device="cuda", dtype=torch.bfloat16, generator=g)
        outs = {k: torch.empty(B, L, W, device="cuda", dtype=torch.bfloat16) for k in libs}

        def call(k):
            rc = libs[k].b200enc_attention(
                qkv.data_ptr(), qkv.stride(0), qkv.stride(1), qkv[:, :, W:].data_ptr(), qkv[:, :, 2 * W:].data_ptr(),
                qkv.stride(0), qkv.stride(1), outs[k].data_ptr(), outs[k].stride(0), outs[k].stride(1), B, H, L, L,
                64, 0.125, _lib.ATTN_CAUSAL, torch.cuda.current_stream().cuda_stream)
            assert rc == 0, (k, rc)

        samples = {k: [] for k in libs}
        for _ in range(rounds):
            for k in libs:
                samples[k].append(timeit(lambda k=k: call(k)))
        row = dict(B=B, H=H, L=L, bit_identical=bool(torch.equal(outs["this"], outs["parent"])))
        for k, s in samples.items():
            row[k] = summary(s)
        row["time_ratio_this_over_parent"] = row["this"]["ms"] / row["parent"]["ms"]
        table[name] = row
        print("causal", name, json.dumps(row), flush=True)
    return table


def _wall(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


@torch.no_grad()
def gpt2_end_to_end(rounds, turns=4, turn=64, reply=64):
    torch.manual_seed(0)
    m = pm.GPT2(12, 768).eval().cuda().bfloat16()
    g = torch.Generator().manual_seed(2)
    conv = torch.randint(0, m.vocab_size, (1, turns * (turn + reply)), generator=g).cuda()
    total = conv.shape[1]
    res = {}

    def conversation(mode, cache, step):
        """Each turn: ingest the user's `turn` tokens, then generate `reply` tokens with graphed steps (teacher forced
        on the recorded conversation, so both modes do the same work)."""
        cache.reset()
        at = 0
        for _ in range(turns):
            if mode == "extend":
                m.prefill(conv[:, :turn], cache) if at == 0 else m.extend(conv[:, at:at + turn], cache)
            else:
                cache.reset()
                m.prefill(conv[:, :at + turn], cache)
            at += turn
            for t in range(reply):
                step(conv[:, at + t])
            at += reply

    cache = m.new_kv_cache(1, total)
    m.prefill(conv[:, :turn], cache)
    step = pm.GraphedStep(m, cache)
    samples = {"extend": [], "reset_prefill": []}
    ingest = {"extend": [], "reset_prefill": []}
    for _ in range(rounds):
        for mode in samples:
            samples[mode].append(_wall(lambda: conversation(mode, cache, step)))

            def ingest_only(mode=mode):  # the turns alone, without the replies
                cache.reset()
                at = 0
                for _ in range(turns):
                    if mode == "extend":
                        m.prefill(conv[:, :turn], cache) if at == 0 else m.extend(conv[:, at:at + turn], cache)
                    else:
                        cache.reset()
                        m.prefill(conv[:, :at + turn], cache)
                    at += turn
                    cache.n += reply  # the replies' rows (stale here), so each turn lands where it would
                    cache.length.add_(reply)
            ingest[mode].append(_wall(ingest_only))
    res["conversation"] = dict(turns=turns, turn_tokens=turn, reply_tokens=reply, total_tokens=total)
    for mode in samples:
        res["conversation"][mode] = dict(summary(samples[mode]),
                                         tokens_s=total / statistics.median(samples[mode]) * 1e3,
                                         ingest_only=summary(ingest[mode]))
    res["conversation"]["speedup_extend"] = (res["conversation"]["reset_prefill"]["ms"]
                                             / res["conversation"]["extend"]["ms"])

    prompt = torch.randint(0, m.vocab_size, (1, 1024), generator=g).cuda()
    big = m.new_kv_cache(1, 1024)

    def one():
        big.reset()
        return m.prefill(prompt, big)

    def chunks():
        big.reset()
        return torch.cat([m.extend(prompt[:, i:i + 128], big) for i in range(0, 1024, 128)], 1)

    a, b = one(), chunks()
    diff = float((a.float() - b.float()).abs().max())
    s = {"prefill_1024": [], "extend_8x128": []}
    for _ in range(rounds):
        s["prefill_1024"].append(timeit(one))
        s["extend_8x128"].append(timeit(chunks))
    res["prompt_1024"] = {k: dict(summary(v), tokens_s=1024 / statistics.median(v) * 1e3) for k, v in s.items()}
    res["prompt_1024"]["max_abs_logit_diff"] = diff
    print("gpt2", json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--parent", default=None, help="another build of libb200enc.so for the causal-kernel comparison")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = dict(device=device_info(), torch=torch.__version__)
    res["attention_extend"] = extend_table(args.rounds)
    if args.parent:
        res["causal_attention_vs_parent"] = causal_regression(args.rounds, args.parent)
    res["gpt2_small"] = gpt2_end_to_end(args.rounds)
    res["device_after"] = device_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
