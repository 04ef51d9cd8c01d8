#!/usr/bin/env python
"""Incremental decoding on the B200 (not product code), in one process on one GPU, timed with CUDA events after warm-up,
median of `--rounds` interleaved rounds:

1. b200enc_attention_decode (csrc/attention_decode.cuh, append mode: L - 1 cached rows plus the new one) against
   F.scaled_dot_product_attention's flash, cuDNN and mem-efficient backends with a one-row query on the same cache
   views, and against the HBM copy bandwidth measured in the same run (a 4 GiB device-to-device copy).
2. GPT-2 small and medium (random weights): tokens/s for 256 new tokens after a 128-token prompt at B = 1, 8, 64:
   cached eager steps, cached CUDA-graph steps (GraphedStep), the uncached loop (B = 1; forward over the prefix per
   token, what DecoderGenerator does by default), and PyTorch bf16 eager with its own KV cache (F.linear + SDPA on the
   same weights).
3. The Whisper-large-v3 decoder step at B = 64 against 1500 memory frames: ms per token (eager and graphed) and the
   eager step split per entry point with ops.profile.

The device name, power limit and SM clocks are queried (nothing is changed) and stored beside the numbers.

    python tests/tools/gpu_decode.py --out profiles/r04/decode.json
"""
import argparse
import collections
import json
import os
import statistics
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
import pytorch_models_b200 as pm  # noqa: E402
from pytorch_models_b200 import ops  # noqa: E402
from gpu_attention_head_dim import device_info, summary, timeit  # noqa: E402

L2_BYTES = 126e6
# name: (B, H, L, head_dim)
SHAPES = {
    "b1_h12_l1024_hd64": (1, 12, 1024, 64),
    "b64_h12_l1024_hd64": (64, 12, 1024, 64),
    "whisper_large_v3_cross_b64_h20_l1500_hd64": (64, 20, 1500, 64),
    "b32_h16_l4096_hd80": (32, 16, 4096, 80),
    "b16_h8_l8192_hd128": (16, 8, 8192, 128),
}


@torch.no_grad()
def copy_bandwidth(rounds):
    n = 1 << 31  # 2^31 bf16 = 4 GiB
    a = torch.empty(n, device="cuda", dtype=torch.bfloat16)
    b = torch.empty_like(a)
    s = [timeit(lambda: b.copy_(a)) for _ in range(rounds)]
    del a, b
    torch.cuda.empty_cache()
    ms = statistics.median(s)
    return dict(summary(s), bytes=2 * 2 * n, tb_s=2 * 2 * n / ms * 1e-9)


@torch.no_grad()
def decode_table(rounds, copy_tb_s):
    from torch.nn.attention import SDPBackend, sdpa_kernel

    backends = {"flash": SDPBackend.FLASH_ATTENTION, "cudnn": SDPBackend.CUDNN_ATTENTION,
                "efficient": SDPBackend.EFFICIENT_ATTENTION}
    table = {}
    for name, (B, H, L, hd) in SHAPES.items():
        W = H * hd
        g = torch.Generator(device="cuda").manual_seed(L + hd)
        kv = torch.randn(B, L, 2 * W, device="cuda", dtype=torch.bfloat16, generator=g)
        qkv = torch.randn(B, 3 * W, device="cuda", dtype=torch.bfloat16, generator=g)
        work = torch.empty(ops.decode_workspace_bytes(B, H, hd, L) // 4, device="cuda")
        length = torch.full((1,), L - 1, device="cuda", dtype=torch.int32)
        out = torch.empty(B, W, device="cuda", dtype=torch.bfloat16)
        ours = lambda: ops.attention_decode(qkv[:, :W], kv[:, :, :W], kv[:, :, W:], out, H, hd ** -0.5, work,  # noqa
                                            k_new=qkv[:, W:2 * W], v_new=qkv[:, 2 * W:], length=length)
        ours()
        # the same keys for SDPA: the cache now holds the new row at L - 1
        qh = qkv[:, :W].view(B, H, 1, hd)
        kh = kv[:, :, :W].unflatten(-1, (H, hd)).transpose(1, 2)
        vh = kv[:, :, W:].unflatten(-1, (H, hd)).transpose(1, 2)
        fns = {"b200enc": ours}
        bytes_kv = 2 * B * L * W * 2
        row = dict(B=B, H=H, L=L, head_dim=hd, kv_bytes=bytes_kv, exceeds_l2=bytes_kv > L2_BYTES)
        for bname, be in backends.items():
            def fn(be=be):
                with sdpa_kernel(be):
                    return F.scaled_dot_product_attention(qh, kh, vh)
            try:
                y = fn().reshape(B, W)
                row[f"max_abs_diff_vs_{bname}"] = float((y.float() - out.float()).abs().max())
                fns[bname] = fn
            except RuntimeError as e:
                row[bname] = dict(unsupported=f"{type(e).__name__}: {str(e)[:160]}")
        samples = {k_: [] for k_ in fns}
        for _ in range(rounds):
            for k_, fn in fns.items():
                samples[k_].append(timeit(fn))
        for k_, s in samples.items():
            tb_s = bytes_kv / statistics.median(s) * 1e-9
            row[k_] = dict(summary(s), tb_s=tb_s, of_copy_bw=tb_s / copy_tb_s)
        for k_ in samples:
            if k_ != "b200enc":
                row[f"speedup_vs_{k_}"] = row[k_]["ms"] / row["b200enc"]["ms"]
        table[name] = row
        print("decode", name, json.dumps(row), flush=True)
        del kv, qkv, work
        torch.cuda.empty_cache()
    return table


class TorchKV:
    """GPT-2 in PyTorch bf16 eager with its own KV cache: F.linear / F.layer_norm / SDPA on the model's weights."""

    def __init__(self, m, B, capacity):
        self.sd = {k: v.detach().bfloat16() for k, v in m.state_dict().items()}
        self.n_layers = len(m.layers)
        self.d = m.token_embs.weight.shape[1]
        self.H = self.d // 64
        self.k = torch.empty(self.n_layers, B, self.H, capacity, 64, device="cuda", dtype=torch.bfloat16)
        self.v = torch.empty_like(self.k)
        self.n = 0

    def __call__(self, ids):
        sd, d, H = self.sd, self.d, self.H
        B, L = ids.shape
        x = F.embedding(ids, sd["token_embs.weight"]) + sd["pos_embs"][self.n:self.n + L]
        for i in range(self.n_layers):
            p = f"layers.{i}."
            h = F.layer_norm(x, (d,), sd[p + "sa_norm.weight"], sd[p + "sa_norm.bias"])
            q, k, v = (F.linear(h, sd[p + f"sa.{n}_proj.weight"], sd[p + f"sa.{n}_proj.bias"])
                       .view(B, L, H, 64).transpose(1, 2) for n in "qkv")
            self.k[i, :, :, self.n:self.n + L] = k
            self.v[i, :, :, self.n:self.n + L] = v
            a = F.scaled_dot_product_attention(q, self.k[i, :, :, :self.n + L], self.v[i, :, :, :self.n + L],
                                               is_causal=L > 1)
            x = x + F.linear(a.transpose(1, 2).reshape(B, L, d), sd[p + "sa.out_proj.weight"], sd[p + "sa.out_proj.bias"])
            h = F.layer_norm(x, (d,), sd[p + "mlp_norm.weight"], sd[p + "mlp_norm.bias"])
            h = F.gelu(F.linear(h, sd[p + "mlp.linear1.weight"], sd[p + "mlp.linear1.bias"]), approximate="tanh")
            x = x + F.linear(h, sd[p + "mlp.linear2.weight"], sd[p + "mlp.linear2.bias"])
        self.n += L
        x = F.layer_norm(x[:, -1], (d,), sd["norm.weight"], sd["norm.bias"])
        return x @ sd["token_embs.weight"].T


def _wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


@torch.no_grad()
def gpt2_table(rounds, prompt=128, new=256):
    table = {}
    for tag in ("gpt2", "gpt2-medium"):
        torch.manual_seed(0)
        m = pm.GPT2.from_hf(tag).eval().cuda().bfloat16()
        for B in (1, 8, 64):
            ids = torch.randint(0, m.vocab_size, (B, prompt + new), device="cuda")

            def cached(graphed):
                cache = m.new_kv_cache(B, prompt + new)
                m.prefill(ids[:, :prompt], cache)
                step = pm.GraphedStep(m, cache) if graphed else (lambda t: m.step(t, cache))
                return lambda: [step(ids[:, t]) for t in range(prompt, prompt + new)]

            def uncached():
                return [m(ids[:, :t])[:, -1] for t in range(prompt, prompt + new)]

            def torch_kv():
                ref = TorchKV(m, B, prompt + new)
                ref(ids[:, :prompt])
                return lambda: [ref(ids[:, t:t + 1]) for t in range(prompt, prompt + new)]

            variants = {"cached_eager": lambda: cached(False), "cached_graphed": lambda: cached(True),
                        "torch_bf16_kv_cache": torch_kv}
            if B == 1:
                variants["uncached_loop"] = lambda: uncached
            samples = {k_: [] for k_ in variants}
            for r in range(rounds + 1):  # round 0 warms up every variant
                for k_, make in variants.items():
                    run = make()  # set-up (cache, prefill, capture) is outside the timed window
                    ms = _wall(run)
                    if r:
                        samples[k_].append(ms)
            row = dict(model=tag, B=B, prompt=prompt, new_tokens=new)
            for k_, s in samples.items():
                ms = statistics.median(s)
                row[k_] = dict(summary(s), tokens_s=B * new / ms * 1e3, ms_per_step=ms / new)
            table[f"{tag}_b{B}"] = row
            print("gpt2", tag, B, json.dumps(row), flush=True)
        del m
        torch.cuda.empty_cache()
    return table


@torch.no_grad()
def whisper_step(rounds, B=64, frames=1500, steps=32):
    torch.manual_seed(0)
    m = pm.WhisperDecoder(51866, 32, 1280).eval().cuda().bfloat16()
    memory = torch.randn(B, frames, 1280, device="cuda", dtype=torch.bfloat16)
    ids = torch.randint(0, 51866, (B, 4 + steps), device="cuda")

    def fresh():
        cache = m.new_kv_cache(memory, 4 + steps)
        m.prefill(ids[:, :4], cache)
        return cache

    samples = {"eager": [], "graphed": []}
    for r in range(rounds + 1):
        cache = fresh()
        ms = _wall(lambda: [m.step(ids[:, 4 + t], cache) for t in range(steps)])
        cache = fresh()
        g = pm.GraphedStep(m, cache)
        ms_g = _wall(lambda: [g(ids[:, 4 + t]) for t in range(steps)])
        if r:
            samples["eager"].append(ms / steps)
            samples["graphed"].append(ms_g / steps)
        del cache, g
    row = dict(B=B, memory_frames=frames, layers=32, d_model=1280, steps=steps)
    for k_, s in samples.items():
        row[f"{k_}_ms_per_token"] = summary(s)
    cache = fresh()
    rec = ops.profile(True)
    for t in range(steps):
        m.step(ids[:, 4 + t], cache)
    torch.cuda.synchronize()
    ops.profile(False)
    per = collections.defaultdict(float)
    for name, meta, e0, e1 in rec:
        key = name if name != "b200enc_attention_decode" else f"{name}_{'self' if meta['append'] else 'cross'}"
        per[key] += e0.elapsed_time(e1) / steps
    row["profiled_ms_per_token_by_entry_point"] = dict(sorted(per.items(), key=lambda kv: -kv[1]))
    row["profiled_ms_per_token_sum"] = sum(per.values())
    print("whisper", json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = dict(device=device_info(), torch=torch.__version__)
    bw = copy_bandwidth(args.rounds)
    res["hbm_copy"] = bw
    res["decode_attention"] = decode_table(args.rounds, bw["tb_s"])
    res["gpt2"] = gpt2_table(args.rounds)
    res["whisper_large_v3_decoder_step"] = whisper_step(args.rounds)
    res["device_after"] = device_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
