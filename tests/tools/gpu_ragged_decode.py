#!/usr/bin/env python
"""Ragged incremental decoding on the B200 (not product code), in one process on one GPU. Kernel times are CUDA events
after warm-up, medians of `--rounds` interleaved rounds; the device name, power limit and SM clocks are queried
(nothing is changed) and stored beside the numbers.

1. b200enc_attention_decode with per-sequence lengths drawn uniformly from [1, capacity], against the shared-length launch
   at the mean length and at the longest length (what padding every sequence to the longest would cost). The K/V
   caches are rotated over enough copies that every launch reads its rows from HBM, not from the 126 MB L2.
2. The shared-length launch of this build against a parent build of libb200enc.so (`--parent-lib`, loaded next to
   this one), alternating the two, on the shapes of profiles/r04/decode.json; outputs compared bitwise. Both builds
   are called through ctypes with the same arguments, so the host cost per call is the same on both sides.
3. GPT-2 small, random weights, greedy, no EOS: `DecoderGenerator.generate_batch` at B = 8 and B = 64 on prompts of
   16-256 tokens with 128 new tokens, against the same prompts one at a time through `generate(use_cache=True)`;
   tokens/s over wall time, prefill and graph capture included.

    python tests/tools/gpu_ragged_decode.py --parent-lib PARENT/libb200enc.so --out profiles/r05/ragged_decode.json
"""
import argparse
import ctypes
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
from pytorch_models_b200 import _lib, ops  # noqa: E402
from gpu_attention_head_dim import device_info, summary, timeit  # noqa: E402
from gpu_decode import SHAPES as SHARED_SHAPES  # noqa: E402

L2_BYTES = 126e6
# name: (B, H, head_dim, capacity)
RAGGED_SHAPES = {
    "gpt2_small_b64_h12_hd64_cap1024": (64, 12, 64, 1024),
    "whisper_large_v3_self_b64_h20_hd64_cap448": (64, 20, 64, 448),
    "b16_h8_hd128_cap8192": (16, 8, 128, 8192),
}


class Caches:
    """Copies of a (B, capacity, 2W) k|v cache and a (B, 3W) q|k|v step buffer, rotated per launch so that the K/V
    rows of consecutive launches do not share L2 lines (together at least 3x the L2)."""

    def __init__(self, B, H, hd, capacity, seed):
        W = H * hd
        self.B, self.H, self.hd, self.W = B, H, hd, W
        g = torch.Generator(device="cuda").manual_seed(seed)
        one = B * capacity * 2 * W * 2
        n = max(1, -(-int(3 * L2_BYTES) // one))
        self.kv = [torch.randn(B, capacity, 2 * W, device="cuda", dtype=torch.bfloat16, generator=g) for _ in range(n)]
        self.qkv = torch.randn(B, 3 * W, device="cuda", dtype=torch.bfloat16, generator=g)
        self.work = torch.empty(ops.decode_workspace_bytes(B, H, hd, capacity) // 4, device="cuda")
        self.out = torch.empty(B, W, device="cuda", dtype=torch.bfloat16)
        self.i = 0

    def launch(self, length, lib=None):
        """One decode attention on the next copy; ``lib``: call this ctypes library's shared-length entry point."""
        W, kv = self.W, self.kv[self.i % len(self.kv)]
        self.i += 1
        q, kn, vn, k, v = self.qkv[:, :W], self.qkv[:, W:2 * W], self.qkv[:, 2 * W:], kv[:, :, :W], kv[:, :, W:]
        if lib is None:
            return ops.attention_decode(q, k, v, self.out, self.H, self.hd ** -0.5, self.work, k_new=kn, v_new=vn,
                                        length=length)
        rc = lib.b200enc_attention_decode(
            q.data_ptr(), q.stride(0), kn.data_ptr(), vn.data_ptr(), kn.stride(0), k.data_ptr(), v.data_ptr(),
            k.stride(0), k.stride(1), k.shape[1], length.data_ptr(), 0, 0, self.out.data_ptr(), self.out.stride(0),
            self.B, self.H, self.hd, self.hd ** -0.5, self.work.data_ptr(), self.work.numel() * 4,
            torch.cuda.current_stream().cuda_stream)
        assert rc == 0, lib.b200enc_last_error()
        return self.out


@torch.no_grad()
def ragged_table(rounds):
    table = {}
    for name, (B, H, hd, cap) in RAGGED_SHAPES.items():
        c = Caches(B, H, hd, cap, B + cap)
        g = torch.Generator().manual_seed(cap)
        keys = torch.randint(1, cap + 1, (B,), generator=g)  # keys per sequence: length + the new row
        lens = (keys - 1).to(torch.int32).cuda()
        mean_len = int(round(float(keys.float().mean()))) - 1
        max_len = int(keys.max()) - 1
        shared_mean = torch.full((1,), mean_len, device="cuda", dtype=torch.int32)
        shared_max = torch.full((1,), max_len, device="cuda", dtype=torch.int32)
        fns = {"ragged": lambda: c.launch(lens), "uniform_mean": lambda: c.launch(shared_mean),
               "uniform_max": lambda: c.launch(shared_max)}
        samples = {k: [] for k in fns}
        for r in range(rounds):
            for k in (list(fns) if r % 2 == 0 else list(fns)[::-1]):
                samples[k].append(timeit(fns[k]))
        row_bytes = c.W * 2 * 2
        read = dict(ragged=int(keys.sum()) * row_bytes, uniform_mean=B * (mean_len + 1) * row_bytes,
                    uniform_max=B * (max_len + 1) * row_bytes)
        row = dict(B=B, H=H, head_dim=hd, capacity=cap, mean_len=mean_len, max_len=max_len, cache_copies=len(c.kv),
                   lengths=lens.tolist())
        for k, s in samples.items():
            row[k] = dict(summary(s), kv_bytes=read[k], tb_s=read[k] / statistics.median(s) * 1e-9)
        row["ragged_over_uniform_mean"] = row["ragged"]["ms"] / row["uniform_mean"]["ms"]
        row["uniform_max_over_ragged"] = row["uniform_max"]["ms"] / row["ragged"]["ms"]
        table[name] = row
        print("ragged", name, json.dumps({k: v for k, v in row.items() if k != "lengths"}), flush=True)
        del c
        torch.cuda.empty_cache()
    return table


def load_parent(path):
    lib = ctypes.CDLL(path)
    restype, argtypes = _lib._SIGNATURES["b200enc_attention_decode"]
    lib.b200enc_attention_decode.restype, lib.b200enc_attention_decode.argtypes = restype, argtypes
    lib.b200enc_last_error.restype = ctypes.c_char_p
    return lib


@torch.no_grad()
def shared_vs_parent(rounds, parent):
    this = _lib.load()
    table = {}
    for name, (B, H, L, hd) in SHARED_SHAPES.items():
        c = Caches(B, H, hd, L, L + hd)
        length = torch.full((1,), L - 1, device="cuda", dtype=torch.int32)
        same = True
        for i in range(len(c.kv)):  # every copy: this build and the parent write the same row and the same output
            before = c.kv[i].clone()
            c.i = i
            a = c.launch(length, this).clone()
            after = c.kv[i].clone()
            c.kv[i].copy_(before)
            c.i = i
            b = c.launch(length, parent).clone()
            same &= torch.equal(a, b) and torch.equal(after, c.kv[i])
        fns = {"this": lambda: c.launch(length, this), "parent": lambda: c.launch(length, parent)}
        samples = {k: [] for k in fns}
        for r in range(rounds):
            for k in (list(fns) if r % 2 == 0 else list(fns)[::-1]):
                samples[k].append(timeit(fns[k]))
        row = dict(B=B, H=H, L=L, head_dim=hd, cache_copies=len(c.kv), bit_identical=bool(same))
        for k, s in samples.items():
            row[k] = summary(s)
        row["this_over_parent"] = row["this"]["ms"] / row["parent"]["ms"]
        table[name] = row
        print("shared", name, json.dumps(row), flush=True)
        del c
        torch.cuda.empty_cache()
    return table


class Tok:  # token ids as text: "3 5 8" <-> [3, 5, 8]; no EOS
    eos_token_id = -1

    def encode(self, s):
        return [int(t) for t in s.split()]

    def decode(self, ids):
        return " ".join(str(i) for i in ids)


def _wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


@torch.no_grad()
def end_to_end(rounds, new=128):
    from pytorch_models_b200.text import DecoderGenerator

    torch.manual_seed(0)
    m = pm.GPT2.from_hf("gpt2").eval().cuda().bfloat16()
    gen = DecoderGenerator(m, Tok())
    g = torch.Generator().manual_seed(5)
    prompts = [" ".join(str(int(t)) for t in torch.randint(0, m.vocab_size, (int(n),), generator=g))
               for n in torch.randint(16, 257, (64,), generator=g)]
    table = {}
    for B in (8, 64):
        ps = prompts[:B]
        gen.generate_batch(ps[:2], max_tokens=4)  # warm-up: module loads, packing
        gen.generate(ps[0], max_tokens=4, use_cache=True)
        samples = {"generate_batch": [], "one_at_a_time": []}
        outs = {}
        for _ in range(rounds):
            ms, outs["generate_batch"] = _wall(lambda: gen.generate_batch(ps, max_tokens=new))
            samples["generate_batch"].append(ms)
            ms, outs["one_at_a_time"] = _wall(lambda: [gen.generate(p, max_tokens=new, use_cache=True) for p in ps])
            samples["one_at_a_time"].append(ms)
        row = dict(B=B, new_tokens=new, prompt_tokens=[len(p.split()) for p in ps],
                   sequences_equal=sum(a == b for a, b in zip(outs["generate_batch"], outs["one_at_a_time"])))
        for k, s in samples.items():
            row[k] = dict(summary(s), tokens_s=B * new / statistics.median(s) * 1e3)
        row["speedup"] = row["generate_batch"]["tokens_s"] / row["one_at_a_time"]["tokens_s"]
        table[f"b{B}"] = row
        print("e2e", B, json.dumps({k: v for k, v in row.items() if k != "prompt_tokens"}), flush=True)
    return table


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--parent-lib", default=None, help="libb200enc.so of the parent build for the shared-length A/B")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = dict(device=device_info(), torch=torch.__version__)
    res["ragged_kernel"] = ragged_table(args.rounds)
    if args.parent_lib:
        res["shared_length_vs_parent"] = shared_vs_parent(args.rounds, load_parent(args.parent_lib))
    res["end_to_end_gpt2_small"] = end_to_end(max(1, args.rounds // 2))
    res["device_after"] = device_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
