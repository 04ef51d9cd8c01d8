#!/usr/bin/env python
"""Wide-head attention on the B200 (not product code): b200enc_attention with head_dim 80 / 96 / 128
(csrc/attention_wide.cuh) against F.scaled_dot_product_attention's flash, cuDNN and mem-efficient backends on the same
fused-QKV views, in one process on one GPU, timed with CUDA events after warm-up; and the ViT-H/14 224 px forward in
img/s at batch 256 against the same math in PyTorch bf16 eager (oracle_torch.vit_forward).

Every timed working set is larger than the 126 MB L2 (the fused QKV buffer alone is 200-500 MB), so K/V are read from
HBM. Each shape is measured in `--rounds` interleaved rounds (ours, then each backend); the median is reported with the
spread. The device name, power limit and SM clocks are queried (nothing is changed) and stored beside the numbers.

    python tests/tools/gpu_attention_head_dim.py --out profiles/r03/attention_head_dim.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import pytorch_models_b200 as pm  # noqa: E402
from pytorch_models_b200 import ops  # noqa: E402
from oracle import oracle_torch  # noqa: E402

# name: (head_dim, B, H, L, causal)
SHAPES = {
    "vit_h14_hd80_b256_h16_l257": (80, 256, 16, 257, False),
    "hd96_b64_h12_l576": (96, 64, 12, 576, False),
    "hd128_b32_h8_l1024": (128, 32, 8, 1024, False),
    "hd128_b32_h8_l1024_causal": (128, 32, 8, 1024, True),
    "hd128_b8_h8_l4096": (128, 8, 8, 4096, False),
}


def device_info():
    q = "name,power.limit,power.max_limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        vals = [v.strip() for v in line.strip().split(",")]
        return dict(zip(q.split(","), vals))
    except (OSError, subprocess.SubprocessError) as e:
        return dict(name=torch.cuda.get_device_name(), query_error=str(e))


def timeit(fn, target_ms=200.0, warm=3):
    """ms per call: warm-up, then enough calls for a window of about target_ms between two CUDA events."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    iters = max(5, min(2000, int(target_ms / max(e0.elapsed_time(e1), 1e-3))))
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def summary(samples):
    return dict(ms=statistics.median(samples), ms_min=min(samples), ms_max=max(samples))


@torch.no_grad()
def attention_table(rounds):
    from torch.nn.attention import SDPBackend, sdpa_kernel

    backends = {"flash": SDPBackend.FLASH_ATTENTION, "cudnn": SDPBackend.CUDNN_ATTENTION,
                "efficient": SDPBackend.EFFICIENT_ATTENTION}
    table = {}
    for name, (hd, B, H, L, causal) in SHAPES.items():
        D = H * hd
        g = torch.Generator(device="cuda").manual_seed(hd + L)
        qkv = torch.randn(B, L, 3 * D, device="cuda", dtype=torch.bfloat16, generator=g)
        q, k, v = (qkv[:, :, i * D:(i + 1) * D] for i in range(3))
        heads = lambda t: t.unflatten(-1, (H, hd)).transpose(1, 2)  # noqa: E731  (B, H, L, hd) views, no copy
        o = torch.empty(B, L, D, device="cuda", dtype=torch.bfloat16)
        ours = lambda: ops.attention(q, k, v, o, H, hd ** -0.5, causal=causal)  # noqa: E731
        fns = {"b200enc": ours}
        for bname, be in backends.items():
            def fn(be=be):
                with sdpa_kernel(be):
                    return F.scaled_dot_product_attention(heads(q), heads(k), heads(v), is_causal=causal)
            fns[bname] = fn
        row = dict(head_dim=hd, B=B, H=H, L=L, causal=causal)
        ours()
        for bname in backends:
            try:
                y = fns[bname]().transpose(1, 2).flatten(-2)
                row[f"max_abs_diff_vs_{bname}"] = float((y.float() - o.float()).abs().max())
            except RuntimeError as e:  # a backend that does not take this shape: reported, not fatal
                row[bname] = dict(error=f"{type(e).__name__}: {str(e)[:200]}")
                fns.pop(bname)
        samples = {k_: [] for k_ in fns}
        for _ in range(rounds):
            for k_, fn in fns.items():
                samples[k_].append(timeit(fn))
        # FLOPs of the two matrix products (causal: the visible half)
        flops = 4.0 * B * H * L * L * hd * (0.5 if causal else 1.0)
        for k_, s in samples.items():
            row[k_] = dict(summary(s), tflops=flops / statistics.median(s) * 1e-9)
        for k_ in samples:
            if k_ != "b200enc":
                row[f"speedup_vs_{k_}"] = row[k_]["ms"] / row["b200enc"]["ms"]
        table[name] = row
        print("attention", name, json.dumps(row), flush=True)
        del qkv, o
        torch.cuda.empty_cache()
    return table


@torch.no_grad()
def vit_h14(batch, rounds):
    torch.manual_seed(0)
    m = pm.ViT.from_google("H/14").eval()
    oracle_torch.randomize_(m.state_dict(), 100)
    m = m.cuda().bfloat16()
    sd = {k: v for k, v in m.state_dict().items()}
    x = torch.randn(batch, 3, 224, 224, device="cuda", dtype=torch.bfloat16)
    ours = lambda: m(x)  # noqa: E731
    eager = lambda: oracle_torch.vit_forward(sd, x, 16, "cls_token")  # noqa: E731
    diff = float((ours().float() - eager().float()).abs().max())
    samples = {"b200enc": [], "torch_eager_bf16": []}
    for _ in range(rounds):
        samples["b200enc"].append(timeit(ours, target_ms=2000.0))
        samples["torch_eager_bf16"].append(timeit(eager, target_ms=2000.0))
    row = dict(batch=batch, img_size=224, tokens=257, head_dim=80, max_abs_diff_pooled=diff)
    for k_, s in samples.items():
        row[k_] = dict(summary(s), img_s=batch / statistics.median(s) * 1e3)
    row["speedup_vs_torch_eager_bf16"] = row["torch_eager_bf16"]["ms"] / row["b200enc"]["ms"]
    print("vit_h14", json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--vit-batch", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = dict(device=device_info(), torch=torch.__version__, l2_note="every working set exceeds the 126 MB L2",
               attention=attention_table(args.rounds), vit_h14_224=vit_h14(args.vit_batch, args.rounds))
    res["device_after"] = device_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
