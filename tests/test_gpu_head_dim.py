"""Attention with head_dim 80, 96, 112 and 128 (csrc/attention_wide.cuh) on the GPU: every mode of the head_dim-64
kernels against fp32 SDPA on the same bf16 inputs, and the modules that use it (Encoder, Decoder, ViT-H/14) against
the fp32 oracle. Tolerances as in test_gpu_ops.py / test_gpu_parity.py."""
from __future__ import annotations

import pytest
import torch
import torch.nn.functional as F

from conftest import error_stats
from oracle import oracle_torch

import pytorch_models_b200 as pm
from pytorch_models_b200 import ops, plans

pytestmark = pytest.mark.gpu

HEAD_DIMS = [80, 96, 112, 128]
MAX_ABS_12, MAX_ABS_32, MIN_COS = 0.125, 0.15, 0.9999


def _close(got, want, atol, rtol):
    err = (got.float() - want.float()).abs()
    bound = atol + rtol * want.float().abs()
    assert bool((err <= bound).all()), f"max err {err.max().item():.4g}, worst excess {(err - bound).max().item():.4g}"


def _heads(t, H, hd, dtype=torch.float32):
    return t.to(dtype).unflatten(-1, (H, hd)).transpose(1, 2)


def _sdpa(q, k, v, H, hd, dtype=torch.float32, **kw):
    o = F.scaled_dot_product_attention(_heads(q, H, hd, dtype), _heads(k, H, hd, dtype), _heads(v, H, hd, dtype), **kw)
    return o.transpose(1, 2).flatten(-2)


def _fused(B, L, H, hd, seed, gain=1.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    qkv = (torch.randn(B, L, 3 * H * hd, device="cuda", generator=g) * gain).bfloat16()
    w = H * hd
    return qkv, qkv[:, :, :w], qkv[:, :, w:2 * w], qkv[:, :, 2 * w:]


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("L", [1, 5, 128, 129, 257, 576, 1370])
def test_attention_matches_sdpa(hd, L):
    """Self-attention out of a fused [B, L, 3*H*hd] buffer: one and many K/V blocks, ragged block ends, one-row tiles."""
    B, H = 2, 3
    _, q, k, v = _fused(B, L, H, hd, 11 * L + hd)
    out = torch.full((B, L, H * hd), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attention(q, k, v, out, H, hd ** -0.5)
    _close(out, _sdpa(q, k, v, H, hd), 0.02, 0.02)


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("L", [1, 200, 257, 1024])
def test_causal_attention_matches_sdpa(hd, L):
    B, H = 2, 2
    _, q, k, v = _fused(B, L, H, hd, 1000 + L + hd)
    out = torch.empty(B, L, H * hd, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, k, v, out, H, hd ** -0.5, causal=True)
    _close(out, _sdpa(q, k, v, H, hd, is_causal=True), 0.02, 0.02)
    assert torch.equal(out[:, 0], v[:, 0])  # the first row attends to key 0 only


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("Lq,Lkv", [(5, 300), (300, 5)])
def test_causal_attention_rectangular(hd, Lq, Lkv):
    """Lq != Lkv keeps SDPA's top-left alignment (key j visible to query i iff j <= i)."""
    B, H = 2, 1
    q = torch.randn(B, Lq, hd, device="cuda").bfloat16()
    kv = torch.randn(B, Lkv, 2 * hd, device="cuda").bfloat16()
    out = torch.empty(B, Lq, hd, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :, :hd], kv[:, :, hd:], out, H, hd ** -0.5, causal=True)
    mask = torch.ones(Lq, Lkv, device="cuda", dtype=torch.bool).tril()
    _close(out, _sdpa(q, kv[:, :, :hd], kv[:, :, hd:], H, hd, attn_mask=mask), 0.02, 0.02)


@pytest.mark.parametrize("hd", HEAD_DIMS)
def test_cross_attention_one_query(hd):
    """The MAP-pooling shape: 1 query row against 576 keys."""
    B, H, L = 3, 2, 576
    q = torch.randn(B, 1, H * hd, device="cuda").bfloat16()
    kv = torch.randn(B, L, 2 * H * hd, device="cuda").bfloat16()
    out = torch.empty(B, 1, H * hd, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :, :H * hd], kv[:, :, H * hd:], out, H, hd ** -0.5)
    _close(out, _sdpa(q, kv[:, :, :H * hd], kv[:, :, H * hd:], H, hd), 0.02, 0.02)


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("shape", ["LL", "HLL", "B1LL", "BHLL", "bool"])
@pytest.mark.parametrize("causal", [False, True])
def test_attention_bias_matches_sdpa(hd, shape, causal):
    """attn_bias through MHA in every broadcast shape SDPA accepts, float and bool, alone and with the causal flag."""
    torch.manual_seed(3)
    B, H, L, d = 2, 2, 200, 128
    mha = pm.MHA(d, n_heads=H, head_dim=hd).eval().cuda()
    x = torch.randn(B, L, d, device="cuda")
    full = torch.randn(B, H, L, L, device="cuda") * 2
    full[:, :, :, 150:170] = float("-inf")   # a band of masked keys
    bias = {"LL": full[0, 0], "HLL": full[0], "B1LL": full[:, :1], "BHLL": full,
            "bool": torch.rand(L, L, device="cuda") > 0.3}[shape]
    if shape == "bool":
        bias = bias | torch.eye(L, device="cuda", dtype=torch.bool)  # keep every row attendable
    with torch.no_grad():
        got = mha(x, attn_bias=bias, causal=causal)
        q, k, v = (getattr(mha, n)(x).unflatten(-1, (H, hd)).transpose(1, 2) for n in ("q_proj", "k_proj", "v_proj"))
        mask = bias if bias.dtype != torch.bool else torch.zeros(L, L, device="cuda").masked_fill(~bias, float("-inf"))
        if causal:
            mask = mask + torch.zeros(L, L, device="cuda").masked_fill(
                ~torch.ones(L, L, device="cuda", dtype=torch.bool).tril(), float("-inf"))
        want = mha.out_proj(F.scaled_dot_product_attention(q, k, v, attn_mask=mask).transpose(1, 2).flatten(-2))
    _close(got, want, 0.03, 0.03)


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("gain", [0.05, 4.0, 12.0])
def test_attention_extreme_score_ranges(hd, gain):
    """Nearly uniform and extremely peaked rows with late dominant keys: the lazy rescale of all head_dim columns of O."""
    B, H, L = 2, 2, 700
    g = torch.Generator(device="cuda").manual_seed(int(gain * 100) + hd)
    w = H * hd
    qkv = torch.randn(B, L, 3 * w, device="cuda", generator=g)
    qkv[..., :2 * w] *= gain               # q and k: scaled scores ~ gain^2 * N(0,1)
    qkv[:, 500:, w:2 * w] *= 3.0           # late keys dominate: forces rescales in later blocks
    qkv = qkv.bfloat16()
    q, k, v = qkv[:, :, :w], qkv[:, :, w:2 * w], qkv[:, :, 2 * w:]
    out = torch.empty(B, L, w, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, k, v, out, H, hd ** -0.5)
    assert bool(torch.isfinite(out).all())
    _close(out, _sdpa(q, k, v, H, hd, dtype=torch.float64).float(), 0.03, 0.03)


@pytest.mark.parametrize("hd", HEAD_DIMS)
def test_many_items_deterministic(hd):
    """More work items than 2 x SMs (the ViT-H/14 shape): the operand ring, the single Q buffer and the output staging
    wrap around many times; a repeated call is bit-identical."""
    B, H, L = 64, 16, 257
    _, q, k, v = _fused(B, L, H, hd, 5 + hd, gain=2.0)
    out = torch.full((B, L, H * hd), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attention(q, k, v, out, H, hd ** -0.5)
    _close(out, _sdpa(q, k, v, H, hd), 0.02, 0.02)
    again = torch.empty_like(out)
    ops.attention(q, k, v, again, H, hd ** -0.5)
    assert torch.equal(out, again)


# ----------------------------------------------------------------------------------------------- modules
@pytest.mark.parametrize("hd", [80, 128])
@pytest.mark.parametrize("pre_norm", [True, False])
def test_encoder_matches_oracle(hd, pre_norm):
    torch.manual_seed(0)
    d, H = 640, 640 // hd
    m = pm.Encoder(4, d, n_heads=H, pre_norm=pre_norm).eval()
    sd = oracle_torch.randomize_(m.state_dict(), 100)
    x = torch.randn(2, 300, d)
    with torch.no_grad():
        want = oracle_torch.encoder(sd, x, H, pre_norm, 1e-5, prefix="")
        got = m.cuda().bfloat16()(x.cuda().bfloat16()).float().cpu()
    max_abs, min_cos = error_stats(got.numpy(), want.numpy())
    assert max_abs <= MAX_ABS_12 and min_cos >= MIN_COS, (max_abs, min_cos)


def test_decoder_with_memory_matches_oracle():
    """Causal self-attention and cross-attention over a memory of another length, head_dim 128."""
    torch.manual_seed(0)
    d, H = 512, 4
    m = pm.Decoder(3, d, n_heads=H, cross_attn=True).eval()
    sd = oracle_torch.randomize_(m.state_dict(), 100)
    x, mem = torch.randn(2, 77, d), torch.randn(2, 300, d)
    with torch.no_grad():
        want = oracle_torch.decoder(sd, x, mem, H, True, 1e-5, prefix="")
        got = m.cuda().bfloat16()(x.cuda().bfloat16(), mem.cuda().bfloat16()).float().cpu()
    max_abs, min_cos = error_stats(got.numpy(), want.numpy())
    assert max_abs <= MAX_ABS_12 and min_cos >= MIN_COS, (max_abs, min_cos)


def test_vit_h14_matches_oracle_and_replays():
    """ViT-H/14 at 224 px (32 layers, d 1280, 16 heads of 80; 257 tokens through the patch-14 path) against the fp32
    oracle with the 24-32-layer bound; the planned forward (third call) is bit-identical to the per-launch one."""
    torch.manual_seed(0)
    m = pm.ViT.from_google("H/14").eval()
    assert m.layers[0].sa.head_dim == 80
    sd = oracle_torch.randomize_(m.state_dict(), 100)
    torch.manual_seed(1)
    x = torch.randn(2, 3, 224, 224)
    with torch.no_grad():
        want = oracle_torch.vit_forward(sd, x, 16, "cls_token")
        m = m.cuda().bfloat16()
        xb = x.cuda().bfloat16()
        prev = plans.enable(False)
        try:
            per_launch = m(xb)
        finally:
            plans.enable(prev)
        plans.clear(m)
        replays = plans.STATS["replayed"]
        m(xb)                # first sight
        m(xb)                # recorded
        replayed = m(xb)     # replayed
    max_abs, min_cos = error_stats(per_launch.float().cpu().numpy(), want.numpy())
    assert max_abs <= MAX_ABS_32 and min_cos >= MIN_COS, (max_abs, min_cos)
    assert plans.STATS["replayed"] == replays + 1 and torch.equal(replayed, per_launch)
