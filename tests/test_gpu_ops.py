"""Per-kernel GPU tests through the C-ABI (ctypes): each op against the same op in fp32 PyTorch on the same bf16-rounded
inputs. Tolerances are bf16 output rounding (2^-9 relative) plus accumulation-order noise."""
from __future__ import annotations

import os
import subprocess

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _close(got, want, atol, rtol):
    err = (got.float() - want.float()).abs()
    bound = atol + rtol * want.float().abs()
    assert bool((err <= bound).all()), f"max err {err.max().item():.4g}, worst excess {(err - bound).max().item():.4g}"


@pytest.mark.parametrize("M,N,K", [(1, 64, 64), (130, 576, 192), (257, 768, 3072), (1000, 2304, 768), (77, 1280, 5120)])
@pytest.mark.parametrize("mode", ["bias", "gelu", "residual", "fold", "fold_gelu"])
def test_linear(M, N, K, mode):
    from pytorch_models_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    x = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    w = (torch.randn(N, K, device="cuda", generator=g) * K ** -0.5).bfloat16()
    b = torch.randn(N, device="cuda", generator=g)
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    ref = x.float() @ w.float().T
    if mode.startswith("fold"):
        stats = torch.stack([torch.randn(M, device="cuda", generator=g) * 0.3,
                             torch.rand(M, device="cuda", generator=g) + 0.5], dim=1).contiguous()
        s = w.float().sum(1)
        ops.linear(x, w, b, out, colsum=s, rowstats=stats, gelu=mode.endswith("gelu"))
        ref = stats[:, 1:2] * (ref - stats[:, 0:1] * s[None]) + b
        if mode.endswith("gelu"):
            ref = F.gelu(ref)
    elif mode == "residual":
        r = torch.randn(M, N, device="cuda", generator=g).bfloat16()
        ops.linear(x, w, b, out, residual=r)
        ref = ref + b + r.float()
    else:
        ops.linear(x, w, b, out, gelu=mode == "gelu")
        ref = ref + b
        if mode == "gelu":
            ref = F.gelu(ref)
    _close(out, ref, 0.02, 0.01)


@pytest.mark.parametrize("L", [1, 5, 64, 128, 129, 197, 257, 576, 1370, 1500])
def test_attention_matches_sdpa(L):
    from pytorch_models_b200 import ops

    B, H = 2, 3
    g = torch.Generator(device="cuda").manual_seed(L)
    qkv = (torch.randn(B, L, 3 * H * 64, device="cuda", generator=g) * 1.5).bfloat16()
    out = torch.empty(B, L, H * 64, device="cuda", dtype=torch.bfloat16)
    q, k, v = qkv[:, :, : H * 64], qkv[:, :, H * 64: 2 * H * 64], qkv[:, :, 2 * H * 64:]
    ops.attention(q, k, v, out, H, 0.125)
    heads = lambda t: t.float().unflatten(-1, (H, 64)).transpose(1, 2)  # noqa: E731
    want = F.scaled_dot_product_attention(heads(q), heads(k), heads(v)).transpose(1, 2).flatten(-2)
    _close(out, want, 0.02, 0.02)


@pytest.mark.parametrize("Lq,Lkv", [(1, 1), (16, 16), (33, 33), (64, 200), (128, 128), (130, 130), (192, 192), (193, 193),
                                    (197, 197), (208, 208), (224, 224), (225, 225), (250, 250), (256, 256), (600, 250),
                                    (700, 100), (1, 197)])
def test_short_sequence_attention(Lq, Lkv):
    """Lkv <= 256 without a mask takes the single-pass kernel (attention_short.cuh): every TMEM layout (rows up to 192,
    224 and 256 keys), ragged row ends, one and many query-tile pairs, cross attention — against fp32 SDPA and against
    the streaming kernel on the same inputs (two independent implementations of the same bf16 contract)."""
    from pytorch_models_b200 import ops

    B, H = 3, 5
    g = torch.Generator(device="cuda").manual_seed(7 * Lq + Lkv)
    q = (torch.randn(B, Lq, H * 64, device="cuda", generator=g) * 1.5).bfloat16()
    kv = (torch.randn(B, Lkv, 2 * H * 64, device="cuda", generator=g) * 1.5).bfloat16()
    k, v = kv[:, :, : H * 64], kv[:, :, H * 64:]
    out = torch.full((B, Lq, H * 64), float("nan"), device="cuda", dtype=torch.bfloat16)
    ref = torch.empty_like(out)
    ops.attention(q, k, v, out, H, 0.125)
    ops.attention(q, k, v, ref, H, 0.125, streaming=True)
    heads = lambda t: t.float().unflatten(-1, (H, 64)).transpose(1, 2)  # noqa: E731
    want = F.scaled_dot_product_attention(heads(q), heads(k), heads(v)).transpose(1, 2).flatten(-2)
    _close(out, want, 0.02, 0.02)
    _close(out, ref.float(), 0.02, 0.02)


def test_short_sequence_attention_many_items():
    """More work items than SMs x 2 stages: the operand ring, the TMEM hand-over between items and the staging buffers
    of the output stores all wrap around many times (ViT-B/16 shape, 197 tokens, 12 heads)."""
    from pytorch_models_b200 import ops

    B, H, L = 96, 12, 197
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = (torch.randn(B, L, 3 * H * 64, device="cuda", generator=g) * 2.0).bfloat16()
    q, k, v = qkv[:, :, : H * 64], qkv[:, :, H * 64: 2 * H * 64], qkv[:, :, 2 * H * 64:]
    out = torch.full((B, L, H * 64), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attention(q, k, v, out, H, 0.125)
    heads = lambda t: t.float().unflatten(-1, (H, 64)).transpose(1, 2)  # noqa: E731
    want = F.scaled_dot_product_attention(heads(q), heads(k), heads(v)).transpose(1, 2).flatten(-2)
    _close(out, want, 0.02, 0.02)
    again = torch.empty_like(out)
    ops.attention(q, k, v, again, H, 0.125)
    assert torch.equal(out, again)  # deterministic


@pytest.mark.parametrize("L", [1, 7, 128, 129, 200, 256, 257, 448, 700, 1024])
def test_causal_attention_matches_sdpa(L):
    """is_causal=True of F.scaled_dot_product_attention (transformer.py:52,97): masked diagonal blocks, K/V blocks
    above the diagonal skipped, query tiles of one item visiting different numbers of blocks."""
    from pytorch_models_b200 import ops

    B, H = 2, 2
    g = torch.Generator(device="cuda").manual_seed(1000 + L)
    qkv = (torch.randn(B, L, 3 * H * 64, device="cuda", generator=g) * 1.5).bfloat16()
    out = torch.empty(B, L, H * 64, device="cuda", dtype=torch.bfloat16)
    q, k, v = qkv[:, :, : H * 64], qkv[:, :, H * 64: 2 * H * 64], qkv[:, :, 2 * H * 64:]
    ops.attention(q, k, v, out, H, 0.125, causal=True)
    heads = lambda t: t.float().unflatten(-1, (H, 64)).transpose(1, 2)  # noqa: E731
    want = F.scaled_dot_product_attention(heads(q), heads(k), heads(v), is_causal=True).transpose(1, 2).flatten(-2)
    _close(out, want, 0.02, 0.02)
    # the first row attends to key 0 only: its output is v[0] exactly
    assert torch.equal(out[:, 0], v[:, 0])


@pytest.mark.parametrize("Lq,Lkv", [(5, 300), (300, 5), (130, 129)])
def test_causal_attention_rectangular(Lq, Lkv):
    """Lq != Lkv keeps SDPA's top-left alignment (key j visible to query i iff j <= i)."""
    from pytorch_models_b200 import ops

    B, H = 2, 1
    q = torch.randn(B, Lq, 64, device="cuda").bfloat16()
    kv = torch.randn(B, Lkv, 128, device="cuda").bfloat16()
    out = torch.empty(B, Lq, 64, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :, :64], kv[:, :, 64:], out, H, 0.125, causal=True)
    mask = torch.ones(Lq, Lkv, device="cuda", dtype=torch.bool).tril()
    heads = lambda t: t.float().unflatten(-1, (H, 64)).transpose(1, 2)  # noqa: E731
    want = F.scaled_dot_product_attention(heads(q), heads(kv[:, :, :64]), heads(kv[:, :, 64:]), attn_mask=mask)
    _close(out, want.transpose(1, 2).flatten(-2), 0.02, 0.02)


@pytest.mark.parametrize("fold", [False, True])
def test_linear_tanh_gelu(fold):
    from pytorch_models_b200 import ops

    M, N, K = 300, 1024, 256
    x = torch.randn(M, K, device="cuda").bfloat16()
    w = (torch.randn(N, K, device="cuda") * K ** -0.5 * 2).bfloat16()
    b = torch.randn(N, device="cuda")
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    ref = x.float() @ w.float().T
    if fold:
        stats = torch.stack([torch.randn(M, device="cuda") * 0.3, torch.rand(M, device="cuda") + 0.5], 1).contiguous()
        s = w.float().sum(1)
        ops.linear(x, w, b, out, colsum=s, rowstats=stats, gelu="tanh")
        ref = stats[:, 1:2] * (ref - stats[:, 0:1] * s[None]) + b
    else:
        ops.linear(x, w, b, out, gelu="tanh")
        ref = ref + b
    _close(out, F.gelu(ref, approximate="tanh"), 0.02, 0.01)
    with pytest.raises(ValueError):
        ops.linear(x, w, b, out, gelu="tanh", residual=out.clone())


@pytest.mark.parametrize("act", ["gelu", "approximate_gelu", "relu", "silu"])
@pytest.mark.parametrize("pre_norm", [True, False])
def test_mlp_and_layer_activations(act, pre_norm):
    """All four activations of the reference MLP (transformer.py:60-65), stand-alone and inside a layer (folded
    LayerNorm for pre-norm), against the same modules in fp32 PyTorch."""
    import pytorch_models_b200 as pm

    torch.manual_seed(0)
    d = 128
    layer = pm.EncoderLayer(d, act=act, pre_norm=pre_norm).eval()
    ref_act = {"gelu": lambda t: F.gelu(t), "approximate_gelu": lambda t: F.gelu(t, approximate="tanh"),
               "relu": F.relu, "silu": F.silu}[act]
    x = torch.randn(3, 50, d)
    mlp = layer.mlp
    want = mlp.linear2(ref_act(mlp.linear1(x)))
    with torch.no_grad():
        got = mlp.cuda()(x.cuda()).cpu()
    _close(got, want.detach(), 0.02, 0.02)
    # whole layer: reference arithmetic in fp32 on the CPU copy of the same parameters
    layer = layer.cpu()
    with torch.no_grad():
        def mha(t):
            q, k, v = (getattr(layer.sa, n)(t).unflatten(-1, (2, 64)).transpose(1, 2) for n in ("q_proj", "k_proj", "v_proj"))
            return layer.sa.out_proj(F.scaled_dot_product_attention(q, k, v).transpose(1, 2).flatten(-2))
        ff = lambda t: mlp.linear2(ref_act(mlp.linear1(t)))  # noqa: E731
        if pre_norm:
            h = x + mha(layer.sa_norm(x))
            want = h + ff(layer.mlp_norm(h))
        else:
            h = layer.sa_norm(x + mha(x))
            want = layer.mlp_norm(h + ff(h))
        got = layer.cuda()(x.cuda()).cpu()
    _close(got, want, 0.05, 0.02)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_embed_rows(dtype):
    from pytorch_models_b200 import ops

    B, L, V, d = 3, 17, 101, 72
    tok = torch.randn(V, d, device="cuda").to(dtype)
    pos = torch.randn(L + 4, d, device="cuda").to(dtype)
    ids = torch.randint(0, V, (B, L), device="cuda")
    out = torch.empty(B, L, d, device="cuda", dtype=torch.bfloat16)
    ops.embed_rows(ids, tok, pos, out)
    want = (tok[ids].float() + pos[:L].float()).bfloat16()
    assert torch.equal(out, want)
    ids[1, 3] = V  # out of range: that row is NaN, the others are untouched
    ops.embed_rows(ids, tok, pos, out)
    assert bool(out[1, 3].isnan().all())
    ok = torch.ones(B, L, dtype=torch.bool, device="cuda")
    ok[1, 3] = False
    assert torch.equal(out[ok], want[ok])


@pytest.mark.parametrize("shape", ["LL", "HLL", "B1LL", "BHLL", "bool"])
@pytest.mark.parametrize("causal", [False, True])
def test_attention_bias_matches_sdpa(shape, causal):
    """attn_bias of MHA.forward (transformer.py:41,52) in every broadcast shape SDPA accepts, float and bool, alone
    and combined with the causal flag; -inf entries mask keys."""
    import pytorch_models_b200 as pm

    torch.manual_seed(3)
    B, H, L, d = 2, 2, 200, 128
    mha = pm.MHA(d).eval().cuda()
    x = torch.randn(B, L, d, device="cuda")
    full = torch.randn(B, H, L, L, device="cuda") * 2
    full[:, :, :, 150:170] = float("-inf")   # a band of masked keys
    bias = {"LL": full[0, 0], "HLL": full[0], "B1LL": full[:, :1], "BHLL": full,
            "bool": torch.rand(L, L, device="cuda") > 0.3}[shape]
    if shape == "bool":
        bias = bias | torch.eye(L, device="cuda", dtype=torch.bool)  # keep every row attendable
    with torch.no_grad():
        got = mha(x, attn_bias=bias, causal=causal)
        q, k, v = (getattr(mha, n)(x).unflatten(-1, (H, 64)).transpose(1, 2) for n in ("q_proj", "k_proj", "v_proj"))
        mask = bias if bias.dtype != torch.bool else torch.zeros(L, L, device="cuda").masked_fill(~bias, float("-inf"))
        if causal:
            mask = mask + torch.zeros(L, L, device="cuda").masked_fill(
                ~torch.ones(L, L, device="cuda", dtype=torch.bool).tril(), float("-inf"))
        want = mha.out_proj(F.scaled_dot_product_attention(q, k, v, attn_mask=mask).transpose(1, 2).flatten(-2))
    _close(got, want, 0.03, 0.03)


@pytest.mark.parametrize("gain", [0.05, 4.0, 12.0])
@pytest.mark.parametrize("causal", [False, True])
def test_attention_extreme_score_ranges(gain, causal):
    """Nearly uniform and extremely peaked softmax rows (|score| up to a few hundred): the lazily updated maximum
    (rescale only beyond 2^8 of head-room), the accumulator rescale in TMEM and the polynomial exp2 must hold."""
    from pytorch_models_b200 import ops

    B, H, L = 2, 2, 700
    g = torch.Generator(device="cuda").manual_seed(int(gain * 100) + causal)
    qkv = torch.randn(B, L, 3 * H * 64, device="cuda", generator=g)
    qkv[..., : 2 * H * 64] *= gain                      # q and k: scores ~ gain^2 * 8 * N(0,1)
    qkv[:, 500:, H * 64: 2 * H * 64] *= 3.0             # late keys dominate: forces rescales in later blocks
    qkv = qkv.bfloat16()
    out = torch.empty(B, L, H * 64, device="cuda", dtype=torch.bfloat16)
    q, k, v = qkv[:, :, : H * 64], qkv[:, :, H * 64: 2 * H * 64], qkv[:, :, 2 * H * 64:]
    ops.attention(q, k, v, out, H, 0.125, causal=causal)
    heads = lambda t: t.double().unflatten(-1, (H, 64)).transpose(1, 2)  # noqa: E731
    want = F.scaled_dot_product_attention(heads(q), heads(k), heads(v), is_causal=causal).transpose(1, 2).flatten(-2)
    assert bool(torch.isfinite(out).all())
    _close(out, want.float(), 0.03, 0.03)


def test_cross_attention_one_query():
    """The MAP-pooling shape (vit.py:41): 1 query row against L keys."""
    from pytorch_models_b200 import ops

    B, H, L = 3, 2, 576
    q = torch.randn(B, 1, H * 64, device="cuda").bfloat16()
    kv = torch.randn(B, L, 2 * H * 64, device="cuda").bfloat16()
    out = torch.empty(B, 1, H * 64, device="cuda", dtype=torch.bfloat16)
    ops.attention(q, kv[:, :, : H * 64], kv[:, :, H * 64:], out, H, 0.125)
    heads = lambda t: t.float().unflatten(-1, (H, 64)).transpose(1, 2)  # noqa: E731
    want = F.scaled_dot_product_attention(heads(q), heads(kv[:, :, : H * 64]), heads(kv[:, :, H * 64:]))
    _close(out, want.transpose(1, 2).flatten(-2), 0.02, 0.02)


@pytest.mark.parametrize("rows,d,eps", [(1, 64, 1e-5), (333, 192, 1e-6), (1000, 768, 1e-6), (77, 1280, 1e-5), (50, 768, 1e-12)])
def test_layernorm_and_row_stats(rows, d, eps):
    from pytorch_models_b200 import ops

    x = (torch.randn(rows, d, device="cuda") * 2 + 0.7).bfloat16()
    gmm, bta = torch.randn(d, device="cuda"), torch.randn(d, device="cuda")
    out = torch.empty_like(x)
    stats = torch.empty(rows, 2, device="cuda")
    ops.layernorm(x, gmm, bta, eps, out, stats)
    want = F.layer_norm(x.float(), (d,), gmm, bta, eps)
    _close(out, want, 0.02, 0.01)
    stats2 = torch.empty(rows, 2, device="cuda")
    ops.row_stats(x, eps, stats2)
    mean = x.float().mean(1)
    rstd = (x.float().var(1, unbiased=False) + eps).rsqrt()
    for s in (stats, stats2):
        torch.testing.assert_close(s[:, 0], mean, atol=1e-5, rtol=1e-5)
        torch.testing.assert_close(s[:, 1], rstd, atol=1e-5, rtol=1e-4)


def test_bad_arguments_raise():
    from pytorch_models_b200 import ops

    x = torch.randn(4, 60, device="cuda").bfloat16()  # K not a multiple of 8
    w = torch.randn(8, 60, device="cuda").bfloat16()
    with pytest.raises(ValueError):
        ops.linear(x, w, None, torch.empty(4, 8, device="cuda", dtype=torch.bfloat16))
    with pytest.raises(RuntimeError):
        ops.linear(x.cpu(), w, None, torch.empty(4, 8, device="cuda", dtype=torch.bfloat16))
    q = torch.randn(1, 4, 96, device="cuda").bfloat16()
    with pytest.raises(ValueError):  # head_dim 32
        ops.attention(q, q, q, torch.empty_like(q), 3, 1.0)


@pytest.mark.parametrize("case", ["linear:tails_tma", "linear:embed_like", "linear:fold_gelu", "linear:fold_gelu_tanh", "linear:relu", "linear:fold_silu",
                                  "attn:l197_tmem", "attn:cross_q1", "attn:causal_l448", "attn:causal_many", "attn:l576_tmem",
                                  "attn:l1370_tmem", "attn:l1500_wide", "attn:causal_l128", "rows:all"])
def test_native_selftest(case):
    """The stand-alone C++ harness (fp64 CPU check inside the binary) on its edge-case shapes."""
    exe = os.path.join(ROOT, "pytorch_models_b200", "b200enc_selftest")
    if not os.path.exists(exe):
        pytest.skip("self-test binary not built")
    r = subprocess.run([exe, case], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("M,d,N", [(300, 768, 2304), (130, 192, 576), (64, 1280, 1280), (257, 1024, 4096)])
def test_fused_layernorm_statistics_chain(M, d, N):
    """Producer GEMM (+residual) emits per-128-column (mean, M2); the next GEMM folds LayerNorm from those partials.
    Must agree with LayerNorm -> Linear computed in fp32 on the producer's (bf16) output."""
    from pytorch_models_b200 import ops
    from pytorch_models_b200.transformer import pack_folded

    g = torch.Generator(device="cuda").manual_seed(d + M)
    a = torch.randn(M, d, device="cuda", generator=g).bfloat16()
    w0 = (torch.randn(d, d, device="cuda", generator=g) * d ** -0.5).bfloat16()
    b0 = torch.randn(d, device="cuda", generator=g)
    res = (torch.randn(M, d, device="cuda", generator=g) * 2 + 0.5).bfloat16()
    x = torch.empty(M, d, device="cuda", dtype=torch.bfloat16)
    parts = torch.empty(M, (d + 127) // 128, 2, device="cuda")
    ops.linear(a, w0, b0, x, residual=res, stats_out=parts)

    lin = torch.nn.Linear(d, N).cuda()
    norm = torch.nn.LayerNorm(d, 1e-6).cuda()
    with torch.no_grad():
        norm.weight.normal_(1.0, 0.1, generator=g)
        norm.bias.normal_(0.0, 0.1, generator=g)
        pk = pack_folded([lin], norm)
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        ops.linear(x, pk.w, pk.bias, out, colsum=pk.colsum, rowstats=parts, ln_eps=1e-6)
        want = lin(norm(x.float()))
        # the standalone statistics kernel must give the same result up to rounding
        stats = torch.empty(M, 2, device="cuda")
        ops.row_stats(x, 1e-6, stats)
        out2 = torch.empty_like(out)
        ops.linear(x, pk.w, pk.bias, out2, colsum=pk.colsum, rowstats=stats)
    _close(out, want, 0.03, 0.02)
    _close(out, out2, 0.01, 0.01)


@pytest.mark.parametrize("n,H,W,d,cls", [(2, 224, 224, 768, True), (1, 384, 384, 1024, False), (3, 64, 48, 256, True),
                                         (5, 16, 16, 64, False), (2, 272, 400, 384, True), (200, 32, 32, 128, True)])
def test_patch_embed16_matches_conv2d(n, H, W, d, cls):
    """The im2col-free patch embedding (b200enc_patch_embed16: the GEMM reads the NCHW image through a 5-D tensor map)
    against ``F.conv2d(stride=16)`` + flatten/transpose + pe in fp32 (image/vit.py:64,78-79), with and without room for
    a class token, ragged patch grids, more tiles than SMs; its fused LayerNorm statistics against the stored rows; and
    against the materialised-patch-row path (patch_rows + linear) on the same inputs."""
    from pytorch_models_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(n * 1000 + H + W)
    imgs = torch.randn(n, 3, H, W, device="cuda", generator=g).bfloat16()
    w = (torch.randn(d, 3, 16, 16, device="cuda", generator=g) * 0.05).bfloat16()
    bias = torch.randn(d, device="cuda", generator=g)
    P = (H // 16) * (W // 16)
    pe = torch.randn(P, d, device="cuda", generator=g).bfloat16()
    off = 1 if cls else 0
    tokens = torch.full((n, P + off, d), 7.0, device="cuda", dtype=torch.bfloat16)
    n_sl = (d + 127) // 128
    stats = torch.full((n, P + off, n_sl, 2), -3.0, device="cuda")
    ops.patch_embed16(imgs, w.view(d, 768), bias, pe, tokens[:, off:, :], stats_out=stats, stats_rows=P + off,
                      stats_row_offset=off)
    want = F.conv2d(imgs.float(), w.float(), bias, stride=16).flatten(2).transpose(1, 2) + pe.float()
    _close(tokens[:, off:], want, 0.03, 0.01)
    if cls:  # the class-token rows (and their statistics) are not touched
        assert torch.all(tokens[:, 0] == 7.0) and torch.all(stats[:, 0] == -3.0)
    got = tokens[:, off:].float()
    pad = n_sl * 128 - d
    sl = F.pad(got, (0, pad)).unflatten(-1, (n_sl, 128))
    cnt = torch.tensor([min(128, d - 128 * i) for i in range(n_sl)], device="cuda", dtype=torch.float32)
    mean = sl.sum(-1) / cnt
    mask = (torch.arange(128, device="cuda")[None, :] < cnt[:, None]).float()
    m2 = (((sl - mean[..., None]) ** 2) * mask).sum(-1)
    assert torch.allclose(stats[:, off:, :, 0], mean, atol=2e-3, rtol=1e-3)
    assert torch.allclose(stats[:, off:, :, 1], m2, atol=2e-2, rtol=2e-3)
    # the other path: materialised patch rows + the generic GEMM
    rows = torch.empty(n, P, 768, device="cuda", dtype=torch.bfloat16)
    ref = torch.empty(n, P, d, device="cuda", dtype=torch.bfloat16)
    ops.patch_rows(imgs, 16, 768, rows)
    ops.linear(rows, w.view(d, 768), bias, ref, residual=pe.unsqueeze(0))
    _close(tokens[:, off:], ref.float(), 0.02, 0.01)


def test_patch_embed16_rejects_bad_arguments():
    from pytorch_models_b200 import ops

    imgs = torch.zeros(1, 3, 40, 32, device="cuda", dtype=torch.bfloat16)
    w = torch.zeros(64, 768, device="cuda", dtype=torch.bfloat16)
    bias = torch.zeros(64, device="cuda")
    with pytest.raises(ValueError):
        ops.patch_embed16(imgs, w, bias, torch.zeros(4, 64, device="cuda", dtype=torch.bfloat16),
                          torch.zeros(1, 4, 64, device="cuda", dtype=torch.bfloat16))
    with pytest.raises(TypeError):
        ops.patch_embed16(torch.zeros(1, 3, 32, 32, device="cuda"), w, bias,
                          torch.zeros(4, 64, device="cuda", dtype=torch.bfloat16),
                          torch.zeros(1, 4, 64, device="cuda", dtype=torch.bfloat16))
