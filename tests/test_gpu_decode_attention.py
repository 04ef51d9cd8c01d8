"""Single-query attention over a KV cache (csrc/attention_decode.cuh) on the GPU, against fp32 SDPA on the same bf16
inputs with the tolerance of test_gpu_head_dim.py: append mode (the new row comes from the fused q|k|v buffer and is
written into the cache) and cross mode (read-only cache). The cache rows past the keys hold NaN (`_Case.poison`): a
kernel that reads one of them gives NaN, however long the sequence. test_gpu_attention_exact.py checks the same kernel
on inputs whose outputs are known exactly."""
from __future__ import annotations

import pytest
import torch
import torch.nn.functional as F

from pytorch_models_b200 import ops

pytestmark = pytest.mark.gpu

HEAD_DIMS = [64, 80, 96, 112, 128]
GUARD = 8  # cache rows past the new one that must stay untouched


def _same(a, b):
    """Bit for bit, NaN included."""
    return torch.equal(a.view(torch.int16), b.view(torch.int16))


def _close(got, want, atol=0.02, rtol=0.02):
    err = (got.float() - want.float()).abs()
    bound = atol + rtol * want.float().abs()
    assert bool((err <= bound).all()), f"max err {err.max().item():.4g}, worst excess {(err - bound).max().item():.4g}"


def _sdpa1(q, k, v, H, hd):
    """q (B, W), k / v (B, L, W) -> fp32 (B, W)."""
    B, L, _ = k.shape
    qh = q.float().view(B, 1, H, hd).transpose(1, 2)
    kh, vh = (t.float().view(B, L, H, hd).transpose(1, 2) for t in (k, v))
    return F.scaled_dot_product_attention(qh, kh, vh).transpose(1, 2).reshape(B, H * hd)


class _Case:
    """A (B, capacity, 2W) k|v cache, a (B, 3W) fused q|k|v step buffer, a workspace and a device length."""

    def __init__(self, B, H, hd, capacity, seed, gain=1.5):
        g = torch.Generator(device="cuda").manual_seed(seed)
        W = H * hd
        self.B, self.H, self.hd, self.W, self.capacity = B, H, hd, W, capacity
        self.kv = (torch.randn(B, capacity, 2 * W, device="cuda", generator=g) * gain).bfloat16()
        self.qkv = (torch.randn(B, 3 * W, device="cuda", generator=g) * gain).bfloat16()
        self.work = torch.empty(ops.decode_workspace_bytes(B, H, hd, capacity) // 4, device="cuda")
        self.length = torch.zeros(1, device="cuda", dtype=torch.int32)
        self.out = torch.full((B, W), float("nan"), device="cuda", dtype=torch.bfloat16)

    def poison(self, lengths):
        """NaN in every cache row past sequence b's new row (row lengths[b]), as after a rolled-back round."""
        for b, n in enumerate(lengths):
            if 0 <= n < self.capacity:
                self.kv[b, n + 1:] = float("nan")

    def append(self, n):
        W = self.W
        self.length.fill_(n)
        ops.attention_decode(self.qkv[:, :W], self.kv[:, :, :W], self.kv[:, :, W:], self.out, self.H, self.hd ** -0.5,
                             self.work, k_new=self.qkv[:, W:2 * W], v_new=self.qkv[:, 2 * W:], length=self.length)
        return self.out

    def want(self, n):
        W = self.W
        k = torch.cat([self.kv[:, :n, :W], self.qkv[:, None, W:2 * W]], 1)
        v = torch.cat([self.kv[:, :n, W:], self.qkv[:, None, 2 * W:]], 1)
        return _sdpa1(self.qkv[:, :W], k, v, self.H, self.hd)


def _check_append(B, H, hd, L, seed):
    """L keys: L - 1 cached rows plus the new one."""
    c = _Case(B, H, hd, L + GUARD, seed)
    c.poison([L - 1] * B)
    before = c.kv.clone()
    want = c.want(L - 1)
    got = c.append(L - 1)
    torch.cuda.synchronize()
    _close(got, want)
    assert torch.equal(c.kv[:, L - 1], c.qkv[:, c.W:]), "the new k|v row was not written bit for bit"
    assert torch.equal(c.kv[:, :L - 1], before[:, :L - 1]), "a cached row changed"
    assert _same(c.kv[:, L:], before[:, L:]), "the guard band past the new row changed"


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("L", [1, 2, 127, 128, 129, 1000, 4096, 32768])
def test_append_matches_sdpa(hd, L):
    """B·H = 6, below the SM count: most work items are chunks of one (b, h)."""
    _check_append(2, 3, hd, L, 7 * L + hd)


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("L", [1, 129, 4096])
def test_append_many_heads_matches_sdpa(hd, L):
    """B·H = 256, above the SM count of a B200 (148)."""
    _check_append(64, 4, hd, L, 3 * L + hd)


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("B,H", [(2, 3), (64, 4)])
def test_cross_matches_sdpa(hd, B, H):
    """Read-only cache of 1500 rows (Whisper's encoder memory); capacity larger than Lkv; the cache is not written."""
    Lkv = 1500
    c = _Case(B, H, hd, Lkv + GUARD, 99 + hd + B)
    c.kv[:, Lkv:] = float("nan")
    before = c.kv.clone()
    W = c.W
    ops.attention_decode(c.qkv[:, :W], c.kv[:, :, :W], c.kv[:, :, W:], c.out, H, hd ** -0.5, c.work, Lkv=Lkv)
    _close(c.out, _sdpa1(c.qkv[:, :W], c.kv[:, :Lkv, :W], c.kv[:, :Lkv, W:], H, hd))
    assert _same(c.kv, before)


@pytest.mark.parametrize("hd", [64, 128])
def test_same_arguments_at_different_lengths(hd):
    """One set of launch arguments; only the device length changes between calls (what a captured step replays)."""
    c = _Case(3, 5, hd, 2048, 5 + hd)
    for n in (0, 1, 63, 64, 700, 2047):
        want = c.want(n)
        _close(c.append(n).clone(), want)
        assert torch.equal(c.kv[:, n], c.qkv[:, c.W:])


def test_length_past_capacity_gives_nan_and_writes_nothing():
    c = _Case(2, 3, 64, 100, 3)
    before = c.kv.clone()
    got = c.append(100)
    torch.cuda.synchronize()
    assert bool(got.float().isnan().all())
    assert torch.equal(c.kv, before)


@pytest.mark.parametrize("hd", [64, 112])
def test_repeats_are_bit_identical(hd):
    c = _Case(16, 12, hd, 5000, 21 + hd)
    c.poison([4000] * 16)
    first = c.append(4000).clone()
    for _ in range(3):
        assert torch.equal(c.append(4000), first)
