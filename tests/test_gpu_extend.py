"""Extending a filled KV cache by several tokens per sequence, on the GPU.

Kernel: `kv_append` + `attention_extend` (causal attention whose queries start at each sequence's cache length, the
kOffset instantiation of csrc/attention_stream.cuh and csrc/attention_wide.cuh) against fp32 SDPA with an explicit
lower-right causal mask, per sequence, with the tolerance of test_gpu_decode_attention.py. The cache rows past each
sequence's new rows hold NaN, which must neither leak into the outputs nor be overwritten. At offset 0 the kernel must
equal the causal `attention` bit for bit.

Models: `extend` on an empty cache against `prefill` (bit for bit), chunked prefills against `forward`, ragged extends
against each sequence on its own, a 12-layer d 768 GPT-2 fed in chunks against the fp32 oracle, and a `GraphedStep`
captured before an extend against eager steps."""
from __future__ import annotations

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import build_model
from oracle import oracle_torch
from test_gpu_decode_attention import HEAD_DIMS, _close
from test_gpu_kv_cache import _assert_logits

import pytorch_models_b200 as pm
from pytorch_models_b200 import ops

pytestmark = pytest.mark.gpu

CAPACITY = 1024


class _Extend:
    """A (B, capacity, 2W) k|v cache whose rows past each sequence's offset + P are NaN, a (B, P, 3W) q|k|v buffer."""

    def __init__(self, B, H, hd, P, offsets, seed, capacity=CAPACITY, gain=1.5):
        g = torch.Generator(device="cuda").manual_seed(seed)
        W = H * hd
        self.B, self.H, self.hd, self.W, self.P, self.offsets = B, H, hd, W, P, list(offsets)
        self.kv = (torch.randn(B, capacity, 2 * W, device="cuda", generator=g) * gain).bfloat16()
        for b, o in enumerate(self.offsets):
            self.kv[b, o + P:] = float("nan")
        self.qkv = (torch.randn(B, P, 3 * W, device="cuda", generator=g) * gain).bfloat16()
        self.before = self.kv.clone()

    def run(self, shared=False):
        W = self.W
        if shared:
            assert len(set(self.offsets)) == 1
        length = torch.tensor(self.offsets[:1] if shared else self.offsets, device="cuda", dtype=torch.int32)
        out = torch.full((self.B, self.P, W), float("nan"), device="cuda", dtype=torch.bfloat16)
        ops.kv_append(self.qkv[:, :, W:], self.kv, length)
        ops.attention_extend(self.qkv[:, :, :W], self.kv[:, :, :W], self.kv[:, :, W:], out, self.H, self.hd ** -0.5,
                             length)
        return out

    def want(self, b):
        """fp32 SDPA of sequence b: P queries at positions o + i over keys [0, o + P), key j visible iff j <= o + i."""
        H, hd, P, W, o = self.H, self.hd, self.P, self.W, self.offsets[b]
        k = torch.cat([self.before[b, :o, :W], self.qkv[b, :, W:2 * W]]).float()
        v = torch.cat([self.before[b, :o, W:], self.qkv[b, :, 2 * W:]]).float()
        q = self.qkv[b, :, :W].float()
        mask = torch.arange(o + P, device="cuda")[None, :] <= o + torch.arange(P, device="cuda")[:, None]
        heads = lambda t: t.view(t.shape[0], H, hd).transpose(0, 1)  # noqa: E731
        out = F.scaled_dot_product_attention(heads(q), heads(k), heads(v), attn_mask=mask, scale=hd ** -0.5)
        return out.transpose(0, 1).reshape(P, W)

    def check_cache(self):
        """Rows [o, o + P) hold the new k|v rows bit for bit; every other row is untouched (NaN included)."""
        W = self.W
        for b, o in enumerate(self.offsets):
            assert torch.equal(self.kv[b, o:o + self.P], self.qkv[b, :, W:]), f"sequence {b}: appended rows"
            for rows in (slice(0, o), slice(o + self.P, None)):
                assert torch.equal(self.kv[b, rows].view(torch.int16), self.before[b, rows].view(torch.int16)), \
                    f"sequence {b}: a row outside [{o}, {o + self.P}) changed"


def _offsets(B, P):
    """Offset 0, exactly one K/V block, values off the block grid and the last one that fits (capacity - P)."""
    pool = [0, 128, CAPACITY - P, 37, 200, 1, 255, 500, 129, 640]
    return [min(pool[b % len(pool)], CAPACITY - P) for b in range(B)]


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("P", [1, 2, 7, 128, 129, 300])
@pytest.mark.parametrize("B,H", [(3, 2), (10, 20)])  # 6 items, and 200-400 items: both sides of 148 SMs
def test_extend_matches_sdpa(hd, P, B, H):
    c = _Extend(B, H, hd, P, _offsets(B, P), seed=hd * 1000 + P)
    out = c.run()
    torch.cuda.synchronize()
    c.check_cache()
    for b in range(B):
        _close(out[b], c.want(b))
    assert torch.equal(c.run(), out), "repeats differ"


@pytest.mark.parametrize("hd", [64, 128])
@pytest.mark.parametrize("P", [7, 300])
@pytest.mark.parametrize("off", [0, 128, 200, CAPACITY - 300])
def test_shared_length_matches_sdpa_and_equal_per_sequence_lengths(hd, P, off):
    c = _Extend(4, 6, hd, P, [off] * 4, seed=off + P)
    shared = c.run(shared=True)
    c.check_cache()
    for b in range(4):
        _close(shared[b], c.want(b))
    assert torch.equal(c.run(shared=False), shared), "equal per-sequence lengths differ from the shared launch"


@pytest.mark.parametrize("hd", [64, 128])
@pytest.mark.parametrize("L", [1, 7, 128, 300, 1500])
def test_offset_zero_is_the_causal_kernel(hd, L):
    """attention_extend over a cache that kv_append filled == b200enc_attention(B200ENC_ATTN_CAUSAL) on the q|k|v."""
    B, H = 3, 4
    c = _Extend(B, H, hd, L, [0] * B, seed=L, capacity=2048)
    got = c.run()
    W = c.W
    want = torch.empty_like(got)
    ops.attention(c.qkv[:, :, :W], c.qkv[:, :, W:2 * W], c.qkv[:, :, 2 * W:], want, H, hd ** -0.5, causal=True)
    assert torch.equal(got, want)


@pytest.mark.parametrize("hd", [64, 96])
def test_offset_past_capacity_gives_nan_for_that_sequence_only(hd):
    P = 9
    c = _Extend(3, 2, hd, P, [5, 0, 40], seed=3)
    n = CAPACITY - P + 1  # the second sequence's device length does not leave room for P rows
    c.offsets = [5, n, 40]
    out = c.run()
    assert bool(out[1].isnan().all())
    for b in (0, 2):
        _close(out[b], c.want(b))
    # the rows that fit are written, the last one (it would land at the capacity) is not
    assert torch.equal(c.kv[1, :n].view(torch.int16), c.before[1, :n].view(torch.int16))
    assert torch.equal(c.kv[1, n:], c.qkv[1, :P - 1, c.W:])


# ---------------------------------------------------------------------------------------------- models
def _model(golden, name):
    g = golden("whisper_full" if name == "whisper" else name)
    m = build_model(g).cuda()
    if name == "whisper":
        x = torch.from_numpy(np.array(g.input)).cuda()
        ids = torch.from_numpy(np.array(g.extra["targets"])).cuda()
        with torch.no_grad():
            memory = m.encoder(x)
        dec = m.decoder
        new_cache = lambda cap, rows=slice(None): dec.new_kv_cache(memory[rows], cap)  # noqa: E731
        return dec, ids, new_cache, lambda t: dec(t, memory)
    ids = torch.from_numpy(np.array(g.input)).cuda()
    new_cache = lambda cap, rows=slice(None): m.new_kv_cache(ids[rows].shape[0], cap)  # noqa: E731
    return m, ids, new_cache, m


@pytest.mark.parametrize("name", ["gpt2", "gpt", "whisper"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_extend_on_an_empty_cache_is_prefill(golden, name, dtype):
    m, ids, new_cache, _ = _model(golden, name)
    m.to(dtype)
    P = ids.shape[1] - 1
    lengths = [P - b % 3 for b in range(ids.shape[0])]
    with torch.no_grad():
        for lens in (None, lengths):
            a, b = new_cache(ids.shape[1]), new_cache(ids.shape[1])
            want = m.prefill(ids[:, :P], a, lengths=lens)
            got = m.extend(ids[:, :P], b, lengths=lens)
            assert torch.equal(got, want), f"logits (lengths {lens})"
            assert a.seq_lengths == b.seq_lengths and torch.equal(a.length, b.length)
            for i, (ka, kb) in enumerate(zip(a.kv, b.kv)):
                assert torch.equal(ka[:, :P], kb[:, :P]), f"layer {i} cache rows (lengths {lens})"


@pytest.mark.parametrize("name", ["gpt2", "gpt", "whisper"])
def test_prefill_then_extends_then_steps_match_forward(golden, name):
    m, ids, new_cache, forward = _model(golden, name)
    L = ids.shape[1]
    a, b, c = 1, 3, L - 2
    cache = new_cache(L)
    with torch.no_grad():
        rows = [m.prefill(ids[:, :a], cache), m.extend(ids[:, a:b], cache), m.extend(ids[:, b:c], cache)]
        rows += [m.step(ids[:, t], cache)[:, None] for t in range(c, L)]
        got = torch.cat([r.float() for r in rows], 1).cpu().numpy()
        own = forward(ids).float().cpu().numpy()
    assert cache.n == L and cache.length.tolist() == [L]
    _assert_logits(got, own, f"{name}: prefill {a} + extend {b - a} + extend {c - b} + steps vs forward")


@pytest.mark.parametrize("name", ["gpt2", "whisper"])
def test_ragged_extends_match_each_sequence_alone(golden, name):
    m, ids, new_cache, _ = _model(golden, name)
    B, L = ids.shape
    assert B >= 2
    first, P = [3, 1] + [2] * (B - 2), 4
    second = [2, 4] + [1] * (B - 2)
    with torch.no_grad():
        cache = new_cache(L)
        pre = m.extend(ids[:, :max(first)], cache, lengths=first)  # a ragged fill through extend
        x = torch.stack([ids[b, n:n + P] for b, n in enumerate(first)])
        ext = m.extend(x, cache, lengths=second)
        assert cache.ragged and cache.seq_lengths == [f + s for f, s in zip(first, second)]
        step_ids = torch.stack([ids[b, f + s] for b, (f, s) in enumerate(zip(first, second))])
        stp = m.step(step_ids, cache)
        for b in range(B):
            alone = new_cache(L, slice(b, b + 1))
            f, s = first[b], second[b]
            want = [m.extend(ids[b:b + 1, :f], alone), m.extend(ids[b:b + 1, f:f + s], alone),
                    m.step(ids[b:b + 1, f + s], alone)[:, None]]
            got = [pre[b:b + 1, :f], ext[b:b + 1, :s], stp[b:b + 1, None]]
            _assert_logits(torch.cat([g.float() for g in got], 1).cpu().numpy(),
                           torch.cat([w.float() for w in want], 1).cpu().numpy(), f"{name} sequence {b}")


def test_gpt2_small_in_chunks_against_oracle():
    """12 layers, d 768, random weights, two sequences fed as extends of 1 + 37 + 200 + 18 tokens, then 8 steps; every
    position against the fp32 oracle with the bound of test_gpu_ragged_decode.py."""
    Small = type("GPT2Vocab", (pm.GPT2,), dict(vocab_size=2048))
    torch.manual_seed(0)
    m = Small(12, 768).eval()
    sd = oracle_torch.randomize_(m.state_dict(), 100)
    chunks, steps = [1, 37, 200, 18], 8
    n = sum(chunks)
    ids = torch.randint(0, 2048, (2, n + steps), generator=torch.Generator().manual_seed(1))
    m = m.cuda()
    x = ids.cuda()
    cache = m.new_kv_cache(2, n + steps)
    rows, at = [], 0
    with torch.no_grad():
        for k in chunks:
            rows.append(m.extend(x[:, at:at + k], cache).float())
            at += k
        rows += [m.step(x[:, t], cache).float()[:, None] for t in range(n, n + steps)]
    got = torch.cat(rows, 1).cpu().numpy()
    for b in range(2):
        with torch.no_grad():
            want = oracle_torch.gpt2_forward(sd, ids[b]).numpy()
        _assert_logits(got[b], want, f"GPT-2 12 x 768 sequence {b} in chunks {chunks} vs oracle")


@pytest.mark.parametrize("lengths", [None, [3, 6]])
def test_graphed_step_captured_before_an_extend(golden, lengths):
    """The step reads the device lengths, so a graph captured before an extend keeps replaying correctly after it
    (here on a ragged fill, so that an extend with unequal lengths keeps the cache's kind)."""
    g = golden("gpt2")
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()[:2]
    L = ids.shape[1]
    fill = [2, 4]
    P = 6
    x = torch.stack([ids[b, n:n + P] for b, n in enumerate(fill)])
    grown = [f + (P if lengths is None else k) for f, k in zip(fill, lengths or [P, P])]
    tokens = [torch.stack([ids[b, n + t] for b, n in enumerate(grown)]) for t in range(L - max(grown))]
    with torch.no_grad():
        eager = m.new_kv_cache(2, L)
        m.prefill(ids[:, :max(fill)], eager, lengths=fill)
        m.extend(x, eager, lengths=lengths)
        want = [m.step(t, eager) for t in tokens]
        cache = m.new_kv_cache(2, L)
        m.prefill(ids[:, :max(fill)], cache, lengths=fill)
        step = pm.GraphedStep(m, cache)
        m.extend(x, cache, lengths=lengths)
        got = [step(t) for t in tokens]
    for t, (a, b) in enumerate(zip(got, want)):
        assert torch.equal(a, b), f"step {t}: graphed and eager logits differ"
    assert cache.seq_lengths == eager.seq_lengths and torch.equal(cache.length, eager.length)
