"""Ragged incremental decoding on the GPU: one batch of sequences of different lengths, each with its own device-side
cache length.

Kernel: b200enc_attention_decode with per-sequence lengths against fp32 SDPA per sequence (tolerance of
test_gpu_decode_attention.py), its cache writes, its repeats, its NaN for an out-of-range length, bit-identity with the
shared-length launch at equal lengths; the per-sequence embedding and length update against torch.
Models: ragged prefill + teacher-forced steps of GPT-2, GPT and the Whisper decoder against each sequence's own
unpadded forward and the reference's logits (bound of test_gpu_kv_cache.py), a 12-layer d 768 GPT-2 against the fp32
oracle, equal-length ragged fills against uniform fills, graphed against eager steps, and `generate_batch` against
`generate`."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import build_model
from oracle import oracle_torch
from attention_inputs import decode_chunk
from test_gpu_decode_attention import GUARD, HEAD_DIMS, _Case, _close, _same, _sdpa1
from test_gpu_kv_cache import MAX_ABS_12, _assert_logits

import pytorch_models_b200 as pm
from pytorch_models_b200 import ops

pytestmark = pytest.mark.gpu


class _Ragged(_Case):
    def append_ragged(self, lengths):
        W = self.W
        self.lens = torch.tensor(lengths, device="cuda", dtype=torch.int32)
        ops.attention_decode(self.qkv[:, :W], self.kv[:, :, :W], self.kv[:, :, W:], self.out, self.H, self.hd ** -0.5,
                             self.work, k_new=self.qkv[:, W:2 * W], v_new=self.qkv[:, 2 * W:], length=self.lens)
        return self.out

    def want_seq(self, b, n):
        W = self.W
        k = torch.cat([self.kv[b:b + 1, :n, :W], self.qkv[b:b + 1, None, W:2 * W]], 1)
        v = torch.cat([self.kv[b:b + 1, :n, W:], self.qkv[b:b + 1, None, 2 * W:]], 1)
        return _sdpa1(self.qkv[b:b + 1, :W], k, v, self.H, self.hd)


def _mixed_lengths(B, H, capacity):
    kc = decode_chunk(B, H, capacity)
    base = [0, 1, kc - 1, kc, kc + 1, capacity - 1]
    return [base[i % len(base)] for i in range(B)]


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("B,H", [(6, 3), (12, 20)])
def test_ragged_append_matches_sdpa(hd, B, H):
    """B·H = 18 (below the SM count) and 240 (above); lengths mix 0, 1, kc - 1, kc, kc + 1 and capacity - 1."""
    capacity = 700
    c = _Ragged(B, H, hd, capacity, 11 * hd + B)
    lengths = _mixed_lengths(B, H, capacity)
    c.poison(lengths)
    before = c.kv.clone()
    got = c.append_ragged(lengths).clone()
    torch.cuda.synchronize()
    for b, n in enumerate(lengths):
        _close(got[b:b + 1], c.want_seq(b, n))
        assert torch.equal(c.kv[b, n], c.qkv[b, c.W:]), f"sequence {b}: the new k|v row was not written bit for bit"
        assert torch.equal(c.kv[b, :n], before[b, :n]), f"sequence {b}: a cached row changed"
        assert _same(c.kv[b, n + 1:], before[b, n + 1:]), f"sequence {b}: a row past the new one changed"
    for _ in range(2):
        assert torch.equal(c.append_ragged(lengths), got), "repeats differ"


def test_ragged_guard_band_and_long_lengths():
    """Lengths up to 4096 with a guard band of GUARD rows past the longest; one sequence of length 0."""
    lengths = [4095, 0, 1000, 63, 64, 2049, 129, 4000]
    c = _Ragged(len(lengths), 4, 128, 4096 + GUARD, 5)
    c.poison(lengths)
    before = c.kv.clone()
    got = c.append_ragged(lengths).clone()
    for b, n in enumerate(lengths):
        _close(got[b:b + 1], c.want_seq(b, n))
        assert torch.equal(c.kv[b, n], c.qkv[b, c.W:])
        mask = torch.ones(c.capacity, dtype=torch.bool, device="cuda")
        mask[n] = False
        assert _same(c.kv[b, mask], before[b, mask]), f"sequence {b}: a row other than {n} changed"


@pytest.mark.parametrize("hd", [64, 112])
def test_ragged_length_at_capacity_gives_nan_for_that_sequence_only(hd):
    capacity = 300
    lengths = [5, capacity, 299, -1, 130]
    c = _Ragged(len(lengths), 3, hd, capacity, 3 + hd)
    c.poison(lengths)
    before = c.kv.clone()
    got = c.append_ragged(lengths).clone()
    for b, n in enumerate(lengths):
        if 0 <= n < capacity:
            _close(got[b:b + 1], c.want_seq(b, n))
            assert torch.equal(c.kv[b, n], c.qkv[b, c.W:])
        else:
            assert bool(got[b].float().isnan().all()), f"sequence {b} (length {n}) is not NaN"
            assert _same(c.kv[b], before[b]), f"sequence {b} (length {n}) wrote to the cache"


@pytest.mark.parametrize("hd", HEAD_DIMS)
@pytest.mark.parametrize("B,H,n", [(3, 5, 700), (64, 4, 129), (16, 12, 4000)])
def test_equal_lengths_are_bit_identical_to_the_shared_launch(hd, B, H, n):
    shared = _Ragged(B, H, hd, 4096, 17 + hd)
    ragged = _Ragged(B, H, hd, 4096, 17 + hd)
    want = shared.append(n).clone()
    got = ragged.append_ragged([n] * B)
    assert torch.equal(got, want)
    assert torch.equal(ragged.kv, shared.kv)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_embed_rows_at_and_advance_per_sequence(dtype):
    g = torch.Generator(device="cuda").manual_seed(4)
    vocab, n_pos, d, B = 300, 64, 128, 5
    tok = torch.randn(vocab, d, device="cuda", generator=g).to(dtype)
    pos = torch.randn(n_pos, d, device="cuda", generator=g).to(dtype)
    ids = torch.randint(0, vocab, (B, 1), device="cuda", generator=g)
    lens = torch.tensor([0, 7, 63, 64, 30], device="cuda", dtype=torch.int32)
    out = torch.empty(B, 1, d, device="cuda", dtype=torch.bfloat16)
    ops.embed_rows_at(ids, tok, pos, lens, out)
    want = (tok[ids[:, 0]].float() + pos[lens.clamp(max=n_pos - 1).long()].float()).bfloat16()
    assert torch.equal(out[[0, 1, 2, 4], 0], want[[0, 1, 2, 4]])
    assert bool(out[3].float().isnan().all()), "a position past the table must give a NaN row"
    ops.decode_advance(lens)
    assert lens.tolist() == [1, 8, 64, 65, 31]
    many = torch.arange(1000, device="cuda", dtype=torch.int32)
    ops.decode_advance(many, 3)
    assert torch.equal(many, torch.arange(3, 1003, device="cuda", dtype=torch.int32))


# ---------------------------------------------------------------------------------------------------- models
def _padded(ids, lengths, fill=7):
    """Right-padded prompts: row b keeps ids[b, :lengths[b]], the rest is ``fill``."""
    P = max(lengths)
    x = ids[:, :P].clone()
    for b, n in enumerate(lengths):
        x[b, n:] = fill
    return x


def _ragged_teacher_forced(m, ids, lengths, cache, steps):
    """Per sequence b, the logits of positions [0, lengths[b] + steps): a ragged prefill, then one step per token."""
    with torch.no_grad():
        pre = m.prefill(_padded(ids, lengths), cache, lengths=lengths).float()
        rows = [[pre[b, :n]] for b, n in enumerate(lengths)]
        for t in range(steps):
            nxt = torch.stack([ids[b, n + t] for b, n in enumerate(lengths)])
            out = m.step(nxt, cache).float()
            for b in range(len(lengths)):
                rows[b].append(out[b:b + 1])
    return [torch.cat(r).cpu().numpy() for r in rows]


@pytest.mark.parametrize("name", ["gpt2", "gpt"])
@pytest.mark.parametrize("lengths", [[5, 17], [17, 1], [9, 9]])
def test_language_model_ragged_teacher_forced(golden, name, lengths):
    g = golden(name)
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    L = ids.shape[1]
    steps = L - max(lengths)
    cache = m.new_kv_cache(ids.shape[0], L)
    got = _ragged_teacher_forced(m, ids, lengths, cache, steps)
    assert cache.seq_lengths == [n + steps for n in lengths] and cache.length.tolist() == cache.seq_lengths
    ref = np.asarray(g.out["logits"])
    for b, n in enumerate(lengths):
        with torch.no_grad():
            own = m(ids[b, :n + steps]).float().cpu().numpy()
        _assert_logits(got[b], own, f"{name} sequence {b} vs its own forward")
        _assert_logits(got[b], ref[b, :n + steps], f"{name} sequence {b} vs reference")


@pytest.mark.parametrize("lengths", [[1, 4], [3, 2]])
def test_whisper_decoder_ragged_teacher_forced(golden, lengths):
    g = golden("whisper_full")
    m = build_model(g).cuda()
    x = torch.from_numpy(np.array(g.input)).cuda()
    targets = torch.from_numpy(np.array(g.extra["targets"])).cuda()
    L = targets.shape[1]
    steps = L - max(lengths)
    ref = np.asarray(g.out["logits"])
    with torch.no_grad():
        memory = m.encoder(x)
        cache = m.decoder.new_kv_cache(memory, L)
        got = _ragged_teacher_forced(m.decoder, targets, lengths, cache, steps)
        for b, n in enumerate(lengths):
            own = m.decoder(targets[b:b + 1, :n + steps], memory[b:b + 1]).float()[0].cpu().numpy()
            _assert_logits(got[b], own, f"whisper sequence {b} vs its own forward")
            _assert_logits(got[b], ref[b, :n + steps], f"whisper sequence {b} vs reference")


def test_gpt2_small_ragged_against_oracle():
    """12 layers, d 768, random weights; B = 4 prompts of 1, 37, 200 and 255 tokens, then 256 steps; every position of
    every sequence against the fp32 oracle."""
    Small = type("GPT2Vocab", (pm.GPT2,), dict(vocab_size=2048))
    torch.manual_seed(0)
    m = Small(12, 768).eval()
    sd = oracle_torch.randomize_(m.state_dict(), 100)
    lengths, steps = [1, 37, 200, 255], 256
    ids = torch.randint(0, 2048, (4, 255 + steps), generator=torch.Generator().manual_seed(1))
    m = m.cuda()
    cache = m.new_kv_cache(4, 255 + steps)
    got = _ragged_teacher_forced(m, ids.cuda(), lengths, cache, steps)
    for b, n in enumerate(lengths):
        with torch.no_grad():
            want = oracle_torch.gpt2_forward(sd, ids[b, :n + steps]).numpy()
        _assert_logits(got[b], want, f"GPT-2 12 x 768 sequence {b} (prompt {n}) vs oracle")


def test_equal_length_ragged_fill_matches_uniform_fill(golden):
    g = golden("gpt2")
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    P, B = 9, ids.shape[0]
    with torch.no_grad():
        uni, rag = m.new_kv_cache(B, 32), m.new_kv_cache(B, 32)
        assert torch.equal(m.prefill(ids[:, :P], uni), m.prefill(ids[:, :P], rag, lengths=[P] * B))
        assert not uni.ragged and rag.ragged
        for t in range(P, P + 16):
            assert torch.equal(m.step(ids[:, t], uni), m.step(ids[:, t], rag)), f"step at position {t}"


def test_graphed_ragged_step_is_bit_identical_to_eager(golden):
    g = golden("gpt2")
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    lengths, n = [3, 11], 12
    x = _padded(ids, lengths)
    tokens = [torch.stack([ids[b, k + t] for b, k in enumerate(lengths)]) for t in range(n)]
    with torch.no_grad():
        eager = m.new_kv_cache(2, ids.shape[1])
        m.prefill(x, eager, lengths=lengths)
        want = [m.step(t, eager) for t in tokens]
        cache = m.new_kv_cache(2, ids.shape[1])
        m.prefill(x, cache, lengths=lengths)
        kv_before = [t.clone() for t in cache.kv]
        step = pm.GraphedStep(m, cache)
        assert cache.n == 11 and cache.length.tolist() == lengths, "capture changed the lengths"
        for kv, before in zip(cache.kv, kv_before):
            for b, k in enumerate(lengths):
                assert torch.equal(kv[b, :k], before[b, :k]), "capture changed a filled cache row"
        got = [step(t) for t in tokens]
        for t, (a, b) in enumerate(zip(got, want)):
            assert torch.equal(a, b), f"step {t}: graphed and eager logits differ"
        assert cache.length.tolist() == [k + n for k in lengths] and cache.seq_lengths == [k + n for k in lengths]
        cache.reset()
        m.prefill(ids[:, :4], cache)  # a shared-length fill: the captured step reads the other tensor
        with pytest.raises(ValueError, match="capture a new GraphedStep"):
            step(tokens[0])


class _Tok:  # stand-in tokenizer: "3 5 8" <-> [3, 5, 8]
    def __init__(self, eos=-1):
        self.eos_token_id = eos

    def encode(self, s):
        return [int(t) for t in s.split()]

    def decode(self, ids):
        return " ".join(str(i) for i in ids)


def _agree(m, plain, other):
    """Equal, or first different after a position where the two best logits lie within the bound of
    test_generator_with_cache_matches_uncached."""
    if other == plain:
        return
    i = next(i for i, (a, b) in enumerate(zip(plain, other)) if a != b)
    with torch.no_grad():
        logits = m(torch.tensor(plain[:i], device="cuda")).float()[-1]
    top2 = logits.topk(2).values
    scale = max(1.0, float(logits.abs().max()) / 4.0)
    assert float(top2[0] - top2[1]) < MAX_ABS_12 * scale, (i, plain, other)


def test_generate_batch_matches_generate(golden):
    from pytorch_models_b200.text import DecoderGenerator

    m = build_model(golden("gpt2")).cuda()
    prompts = ["5 17 300 2 41", "9", "1 2 3 4 5 6 7 8 9 10 11 12", "40 41"]
    gen = DecoderGenerator(m, _Tok())
    batch = gen.generate_batch(prompts, max_tokens=20)
    assert len(batch) == len(prompts)
    for p, got in zip(prompts, batch):
        one = [int(t) for t in gen.generate(p, max_tokens=20, use_cache=True).split()]
        got = [int(t) for t in got.split()]
        assert len(got) == len(one) == len(p.split()) + 20
        _agree(m, one, got)


def test_generate_batch_stops_each_sequence_at_its_eos(golden):
    from pytorch_models_b200.text import DecoderGenerator

    m = build_model(golden("gpt2")).cuda()
    prompts = ["5 17 300 2 41", "9", "1 2 3 4 5 6 7 8 9 10 11 12"]
    free = [[int(t) for t in s.split()] for s in DecoderGenerator(m, _Tok()).generate_batch(prompts, max_tokens=12)]
    eos = free[0][len(prompts[0].split()) + 3]  # the 4th token generated for the first prompt
    gen = DecoderGenerator(m, _Tok(eos))
    got = [[int(t) for t in s.split()] for s in gen.generate_batch(prompts, max_tokens=12)]
    for p, f, g_ in zip(prompts, free, got):
        n = len(p.split())
        new = f[n:]
        want = f[:n + new.index(eos) + 1] if eos in new else f
        assert g_ == want, (p, f, g_)
    assert [len(s.split()) for s in gen.generate_batch(prompts, max_tokens=1)] == [len(p.split()) + 1 for p in prompts]
    assert gen.generate_batch(prompts, max_tokens=0) == prompts
