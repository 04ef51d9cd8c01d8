"""Incremental decoding on the GPU: prefill + KV-cached steps of GPT-2, GPT (post-norm) and the Whisper decoder against
the reference's recorded logits (teacher forcing, the logits bound of test_gpu_parity.py), against the module's own
forward, and a 12-layer d 768 GPT-2 over 512 tokens against the fp32 oracle; CUDA-graph replay of the step; the
cached generator."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from conftest import build_model, error_stats
from oracle import oracle_torch

import pytorch_models_b200 as pm

pytestmark = pytest.mark.gpu

MAX_ABS_12, MIN_COS = 0.125, 0.9999


def _assert_logits(got, want, what):
    """The logits bound of test_gpu_parity.py: max-abs scaled with the output range, per-row cosine."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    scale = max(1.0, float(np.abs(want).max()) / 4.0)
    max_abs, min_cos = error_stats(got, want)
    assert max_abs <= MAX_ABS_12 * scale and min_cos >= MIN_COS, f"{what}: max_abs={max_abs} cos={min_cos}"


def _teacher_forced(m, ids, P, cache):
    """Logits of every position: prefill of ids[:, :P], then one step per remaining token."""
    with torch.no_grad():
        rows = [m.prefill(ids[:, :P], cache).float()]
        for t in range(P, ids.shape[1]):
            rows.append(m.step(ids[:, t], cache).float()[:, None])
    return torch.cat(rows, 1).cpu().numpy()


@pytest.mark.parametrize("name", ["gpt2", "gpt"])
@pytest.mark.parametrize("P", [1, 5, 17])
def test_language_model_teacher_forced(golden, name, P):
    g = golden(name)
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    cache = m.new_kv_cache(ids.shape[0], ids.shape[1])
    got = _teacher_forced(m, ids, P, cache)
    assert cache.n == ids.shape[1] and int(cache.length.item()) == ids.shape[1]
    _assert_logits(got, g.out["logits"], f"{name} vs reference")
    with torch.no_grad():
        own = m(ids).float().cpu().numpy()
    _assert_logits(got, own, f"{name} vs forward")


@pytest.mark.parametrize("P", [1, 4])
def test_whisper_decoder_teacher_forced(golden, P):
    g = golden("whisper_full")
    m = build_model(g).cuda()
    x = torch.from_numpy(np.array(g.input)).cuda()
    targets = torch.from_numpy(np.array(g.extra["targets"])).cuda()
    with torch.no_grad():
        memory = m.encoder(x)
        cache = m.decoder.new_kv_cache(memory, targets.shape[1])
        got = _teacher_forced(m.decoder, targets, P, cache)
        own = m.decoder(targets, memory).float().cpu().numpy()
    _assert_logits(got, g.out["logits"], "whisper vs reference")
    _assert_logits(got, own, "whisper vs forward")


def test_gpt2_small_512_tokens_against_oracle():
    """12 layers, d 768, random weights; prefill 256 tokens, 256 steps; every position against the fp32 oracle."""
    Small = type("GPT2Vocab", (pm.GPT2,), dict(vocab_size=2048))
    torch.manual_seed(0)
    m = Small(12, 768).eval()
    sd = oracle_torch.randomize_(m.state_dict(), 100)
    ids = torch.randint(0, 2048, (1, 512), generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        want = oracle_torch.gpt2_forward(sd, ids[0]).numpy()[None]
    m = m.cuda()
    cache = m.new_kv_cache(1, 512)
    got = _teacher_forced(m, ids.cuda(), 256, cache)
    _assert_logits(got[0], want[0], "GPT-2 12 x 768 vs oracle")


def test_graphed_step_is_bit_identical_to_eager(golden):
    g = golden("gpt2")
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    P, n = 7, 12
    with torch.no_grad():
        eager = m.new_kv_cache(ids.shape[0], ids.shape[1])
        m.prefill(ids[:, :P], eager)
        want = [m.step(ids[:, t], eager) for t in range(P, P + n)]
        cache = m.new_kv_cache(ids.shape[0], ids.shape[1])
        m.prefill(ids[:, :P], cache)
        kv_before = [t.clone() for t in cache.kv]
        step = pm.GraphedStep(m, cache)
        assert cache.n == P and int(cache.length.item()) == P, "capture changed the cache length"
        for kv, before in zip(cache.kv, kv_before):
            assert torch.equal(kv[:, :P], before[:, :P]), "capture changed a filled cache row"
        got = [step(ids[:, t]) for t in range(P, P + n)]
    for t, (a, b) in enumerate(zip(got, want)):
        assert torch.equal(a, b), f"step {t}: graphed and eager logits differ"
    assert cache.n == P + n and int(cache.length.item()) == P + n


def test_generator_with_cache_matches_uncached(golden):
    from pytorch_models_b200.text import DecoderGenerator

    class Tok:  # stand-in tokenizer: "3 5 8" <-> [3, 5, 8]
        eos_token_id = -1

        def encode(self, s):
            return [int(t) for t in s.split()]

        def decode(self, ids):
            return " ".join(str(i) for i in ids)

    g = golden("gpt2")
    m = build_model(g).cuda()
    prompt = "5 17 300 2 41"
    gen = DecoderGenerator(m, Tok())
    plain = [int(t) for t in gen.generate(prompt, max_tokens=20).split()]
    cached = [int(t) for t in gen.generate(prompt, max_tokens=20, use_cache=True).split()]
    assert len(cached) == len(plain) == 25
    if cached != plain:
        i = next(i for i, (a, b) in enumerate(zip(plain, cached)) if a != b)
        with torch.no_grad():
            logits = m(torch.tensor(plain[:i], device="cuda")).float()[-1]
        top2 = logits.topk(2).values
        scale = max(1.0, float(logits.abs().max()) / 4.0)
        assert float(top2[0] - top2[1]) < MAX_ABS_12 * scale, (i, plain, cached)


def test_step_refusals_on_the_gpu(golden):
    g = golden("gpt2")
    m = build_model(g).cuda()
    ids = torch.from_numpy(np.array(g.input)).cuda()
    cache = m.new_kv_cache(2, 3)
    with torch.no_grad():
        m.prefill(ids[:, :2], cache)
        with pytest.raises(ValueError, match="empty cache"):
            m.prefill(ids[:, :1], cache)
        with pytest.raises(ValueError, match="batch"):
            m.step(ids[:1, 2], cache)
        m.step(ids[:, 2], cache)
        with pytest.raises(ValueError, match="full"):
            m.step(ids[:, 2], cache)
        cache.reset()
        m.prefill(ids[:, :3], cache)
    assert cache.n == 3
