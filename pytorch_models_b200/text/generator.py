"""Text generation around a decoder-only language model, API-compatible with the reference's ``DecoderGenerator``
(``pytorch_models/text/generator.py:11-39``): ``DecoderGenerator(model, tokenizer).generate(prompt, max_tokens, topk)``.

Behaviour kept from the reference: the prompt is encoded with ``tokenizer.encode``, one token is appended per model
call on the whole prefix (no KV cache; ``use_cache=True`` decodes incrementally instead), ``topk == 1`` is greedy, otherwise the next token is sampled from the softmax of
the ``topk`` largest logits, and generation stops after ``max_tokens`` new tokens or at ``tokenizer.eos_token_id``.
The model call is the sm_100a forward of ``GPT2`` / ``GPT`` (1-D token tensor in, ``(L, vocab)`` logits out).
"""
from __future__ import annotations

import torch
from torch import Tensor, nn

from .. import speculative
from ..graphs import GraphedStep, SpeculativeRound


def _pick(last_logits: Tensor, topk: int) -> int:
    """Next token id from the logits of the last position."""
    scores = last_logits.float()
    if topk <= 1:
        return int(scores.argmax(dim=-1))
    best, ids = scores.topk(topk)
    choice = torch.multinomial(torch.softmax(best, dim=-1), num_samples=1)
    return int(ids[choice])


def _pick_rows(logits: Tensor, topk: int) -> Tensor:
    """`_pick` for every row of (B, vocab) logits at once -> (B,) int64 device tensor, without a host synchronisation."""
    scores = logits.float()
    if topk <= 1:
        return scores.argmax(dim=-1)
    best, ids = scores.topk(topk, dim=-1)
    choice = torch.multinomial(torch.softmax(best, dim=-1), num_samples=1)
    return ids.gather(1, choice)[:, 0]


class DecoderGenerator:
    def __init__(self, model: nn.Module, tokenizer) -> None:
        self.model = model
        self.tokenizer = tokenizer

    @staticmethod
    def _check_draft(draft, topk: int, use_cache: bool = True) -> None:
        if draft is None:
            return
        if topk > 1:
            raise NotImplementedError(f"speculative decoding is greedy (topk=1), got topk={topk}")
        if not use_cache:
            raise ValueError("speculative decoding (draft=...) needs use_cache=True")

    @torch.inference_mode()
    def generate(self, prompt: str, max_tokens: int = 100, topk: int = 1, use_cache: bool = False, draft=None,
                 draft_tokens: int = 4) -> str:
        """``use_cache=True``: one prefill of the prompt into a KV cache, then one CUDA-graph replay of
        ``model.step`` per new token (`graphs.GraphedStep`) instead of a forward over the whole prefix. Same stopping
        rules and sampling; the logits agree with the uncached ones within bf16 rounding, so greedy decoding can take
        a different branch where the two best logits are closer than that.

        ``draft``: a smaller model of the same vocabulary (``GPT2`` / ``GPT``) for greedy speculative decoding
        (``use_cache=True``, ``topk=1``): it proposes ``draft_tokens`` tokens per round, one extend of the model
        verifies them, and the accepted ones cost no step of the model (`graphs.SpeculativeRound`). The result is the
        model's own greedy result, up to the near-ties above. ``draft=NGramDraft()`` proposes without a second model:
        the tokens that followed the latest earlier occurrence of the sequence's last few tokens in its own prompt and
        output (`speculative.NGramDraft`)."""
        self._check_draft(draft, topk, use_cache)
        device = next(self.model.parameters()).device
        eos = self.tokenizer.eos_token_id
        ids = list(self.tokenizer.encode(prompt))
        if draft is not None and max_tokens > 0:
            return self.tokenizer.decode(self._generate_speculative([ids], max_tokens, eos, draft, draft_tokens,
                                                                    device, ragged=False)[0])
        if use_cache and max_tokens > 0:
            return self.tokenizer.decode(self._generate_cached(ids, max_tokens, topk, eos, device))
        for _ in range(max_tokens):
            prefix = torch.tensor(ids, device=device, dtype=torch.long)
            ids.append(_pick(self.model(prefix)[-1], topk))
            if ids[-1] == eos:
                break
        return self.tokenizer.decode(ids)

    @torch.inference_mode()
    def generate_batch(self, prompts: list[str], max_tokens: int = 100, topk: int = 1, draft=None,
                       draft_tokens: int = 4) -> list[str]:
        """`generate` (``use_cache=True``) for several prompts of any lengths at once: one ragged prefill of the
        right-padded prompts (``model.prefill(..., lengths=...)``), then one CUDA-graph replay of ``model.step`` per
        token for the whole batch, with one host synchronisation per step to read the picked tokens. Each sequence
        stops at its own EOS (the batch keeps stepping; its later tokens are dropped) or after ``max_tokens`` new
        tokens. Returns one string per prompt, what ``generate(prompt, max_tokens, topk, use_cache=True)`` returns up
        to bf16 rounding (see `generate`). ``draft``: speculative decoding of the whole batch, as in `generate`."""
        self._check_draft(draft, topk)
        device = next(self.model.parameters()).device
        eos = self.tokenizer.eos_token_id
        seqs = [list(self.tokenizer.encode(p)) for p in prompts]
        if not seqs or max_tokens <= 0:
            return [self.tokenizer.decode(s) for s in seqs]
        if draft is not None:
            seqs = self._generate_speculative(seqs, max_tokens, eos, draft, draft_tokens, device, ragged=True)
            return [self.tokenizer.decode(s) for s in seqs]
        lengths = [len(s) for s in seqs]
        P = max(lengths)
        ids = torch.zeros(len(seqs), P, dtype=torch.long)
        for b, s in enumerate(seqs):
            ids[b, :len(s)] = torch.tensor(s, dtype=torch.long)
        cache = self.model.new_kv_cache(len(seqs), min(self.model.max_seq_len, P + max_tokens))
        logits = self.model.prefill(ids.to(device), cache, lengths=lengths)
        last = logits[torch.arange(len(seqs), device=device), torch.tensor(lengths, device=device) - 1]
        done = [False] * len(seqs)
        step = None
        for i in range(max_tokens):
            picked = _pick_rows(last, topk)
            for b, t in enumerate(picked.tolist()):
                if not done[b]:
                    seqs[b].append(t)
                    done[b] = t == eos
            if all(done) or i + 1 == max_tokens:
                break
            if step is None:
                step = GraphedStep(self.model, cache)
            last = step(picked)
        return [self.tokenizer.decode(s) for s in seqs]

    def _generate_cached(self, ids: list, max_tokens: int, topk: int, eos, device) -> list:
        cache = self.model.new_kv_cache(1, min(self.model.max_seq_len, len(ids) + max_tokens))
        logits = self.model.prefill(torch.tensor(ids, device=device, dtype=torch.long), cache)[-1]
        step = None
        for i in range(max_tokens):
            ids.append(_pick(logits, topk))
            if ids[-1] == eos or i + 1 == max_tokens:
                break
            if step is None:
                step = GraphedStep(self.model, cache)
            logits = step(torch.tensor([ids[-1]], device=device, dtype=torch.long))[0]
        return ids

    def _generate_speculative(self, seqs: list, max_tokens: int, eos, draft, k: int, device, ragged: bool) -> list:
        """Greedy decoding of every sequence by speculative rounds of k draft tokens; ``ragged``: fill the caches
        with per-sequence lengths (a batch), else with one shared length (one prompt)."""
        speculative.check_models(self.model, draft, k)
        B, lengths = len(seqs), [len(s) for s in seqs]
        P = max(lengths)
        ids = torch.zeros(B, P, dtype=torch.long)
        for b, s in enumerate(seqs):
            ids[b, :len(s)] = torch.tensor(s, dtype=torch.long)
        ids = ids.to(device) if ragged else ids[0].to(device)
        fill = dict(lengths=lengths) if ragged else {}
        # every sequence fits: a finished one never grows, an unfinished one holds at most P + max_tokens - 1 tokens
        # after a round that started with room for k + 1 more
        need = P + max_tokens + k + 1
        cache = self.model.new_kv_cache(B, min(self.model.max_seq_len, need))
        draft_cache = draft.new_kv_cache(B, min(draft.max_seq_len, need))
        logits = self.model.prefill(ids, cache, **fill).reshape(B, P, -1)
        draft.prefill(ids, draft_cache, **fill)
        last = _pick_rows(logits[torch.arange(B, device=device), torch.tensor(lengths, device=device) - 1], 1)
        budget = []
        for b, t in enumerate(last.tolist()):
            seqs[b].append(t)
            budget.append(0 if t == eos else max_tokens - 1)
        rnd = None
        while any(budget) and cache.n + k + 1 <= cache.capacity and draft_cache.n + k + 1 <= draft_cache.capacity:
            if rnd is None:
                rnd = SpeculativeRound(self.model, cache, draft, draft_cache, k, eos=-1 if eos is None else eos)
                rnd.start(last, budget)
            for b, toks in enumerate(rnd()):
                seqs[b].extend(toks)
                budget[b] = 0 if toks and toks[-1] == eos else budget[b] - len(toks)
        if any(budget):  # near the end of the position table: the model's own steps finish the sequences
            self._finish_with_steps(seqs, budget, cache, eos, device)
        return seqs

    def _finish_with_steps(self, seqs: list, budget: list, cache, eos, device) -> None:
        """Greedy steps of the model on a cache that holds every sequence but its newest token, until every budget is
        spent. A finished sequence is cut to no rows before each step, so that it cannot outgrow the cache while the
        others finish (its outputs are dropped)."""
        step = None
        last = torch.tensor([s[-1] for s in seqs], device=device, dtype=torch.long)
        while any(budget):
            if any(n and not r for n, r in zip(cache.seq_lengths, budget)):
                cache.truncate([n if r else 0 for n, r in zip(cache.seq_lengths, budget)])
            if step is None:
                step = GraphedStep(self.model, cache)
            last = _pick_rows(step(last), 1)
            for b, t in enumerate(last.tolist()):
                if budget[b]:
                    seqs[b].append(t)
                    budget[b] = 0 if t == eos else budget[b] - 1
