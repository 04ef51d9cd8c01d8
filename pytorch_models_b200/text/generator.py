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

from ..graphs import GraphedStep


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

    @torch.inference_mode()
    def generate(self, prompt: str, max_tokens: int = 100, topk: int = 1, use_cache: bool = False) -> str:
        """``use_cache=True``: one prefill of the prompt into a KV cache, then one CUDA-graph replay of
        ``model.step`` per new token (`graphs.GraphedStep`) instead of a forward over the whole prefix. Same stopping
        rules and sampling; the logits agree with the uncached ones within bf16 rounding, so greedy decoding can take
        a different branch where the two best logits are closer than that."""
        device = next(self.model.parameters()).device
        eos = self.tokenizer.eos_token_id
        ids = list(self.tokenizer.encode(prompt))
        if use_cache and max_tokens > 0:
            return self.tokenizer.decode(self._generate_cached(ids, max_tokens, topk, eos, device))
        for _ in range(max_tokens):
            prefix = torch.tensor(ids, device=device, dtype=torch.long)
            ids.append(_pick(self.model(prefix)[-1], topk))
            if ids[-1] == eos:
                break
        return self.tokenizer.decode(ids)

    @torch.inference_mode()
    def generate_batch(self, prompts: list[str], max_tokens: int = 100, topk: int = 1) -> list[str]:
        """`generate` (``use_cache=True``) for several prompts of any lengths at once: one ragged prefill of the
        right-padded prompts (``model.prefill(..., lengths=...)``), then one CUDA-graph replay of ``model.step`` per
        token for the whole batch, with one host synchronisation per step to read the picked tokens. Each sequence
        stops at its own EOS (the batch keeps stepping; its later tokens are dropped) or after ``max_tokens`` new
        tokens. Returns one string per prompt, what ``generate(prompt, max_tokens, topk, use_cache=True)`` returns up
        to bf16 rounding (see `generate`)."""
        device = next(self.model.parameters()).device
        eos = self.tokenizer.eos_token_id
        seqs = [list(self.tokenizer.encode(p)) for p in prompts]
        if not seqs or max_tokens <= 0:
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
