"""Greedy speculative decoding for ``GPT2`` / ``GPT`` / ``WhisperDecoder`` pairs that share a vocabulary, or for any of
them alone with draft-free proposals (`NGramDraft`).

A round with k draft tokens keeps one invariant: before and after it, the target's and the draft's KV caches hold the
same tokens of each sequence, and ``last``, the newest emitted token, is in neither. The round

1. runs k + 1 decode steps of the draft, fed ``last``, d_1, .., d_k, where d_{j+1} is the argmax of step j's logits
   (the last step only writes d_k's k|v row, so its logits are not computed);
2. verifies with one target extend of [last, d_1 .. d_k], whose lengths advance on the device;
3. picks the target's argmax t_0 .. t_k of each verify row;
4. accepts d_1 .. d_a, t_a per sequence (a = the number of leading drafts equal to the target's picks), cut at EOS and
   at the sequence's token budget, and rolls both caches back past the rows it did not keep.

Every kept token is the target's argmax at its prefix, so the output is the target's greedy output (up to near-ties of
two logits, which a verify row computed by `extend` can order differently than a `step` does). No step needs the host,
so `graphs.SpeculativeRound` replays a whole round as one CUDA graph.

With an `NGramDraft` in place of the draft model, step 1 is one kernel: the drafts are the tokens that followed the
latest earlier occurrence of the sequence's last n-gram in its own prompt and output, read from a `TokenHistory` that
plays the draft cache's part (it holds the same tokens as the target's cache, and ``last`` is in neither).
"""
from __future__ import annotations

import torch
from torch import Tensor

from . import ops
from .transformer import CacheLengths, KVCache, embed_tokens_at

MAX_DRAFT_TOKENS = 15
MAX_NGRAM = 8  # the longest n-gram b200enc_ngram_draft matches


class TokenHistory(CacheLengths):
    """The token ids each sequence holds, in place of a draft model's KV cache: ``tokens`` (batch, capacity) int64,
    row b's first ``seq_lengths[b]`` entries valid, with the length bookkeeping of `KVCache`."""

    def __init__(self, batch: int, capacity: int, device: torch.device) -> None:
        super().__init__(batch, capacity, device)
        self.tokens = torch.zeros(batch, capacity, device=device, dtype=torch.int64)


class NGramDraft:
    """Draft-free proposals for a speculative round: the drafts of a sequence are the tokens that followed the latest
    earlier occurrence of its longest final n-gram (``max_ngram`` down to ``min_ngram`` tokens, of the prompt and the
    output so far), or its newest token repeated when none occurs (`ops.ngram_draft`). No weights, so it serves every
    decoder; the generator and `graphs.SpeculativeRound` take it where they take a draft model."""

    max_seq_len = 2 ** 31 - 1  # no position table: the history is as long as the target's cache needs

    def __init__(self, max_ngram: int = 3, min_ngram: int = 1) -> None:
        if not 1 <= min_ngram <= max_ngram <= MAX_NGRAM:
            raise ValueError(f"min_ngram={min_ngram} and max_ngram={max_ngram} must satisfy "
                             f"1 <= min_ngram <= max_ngram <= {MAX_NGRAM}")
        self.max_ngram, self.min_ngram = max_ngram, min_ngram

    def new_kv_cache(self, batch: int, capacity: int, device=None) -> TokenHistory:
        """An empty token history for ``batch`` sequences of up to ``capacity`` tokens, on ``device`` (default: the
        current CUDA device)."""
        if batch < 1 or capacity < 1:
            raise ValueError(f"batch={batch} and capacity={capacity} must be >= 1")
        return TokenHistory(batch, capacity, torch.device("cuda") if device is None else torch.device(device))

    def prefill(self, ids: Tensor, history: TokenHistory, lengths=None) -> None:
        """Copy the prompts, (B, P) or (P,) ids, into an empty ``history``; ``lengths`` as in ``GPT2.prefill``
        (B host ints in [1, P] for right-padded prompts)."""
        P = ids.shape[-1]
        ids = ids.reshape(-1, P)
        history.check_prefill(ids.shape[0], P)
        lengths = history.check_lengths(lengths, P)
        history.tokens[:, :P].copy_(ids)
        history.set_lengths(P, lengths)

    def propose(self, history: TokenHistory, ids: Tensor) -> None:
        """Step 1 of a round: the drafts into ``ids[:, 1:]`` and [last, drafts] into the history, on the device."""
        ops.ngram_draft(history.tokens, history.length, ids, ids.shape[1] - 1, self.max_ngram, self.min_ngram)


def check_models(target, draft, k: int) -> None:
    """Refuse a pair of models or a draft length that a round cannot run, before anything is enqueued."""
    if not 1 <= k <= MAX_DRAFT_TOKENS:
        raise ValueError(f"k={k} draft tokens per round; a round takes 1 to {MAX_DRAFT_TOKENS}")
    if isinstance(draft, NGramDraft):  # no vocabulary of its own: it proposes the sequence's own tokens
        target.layers._check_decodable()
        return
    vt, vd = target.token_embs.weight.shape[0], draft.token_embs.weight.shape[0]
    if vt != vd:
        raise ValueError(f"the draft's vocabulary of {vd} tokens differs from the target's {vt}")
    target.layers._check_decodable()
    draft.layers._check_decodable()


def check_room(target_cache: KVCache, draft_cache: CacheLengths, k: int) -> None:
    """Both caches need k + 1 free rows past their longest sequence (the rows a round writes before it rolls back)."""
    for name, cache in (("target", target_cache), ("draft", draft_cache)):
        if cache.n + k + 1 > cache.capacity:
            raise ValueError(f"a round of k={k} draft tokens writes {k + 1} rows past the {cache.n} tokens the {name} "
                             f"cache holds, more than its capacity of {cache.capacity}")


def check_round(target, target_cache: KVCache, draft, draft_cache: CacheLengths, k: int) -> None:
    check_models(target, draft, k)
    if isinstance(draft, NGramDraft) != isinstance(draft_cache, TokenHistory):
        raise ValueError("an NGramDraft drafts from a TokenHistory (NGramDraft.new_kv_cache), a draft model from its "
                         f"own KV cache; got {type(draft).__name__} with a {type(draft_cache).__name__}")
    if target_cache.batch != draft_cache.batch:
        raise ValueError(f"the target cache holds {target_cache.batch} sequences, the draft cache "
                         f"{draft_cache.batch}")
    for name, cache in (("target", target_cache), ("draft", draft_cache)):
        if cache.batch > 1 and not cache.ragged:
            raise ValueError(f"the {name} cache holds one shared length for a batch of {cache.batch}; a round rolls "
                             "each sequence back by its own count and needs per-sequence lengths: fill it with "
                             "prefill(..., lengths=...)")
    check_room(target_cache, draft_cache, k)


def speculative_round(target, target_cache: KVCache, draft, draft_cache: CacheLengths, ids: Tensor,
                      budget: Tensor, eos: int = -1) -> Tensor:
    """Enqueue one round (steps 1-4 of the module docstring) without a host synchronisation.

    ``ids``: (B, k+1) int64 device buffer whose column 0 holds each sequence's ``last``; the round writes the drafts
    into columns 1..k and the next round's ``last`` into column 0. ``budget``: (B,) int32 device tokens each sequence
    may still emit, decremented here. ``eos``: token id that ends a sequence, -1 for none.

    Returns a (B, k+2) int64 device tensor: the tokens emitted by sequence b in ``[b, :m_b]`` (-1 after them) and m_b
    in ``[b, k+1]``. The device lengths of both caches end at the kept rows; their host mirrors are left as they were
    found, and `finish_round` brings them up to date from m_b."""
    B, P = ids.shape
    k = P - 1
    check_round(target, target_cache, draft, draft_cache, k)
    if B != target_cache.batch:
        raise ValueError(f"ids hold {B} sequences, the caches {target_cache.batch}")
    saved_n = target_cache.n, draft_cache.n
    if isinstance(draft, NGramDraft):
        draft.propose(draft_cache, ids)
    else:
        for j in range(P):
            x = embed_tokens_at(ids[:, j], draft.token_embs, draft.pos_embs, draft_cache)
            h, stats = draft.layers.step(x, draft_cache)
            if j < k:
                ops.argmax_rows(draft.logits_bf16(h, stats)[:, 0], ids[:, j + 1])
    x = embed_tokens_at(ids, target.token_embs, target.pos_embs, target_cache)
    h, stats = target.layers.extend_launches(x, target_cache)
    ops.decode_advance(target_cache.length, P)  # on the device: a host-valued length would be baked into a graph
    logits = target.logits_bf16(h, stats)
    picks = torch.empty(B, P, device=ids.device, dtype=torch.int64)
    ops.argmax_rows(logits.reshape(B * P, logits.shape[-1]), picks.view(-1))
    result = torch.empty(B, P + 1, device=ids.device, dtype=torch.int64)
    ops.speculative_accept(picks, ids, budget, eos, target_cache.length, draft_cache.length, result[:, :P],
                           result[:, P])
    target_cache.n, draft_cache.n = saved_n
    return result


def finish_round(target_cache: KVCache, draft_cache: CacheLengths, result: Tensor) -> list[list[int]]:
    """Read a round's result back (one device-to-host copy, the round's one host synchronisation), move both caches'
    host mirrors to the kept rows and return the tokens each sequence emitted."""
    res = result.cpu()
    k = res.shape[1] - 2
    counts = res[:, k + 1].tolist()
    for cache in (target_cache, draft_cache):
        cache.store_lengths([n + m for n, m in zip(cache.seq_lengths, counts)], device=False)
    return [row[:m] for row, m in zip(res[:, :k + 1].tolist(), counts)]
