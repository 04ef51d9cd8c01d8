"""CUDA-graph replay of a forward pass (launch-bound regime: small batches).

A ViT-B/16 forward is 65 kernel launches; below ~64 images the per-launch enqueue time of the Python host layer
(~1.9 ms; 0.25 ms through a launch plan, plans.py) exceeds the GPU time, and even where it does not the GPU itself
runs a captured forward faster than 65 stream launches (4.44 vs 4.75 ms at 128 images, round 2). All libb200enc entry
points are capturable (no host synchronisation, tensor maps passed by value, workspaces from
the caching allocator), so the whole forward can be captured once per input shape and replayed.
"""
from __future__ import annotations

import torch
from torch import Tensor, nn

from . import ops, plans, speculative
from .transformer import step_ids_batch


class GraphedForward:
    """``g = GraphedForward(model, example)``; ``y = g(x)`` replays the captured forward on ``x`` (same shape/dtype).

    The packed-weight caches are built during the warm-up calls, so the graph reads the kernel-ready copies; after
    changing weights call :meth:`capture` again.
    """

    def __init__(self, module: nn.Module, example: Tensor, warmup: int = 2) -> None:
        if not example.is_cuda:
            raise RuntimeError("GraphedForward needs a CUDA example input")
        self.module = module
        self.static_in = example.detach().clone()
        self.capture(warmup)

    @torch.no_grad()
    def capture(self, warmup: int = 2) -> None:
        side = torch.cuda.Stream(self.static_in.device)
        side.wait_stream(torch.cuda.current_stream())
        prev = plans.enable(False)  # the warm-up runs on a side stream: no point in recording a launch plan for it
        try:
            with torch.cuda.stream(side):
                for _ in range(max(1, warmup)):
                    self.module(self.static_in)
        finally:
            plans.enable(prev)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        n0 = ops.LAUNCHES
        with torch.cuda.graph(self.graph):
            self.static_out = self.module(self.static_in)
        self.launches = ops.LAUNCHES - n0  # libb200enc kernels inside the graph (counted on every replay)

    @torch.no_grad()
    def __call__(self, x: Tensor) -> Tensor:
        if x.shape != self.static_in.shape or x.dtype != self.static_in.dtype:
            raise ValueError(f"captured for {tuple(self.static_in.shape)} {self.static_in.dtype}, "
                             f"got {tuple(x.shape)} {x.dtype}")
        self.static_in.copy_(x, non_blocking=True)
        self.graph.replay()
        ops.LAUNCHES += self.launches
        return self.static_out.clone()


class GraphedStep:
    """``g = GraphedStep(model, cache)``; ``logits = g(ids)`` replays one captured ``model.step(ids, cache)``: the
    decode step's counterpart of `GraphedForward` for ``GPT2`` / ``GPT`` / ``WhisperDecoder``.

    A step's launches read the position from the cache's device-side length and advance it on the device, so one
    captured graph serves every position. Capture runs warm-up steps (which write the rows past the current length and
    advance it) and then restores the cache's length, so the cache is left as it was found. ``ids``: (B,) or (B, 1).

    The graph reads the length tensor the cache used at capture: the shared length, or the per-sequence lengths of a
    ragged fill (`KVCache.seq_lengths`). Replay is refused once the cache has switched to the other kind (``reset()``
    and a prefill with or without ``lengths``); capture again then.
    """

    def __init__(self, model: nn.Module, cache, warmup: int = 2) -> None:
        self.model, self.cache = model, cache
        self.static_ids = torch.zeros(cache.batch, 1, device=cache.length.device, dtype=torch.long)
        self.capture(warmup)

    @torch.no_grad()
    def capture(self, warmup: int = 2) -> None:
        cache = self.cache
        cache.check_step(cache.batch)  # the warm-up needs at least one free row
        self.length = cache.length  # the tensor the captured launches read and advance
        saved_len, saved_n = cache.length.clone(), cache.n
        side = torch.cuda.Stream(cache.length.device)
        side.wait_stream(torch.cuda.current_stream())
        try:
            with torch.cuda.stream(side):
                for _ in range(max(1, min(warmup, cache.capacity - cache.n))):
                    self.model.step(self.static_ids, cache)
            cache.n = saved_n  # the captured step's argument checks see the cache as it was found
            self.graph = torch.cuda.CUDAGraph()
            n0 = ops.LAUNCHES
            with torch.cuda.graph(self.graph):
                self.static_out = self.model.step(self.static_ids, cache)
            self.launches = ops.LAUNCHES - n0
        finally:
            torch.cuda.current_stream().wait_stream(side)
            cache.length.copy_(saved_len)
            cache.n = saved_n

    @torch.no_grad()
    def __call__(self, ids: Tensor) -> Tensor:
        self.cache.check_step(step_ids_batch(ids))
        if self.cache.length is not self.length:
            kind = "per-sequence" if self.cache.ragged else "shared"
            raise ValueError(f"the cache now holds {kind} lengths, not the kind it held when this step was captured; "
                             "capture a new GraphedStep")
        self.static_ids.copy_(ids.reshape(-1, 1), non_blocking=True)
        self.graph.replay()
        self.cache.n += 1
        ops.LAUNCHES += self.launches
        return self.static_out.clone()


class SpeculativeRound:
    """``r = SpeculativeRound(target, target_cache, draft, draft_cache, k)``; ``r.start(last, budget)``; then each
    ``tokens = r()`` replays one captured greedy speculative round (`speculative.speculative_round`) with k draft
    tokens and returns the tokens each sequence emitted, as host lists. ``draft`` may be a `speculative.NGramDraft`
    with its token history (``draft.new_kv_cache``) as ``draft_cache``.

    Both caches hold the same tokens of every sequence and ``last`` (the newest token, in neither cache) lives on the
    device between rounds, so a replay needs no input from the host; `__call__` reads the result back with one small
    device-to-host copy and updates both caches' host mirrors. Capture runs a warm-up round on a side stream and then
    restores both caches' lengths, the ids and the budget. As for `GraphedStep`, the graph reads the length tensors
    the caches used at capture; replay is refused once either cache has switched to the other kind."""

    def __init__(self, target: nn.Module, target_cache, draft: nn.Module, draft_cache, k: int = 4, eos: int = -1,
                 warmup: int = 1) -> None:
        speculative.check_round(target, target_cache, draft, draft_cache, k)
        self.target, self.target_cache, self.draft, self.draft_cache = target, target_cache, draft, draft_cache
        self.k, self.eos = k, -1 if eos is None else int(eos)
        dev = target_cache.length.device
        self.ids = torch.zeros(target_cache.batch, k + 1, device=dev, dtype=torch.long)
        self.budget = torch.zeros(target_cache.batch, device=dev, dtype=torch.int32)
        self.capture(warmup)

    def start(self, last: Tensor, budget: list[int]) -> None:
        """Each sequence's newest token ((B,) ids on the device, not yet in either cache) and how many more tokens it
        may emit (B host ints)."""
        self.ids[:, 0].copy_(last.reshape(-1))
        self.budget.copy_(torch.tensor(budget, dtype=torch.int32))

    def _round(self) -> Tensor:
        return speculative.speculative_round(self.target, self.target_cache, self.draft, self.draft_cache, self.ids,
                                             self.budget, self.eos)

    @torch.no_grad()
    def capture(self, warmup: int = 1) -> None:
        caches = (self.target_cache, self.draft_cache)
        speculative.check_room(*caches, self.k)
        self.lengths = tuple(c.length for c in caches)  # the tensors the captured launches read and update
        saved = [(c.length.clone(), c.n) for c in caches]
        saved_ids, saved_budget = self.ids.clone(), self.budget.clone()
        side = torch.cuda.Stream(self.ids.device)
        side.wait_stream(torch.cuda.current_stream())
        try:
            with torch.cuda.stream(side):
                for _ in range(max(1, warmup)):
                    self._round()
                    for c, (length, _) in zip(caches, saved):
                        c.length.copy_(length)
            self.graph = torch.cuda.CUDAGraph()
            n0 = ops.LAUNCHES
            with torch.cuda.graph(self.graph):
                self.result = self._round()
            self.launches = ops.LAUNCHES - n0
        finally:
            torch.cuda.current_stream().wait_stream(side)
            for c, (length, n) in zip(caches, saved):
                c.length.copy_(length)
                c.n = n
            self.ids.copy_(saved_ids)
            self.budget.copy_(saved_budget)

    @torch.no_grad()
    def __call__(self) -> list[list[int]]:
        for name, cache, length in (("target", self.target_cache, self.lengths[0]),
                                    ("draft", self.draft_cache, self.lengths[1])):
            if cache.length is not length:
                kind = "per-sequence" if cache.ragged else "shared"
                raise ValueError(f"the {name} cache now holds {kind} lengths, not the kind it held when this round was "
                                 "captured; capture a new SpeculativeRound")
        speculative.check_room(self.target_cache, self.draft_cache, self.k)
        self.graph.replay()
        ops.LAUNCHES += self.launches
        return speculative.finish_round(self.target_cache, self.draft_cache, self.result)
