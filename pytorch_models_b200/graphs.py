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

from . import ops, plans
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
