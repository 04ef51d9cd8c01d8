"""Thin Python wrappers over the C-ABI: one function per libb200enc entry point.

All tensors must be CUDA bf16 (fp32 for vectors / statistics); the wrappers only validate, fetch raw pointers and the
current stream, and call into the library. No arithmetic happens in PyTorch here.
"""
from __future__ import annotations

import ctypes
import threading

import torch
from torch import Tensor

from . import _lib


LAUNCHES = 0  # kernels launched through the C-ABI by this process (every entry point launches exactly one)
_PROFILE: list | None = None  # when a list: (entry point, meta, start event, end event) per launch
_RECORD = None  # plans._Recorder while a forward is being recorded into a launch plan (plans.py), else None


def profile(enable: bool) -> list | None:
    """Start (returns the record list) or stop per-launch CUDA-event timing on the launching stream."""
    global _PROFILE
    _PROFILE = [] if enable else None
    return _PROFILE


def _call(name: str, meta: dict | None, dev: torch.device, *args) -> None:
    """Enqueue one entry point on ``dev``'s current stream (appended as the last argument). The library launches on
    the CUDA runtime's current device, so a tensor that lives on another GPU than the current one (``model.to("cuda:1")``
    without ``torch.cuda.set_device``) switches the device for the duration of the call."""
    global LAUNCHES
    if dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):
            return _call(name, meta, dev, *args)
    fn = getattr(_lib.load(), name)
    stream = torch.cuda.current_stream(dev)
    plan_rec = _RECORD
    if plan_rec is not None and plan_rec.thread == threading.get_ident():
        if name in _lib.OP_KINDS:
            plan_rec.calls.append((name, args))
        else:
            plan_rec.ok = False  # an entry point b200enc_run_ops cannot replay: this forward stays on the per-call path
    rec = _PROFILE
    if rec is None:
        rc = fn(*args, stream.cuda_stream)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        rc = fn(*args, stream.cuda_stream)
        e1.record(stream)
        rec.append((name, meta, e0, e1))
    LAUNCHES += 1
    _lib.check(rc, name)


def _ptr(t: Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts: Tensor | None) -> torch.device:
    """All tensors must live on one CUDA device; returns it."""
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "pytorch_models_b200 runs only on CUDA (sm_100a) tensors; there is no CPU fallback "
                f"(got a {t.device} tensor)"
            )
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"tensors of one kernel call live on different devices ({dev} and {t.device})")
    if dev is None:
        raise RuntimeError("no tensor arguments")
    if _RECORD is not None:  # a launch plan keeps every tensor its launches touch alive (plans.py)
        _RECORD.keep.extend(t for t in ts if t is not None)
    return dev


def _need(t: Tensor | None, dtype: torch.dtype, name: str) -> None:
    if t is not None and t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")


def linear(
    x: Tensor,
    w: Tensor,
    bias: Tensor | None,
    out: Tensor,
    *,
    colsum: Tensor | None = None,
    rowstats: Tensor | None = None,
    residual: Tensor | None = None,
    gelu: bool | str = False,
    ln_eps: float = 0.0,
    stats_out: Tensor | None = None,
    stats_rows: int = 0,
    stats_row_offset: int = 0,
) -> Tensor:
    """out[b, m, :] = epilogue(x[b, m, :] @ w.T); x, out, residual are (batches, M, *) views with unit inner stride.

    ``gelu`` selects the activation: False, True (exact erf GELU), "tanh" (``nn.GELU(approximate="tanh")``), "relu" or
    "silu" (the last three not together with a residual).
    A residual with a leading dimension of 1 is broadcast over the batch (positional embedding).
    ``rowstats`` is either (batches*M, 2) = (mean, rstd) from `row_stats`, or (batches*M, parts, 2) partial
    (mean, M2) per 128 input columns as written through ``stats_out`` by the linear that produced ``x``
    (then ``ln_eps`` is required). ``stats_out``: (batches*M, ceil(N/128), 2) fp32, needs a residual epilogue; with
    ``stats_rows`` > 0 it is (batches*stats_rows, ceil(N/128), 2) and row (b, m) goes to b*stats_rows + stats_row_offset + m.
    """
    dev = _need_cuda(x, w, bias, out, colsum, rowstats, residual, stats_out)
    _need(x, torch.bfloat16, "x"), _need(w, torch.bfloat16, "w"), _need(out, torch.bfloat16, "out")
    _need(bias, torch.float32, "bias"), _need(colsum, torch.float32, "colsum"), _need(rowstats, torch.float32, "rowstats")
    _need(residual, torch.bfloat16, "residual"), _need(stats_out, torch.float32, "stats_out")
    if x.dim() == 2:
        x, out = x.unsqueeze(0), out.unsqueeze(0)
        residual = None if residual is None else residual.unsqueeze(0)
    batches, M, K = x.shape
    N = w.shape[0]
    if w.shape[1] != K or out.shape != (batches, M, N):
        raise ValueError(f"shape mismatch: x {tuple(x.shape)}, w {tuple(w.shape)}, out {tuple(out.shape)}")
    if x.stride(2) != 1 or w.stride(1) != 1 or out.stride(2) != 1:
        raise ValueError("inner strides must be 1")
    res_bs, ldr = 0, 0
    if residual is not None:
        if residual.shape[-2:] != (M, N) or residual.stride(2) != 1:
            raise ValueError(f"residual shape {tuple(residual.shape)} does not match ({M}, {N})")
        res_bs = 0 if residual.shape[0] == 1 else residual.stride(0)
        ldr = residual.stride(1)
    parts = 0
    if rowstats is not None:
        if not rowstats.is_contiguous() or rowstats.numel() % (2 * batches * M) != 0:
            raise ValueError("rowstats must be a contiguous (batches*M, 2) or (batches*M, parts, 2) tensor")
        parts = 0 if rowstats.dim() == 2 else rowstats.shape[1]
    srows = stats_rows if stats_rows > 0 else M
    if stats_out is not None and (not stats_out.is_contiguous() or srows < M + stats_row_offset or stats_row_offset < 0
                                  or stats_out.numel() != 2 * batches * srows * ((N + 127) // 128)):
        raise ValueError("stats_out must be a contiguous (batches*rows, ceil(N/128), 2) tensor that holds every row")
    acts = {False: 0, True: _lib.LINEAR_GELU, "tanh": _lib.LINEAR_GELU_TANH, "relu": _lib.LINEAR_RELU,
            "silu": _lib.LINEAR_SILU}
    if isinstance(gelu, (bool, str)) and gelu in acts:
        act = acts[gelu]
    else:
        raise ValueError(f"gelu must be False, True, 'tanh', 'relu' or 'silu', got {gelu!r}")
    args = _lib.LinearArgs(
        x.data_ptr(), x.stride(0), x.stride(1), w.data_ptr(), w.stride(0), _ptr(bias), _ptr(colsum),
        _ptr(rowstats), parts, float(ln_eps), _ptr(residual), res_bs, ldr, out.data_ptr(), out.stride(0), out.stride(1),
        _ptr(stats_out), batches, M, N, K, act, int(stats_rows), int(stats_row_offset), None,
    )
    _call(
        "b200enc_linear", dict(batches=batches, M=M, N=N, K=K, fold=colsum is not None, gelu=gelu, res=residual is not None),
        dev, ctypes.byref(args),
    )
    return out


def linear_fp8(x8: Tensor, w8: Tensor, acc_scale: Tensor, bias: Tensor | None, out: Tensor, *, gelu: bool = False,
               residual: Tensor | None = None) -> Tensor:
    """OPTIONAL FP8 variant (never used unless asked for): out = epi(acc_scale * (x8 @ w8.T) + bias) with e4m3 operands.

    x8: (M, K) or (batches, M, K) ``torch.float8_e4m3fn``, w8: (N, K) e4m3, acc_scale: 1-element fp32 CUDA tensor holding
    the product of the two per-tensor dequantisation scales, bias fp32 (N) or None, out bf16. Epilogues: bias,
    bias + erf-GELU, bias + residual. K must be a multiple of 16."""
    dev = _need_cuda(x8, w8, acc_scale, bias, out, residual)
    _need(x8, torch.float8_e4m3fn, "x8"), _need(w8, torch.float8_e4m3fn, "w8"), _need(out, torch.bfloat16, "out")
    _need(acc_scale, torch.float32, "acc_scale"), _need(bias, torch.float32, "bias"), _need(residual, torch.bfloat16, "residual")
    ret = out
    if x8.dim() == 2:
        x8, out = x8.unsqueeze(0), out.unsqueeze(0)
        residual = None if residual is None else residual.unsqueeze(0)
    batches, M, K = x8.shape
    N = w8.shape[0]
    if w8.shape[1] != K or out.shape != (batches, M, N) or acc_scale.numel() != 1:
        raise ValueError(f"shape mismatch: x8 {tuple(x8.shape)}, w8 {tuple(w8.shape)}, out {tuple(out.shape)}")
    if x8.stride(2) != 1 or w8.stride(1) != 1 or out.stride(2) != 1:
        raise ValueError("inner strides must be 1")
    res_bs, ldr = 0, 0
    if residual is not None:
        if residual.shape[-2:] != (M, N) or residual.stride(2) != 1:
            raise ValueError(f"residual shape {tuple(residual.shape)} does not match ({M}, {N})")
        res_bs = 0 if residual.shape[0] == 1 else residual.stride(0)
        ldr = residual.stride(1)
    flags = _lib.LINEAR_FP8 | (_lib.LINEAR_GELU if gelu else 0)
    args = _lib.LinearArgs(
        x8.data_ptr(), x8.stride(0), x8.stride(1), w8.data_ptr(), w8.stride(0), _ptr(bias), None, None, 0, 0.0,
        _ptr(residual), res_bs, ldr, out.data_ptr(), out.stride(0), out.stride(1), None, batches, M, N, K, flags, 0, 0,
        acc_scale.data_ptr(),
    )
    _call("b200enc_linear", dict(batches=batches, M=M, N=N, K=K, fold=False, gelu=gelu, res=residual is not None, fp8=True),
          dev, ctypes.byref(args))
    return ret


def attention(q: Tensor, k: Tensor, v: Tensor, out: Tensor, n_heads: int, scale: float, causal: bool = False,
              bias: Tensor | None = None, streaming: bool = False) -> Tensor:
    """q: (B, Lq, H*hd) view, k/v: (B, Lkv, H*hd) views sharing strides, out: (B, Lq, H*hd), with head_dim
    hd = D // n_heads in {64, 80, 96, 112, 128}.

    ``causal``: query i sees keys 0..i (top-left aligned like ``F.scaled_dot_product_attention(is_causal=True)``).
    ``bias``: fp32 (B, H, Lq, Lkv) view added to the scaled scores (``attn_mask`` of SDPA); broadcast dimensions may
    have stride 0 (``Tensor.expand``), the last stride must be 1.
    head_dim 64: unmasked calls with Lkv <= 256 run the single-pass kernel (csrc/attention_short.cuh); ``streaming=True``
    forces the online-softmax kernel there too (the reference the tests check the single-pass kernel against). Wider
    heads run csrc/attention_wide.cuh for every shape, mask and bias (``streaming`` has nothing to select there)."""
    dev = _need_cuda(q, k, v, out, bias)
    for name, t in (("q", q), ("k", k), ("v", v), ("out", out)):
        _need(t, torch.bfloat16, name)
        if t.dim() != 3 or t.stride(2) != 1:
            raise ValueError(f"{name} must be a (B, L, H*head_dim) view with unit inner stride")
    B, Lq, D = q.shape
    Lkv = k.shape[1]
    if D % n_heads != 0:
        raise ValueError("width not divisible by n_heads")
    if k.shape != v.shape or k.stride() != v.stride() or k.shape[0] != B or k.shape[2] != D or out.shape != q.shape:
        raise ValueError("q/k/v/out shapes or strides are inconsistent")
    if bias is not None:
        _need(bias, torch.float32, "bias")
        if bias.shape != (B, n_heads, Lq, Lkv) or (Lkv > 1 and bias.stride(3) != 1) or min(bias.stride()) < 0:
            raise ValueError(f"bias must be a (B, H, Lq, Lkv) = {(B, n_heads, Lq, Lkv)} view with unit inner stride")
        _call(
            "b200enc_attention_bias", dict(B=B, H=n_heads, Lq=Lq, Lkv=Lkv, causal=bool(causal), bias=True), dev,
            q.data_ptr(), q.stride(0), q.stride(1), k.data_ptr(), v.data_ptr(), k.stride(0), k.stride(1),
            out.data_ptr(), out.stride(0), out.stride(1), B, n_heads, Lq, Lkv, D // n_heads, float(scale),
            _lib.ATTN_CAUSAL if causal else 0, bias.data_ptr(), bias.stride(0), bias.stride(1), bias.stride(2),
        )
        return out
    _call(
        "b200enc_attention", dict(B=B, H=n_heads, Lq=Lq, Lkv=Lkv, causal=bool(causal)), dev,
        q.data_ptr(), q.stride(0), q.stride(1), k.data_ptr(), v.data_ptr(), k.stride(0), k.stride(1), out.data_ptr(),
        out.stride(0), out.stride(1), B, n_heads, Lq, Lkv, D // n_heads, float(scale),
        (_lib.ATTN_CAUSAL if causal else 0) | (_lib.ATTN_GENERAL if streaming else 0),
    )
    return out


def layernorm(x: Tensor, gamma: Tensor, beta: Tensor, eps: float, out: Tensor, stats: Tensor | None = None) -> Tensor:
    """x: (rows, d) view (any row stride), out: (rows, d)."""
    dev = _need_cuda(x, gamma, beta, out, stats)
    _need(x, torch.bfloat16, "x"), _need(out, torch.bfloat16, "out")
    _need(gamma, torch.float32, "gamma"), _need(beta, torch.float32, "beta"), _need(stats, torch.float32, "stats")
    rows, d = x.shape
    if x.stride(1) != 1 or out.stride(1) != 1 or out.shape != x.shape:
        raise ValueError("layernorm expects (rows, d) views with unit inner stride")
    _call(
        "b200enc_layernorm", dict(rows=rows, d=d), dev,
        x.data_ptr(), x.stride(0), gamma.data_ptr(), beta.data_ptr(), float(eps), rows, d, out.data_ptr(),
        out.stride(0), _ptr(stats),
    )
    return out


def row_stats(x: Tensor, eps: float, stats: Tensor) -> Tensor:
    dev = _need_cuda(x, stats)
    _need(x, torch.bfloat16, "x"), _need(stats, torch.float32, "stats")
    rows, d = x.shape
    if x.stride(1) != 1 or stats.numel() != 2 * rows or not stats.is_contiguous():
        raise ValueError("row_stats expects a (rows, d) view and a contiguous (rows, 2) stats tensor")
    _call(
        "b200enc_row_stats", dict(rows=rows, d=d), dev,
        x.data_ptr(), x.stride(0), float(eps), rows, d, stats.data_ptr(),
    )
    return stats


def mean_tokens(x: Tensor, out: Tensor) -> Tensor:
    dev = _need_cuda(x, out)
    _need(x, torch.bfloat16, "x"), _need(out, torch.bfloat16, "out")
    B, L, d = x.shape
    if x.stride(2) != 1 or out.shape != (B, d) or out.stride(1) != 1:
        raise ValueError("mean_tokens expects x (B, L, d) and out (B, d)")
    _call(
        "b200enc_mean_tokens", dict(B=B, L=L, d=d), dev,
        x.data_ptr(), x.stride(0), x.stride(1), B, L, d, out.data_ptr(), out.stride(0),
    )
    return out


def patch_embed16(imgs: Tensor, w: Tensor, bias: Tensor, pe: Tensor, tokens: Tensor, *, stats_out: Tensor | None = None,
                  stats_rows: int = 0, stats_row_offset: int = 0) -> Tensor:
    """tokens[b, patch, :] = conv16x16(imgs[b])[patch] + bias + pe[patch]: the patch embedding of a 16-pixel-patch ViT
    (``nn.Conv2d(3, d, 16, 16)`` + flatten/transpose + ``pe``, image/vit.py:64,78-79) as ONE GEMM that reads the NCHW
    bf16 image through a 5-D tensor map — no im2col buffer (other patch sizes / fp32 images: `patch_rows` + `linear`).

    imgs: (N, 3, H, W) bf16 contiguous, H and W multiples of 16; w: (d, 768) bf16 = ``conv.weight.view(d, -1)``;
    bias: (d,) fp32; pe: (P, d) bf16 with P = (H/16)*(W/16); tokens: (N, P, d) bf16 view (row stride >= d, e.g.
    ``buf[:, 1:, :]`` behind a class token). ``stats_out`` as in `linear`."""
    dev = _need_cuda(imgs, w, bias, pe, tokens, stats_out)
    _need(imgs, torch.bfloat16, "imgs"), _need(w, torch.bfloat16, "w"), _need(pe, torch.bfloat16, "pe")
    _need(tokens, torch.bfloat16, "tokens"), _need(bias, torch.float32, "bias"), _need(stats_out, torch.float32, "stats_out")
    if imgs.dim() != 4 or imgs.shape[1] != 3 or not imgs.is_contiguous():
        raise ValueError("images must be a contiguous (N, 3, H, W) tensor")
    N, _, H, W = imgs.shape
    if H % 16 or W % 16:
        raise ValueError(f"image {H}x{W} is not a multiple of the 16-pixel patch")
    P, d = (H // 16) * (W // 16), w.shape[0]
    if w.shape != (d, 768) or w.stride(1) != 1 or bias.shape != (d,) or pe.shape != (P, d) or pe.stride(1) != 1:
        raise ValueError(f"shape mismatch: w {tuple(w.shape)}, bias {tuple(bias.shape)}, pe {tuple(pe.shape)} for {P} patches")
    if tokens.shape != (N, P, d) or tokens.stride(2) != 1:
        raise ValueError(f"tokens must be a ({N}, {P}, {d}) view with unit inner stride, got {tuple(tokens.shape)}")
    srows = stats_rows if stats_rows > 0 else P
    if stats_out is not None and (not stats_out.is_contiguous() or srows < P + stats_row_offset or stats_row_offset < 0
                                  or stats_out.numel() != 2 * N * srows * ((d + 127) // 128)):
        raise ValueError("stats_out must be a contiguous (N*rows, ceil(d/128), 2) tensor that holds every row")
    args = _lib.LinearArgs(
        imgs.data_ptr(), 0, 0, w.data_ptr(), w.stride(0), _ptr(bias), None, None, 0, 0.0, pe.data_ptr(), 0, pe.stride(0),
        tokens.data_ptr(), tokens.stride(0), tokens.stride(1), _ptr(stats_out), N, P, d, 768, 0, int(stats_rows),
        int(stats_row_offset), None,
    )
    _call("b200enc_patch_embed16", dict(B=N, H=H, W=W, N=d), dev, ctypes.byref(args), H, W)
    return tokens


def patch_rows(imgs: Tensor, patch: int, kpad: int, rows: Tensor) -> Tensor:
    dev = _need_cuda(imgs, rows)
    if imgs.dtype == torch.bfloat16:
        dt = _lib.DTYPE_BF16
    elif imgs.dtype == torch.float32:
        dt = _lib.DTYPE_F32
    else:
        raise TypeError(f"images must be bfloat16 or float32, got {imgs.dtype}")
    if imgs.dim() != 4 or imgs.shape[1] != 3 or not imgs.is_contiguous():
        raise ValueError("images must be a contiguous (N, 3, H, W) tensor")
    _need(rows, torch.bfloat16, "rows")
    B, _, H, W = imgs.shape
    _call(
        "b200enc_patch_rows", dict(B=B, H=H, W=W, p=patch, kpad=kpad, f32=imgs.dtype == torch.float32), dev,
        imgs.data_ptr(), dt, B, H, W, patch, kpad, rows.data_ptr(),
    )
    return rows


def cls_rows(cls: Tensor, tokens: Tensor) -> Tensor:
    dev = _need_cuda(cls, tokens)
    _need(cls, torch.bfloat16, "cls"), _need(tokens, torch.bfloat16, "tokens")
    B, _, d = tokens.shape
    _call(
        "b200enc_cls_rows", dict(B=B, d=d), dev,
        cls.data_ptr(), B, d, tokens.data_ptr(), tokens.stride(0),
    )
    return tokens


def broadcast_row(row: Tensor, dst: Tensor) -> Tensor:
    """dst[b, 0, ...] = row for every b: dst (B, rows, *) fp32 / bf16 contiguous, row = one (*)-shaped slice. The same
    kernel as `cls_rows` (a strided broadcast of raw 16-bit units), used for the class token's LayerNorm statistics."""
    dev = _need_cuda(row, dst)
    if row.dtype != dst.dtype or not (row.is_contiguous() and dst.is_contiguous()) or dst[0, 0].numel() != row.numel():
        raise ValueError("broadcast_row expects a contiguous row that matches dst[b, 0]")
    units = row.element_size() // 2
    _call(
        "b200enc_cls_rows", dict(B=dst.shape[0], d=row.numel() * units), dev,
        row.data_ptr(), dst.shape[0], row.numel() * units, dst.data_ptr(), dst.stride(0) * units,
    )
    return dst


def time_rows(x: Tensor, rows: Tensor) -> Tensor:
    """x: (N, C, T) fp32/bf16 -> rows (N, T + 2, C) bf16 with zero first/last rows (conv padding)."""
    dev = _need_cuda(x, rows)
    if x.dtype == torch.bfloat16:
        dt = _lib.DTYPE_BF16
    elif x.dtype == torch.float32:
        dt = _lib.DTYPE_F32
    else:
        raise TypeError(f"input must be bfloat16 or float32, got {x.dtype}")
    if x.dim() != 3 or not x.is_contiguous() or not rows.is_contiguous():
        raise ValueError("time_rows expects contiguous (N, C, T) input and (N, T+2, C) output")
    N, C, T = x.shape
    if rows.shape != (N, T + 2, C):
        raise ValueError(f"rows must have shape {(N, T + 2, C)}")
    _need(rows, torch.bfloat16, "rows")
    _call(
        "b200enc_time_rows", dict(N=N, C=C, T=T), dev,
        x.data_ptr(), dt, N, C, T, rows.data_ptr(),
    )
    return rows


def _embed_args(name: str, ids: Tensor, tok: Tensor, pos: Tensor, out: Tensor) -> int:
    """Argument checks shared by `embed_rows` and `embed_rows_at`; returns the library's dtype code of the tables."""
    _need(ids, torch.int64, "ids"), _need(out, torch.bfloat16, "out")
    if tok.dtype != pos.dtype:
        raise TypeError(f"token and position tables must share a dtype, got {tok.dtype} and {pos.dtype}")
    dt = {torch.bfloat16: _lib.DTYPE_BF16, torch.float32: _lib.DTYPE_F32}.get(tok.dtype)
    if dt is None:
        raise TypeError(f"embedding tables must be bfloat16 or float32, got {tok.dtype}")
    if ids.dim() != 2 or not (ids.is_contiguous() and tok.is_contiguous() and pos.is_contiguous() and out.is_contiguous()):
        raise ValueError(f"{name} expects contiguous (B, L) ids, (vocab, d) / (P, d) tables and (B, L, d) output")
    if pos.shape[1] != tok.shape[1] or out.shape != (*ids.shape, tok.shape[1]):
        raise ValueError(f"shape mismatch: ids {tuple(ids.shape)}, tok {tuple(tok.shape)}, pos {tuple(pos.shape)}")
    return dt


def embed_rows(ids: Tensor, tok: Tensor, pos: Tensor, out: Tensor) -> Tensor:
    """ids: (B, L) int64, tok: (vocab, d), pos: (>= L, d) [both fp32 or both bf16] -> out (B, L, d) bf16 =
    tok[ids] + pos[:L]. Rows whose id is out of range come back as NaN (device code cannot raise)."""
    dev = _need_cuda(ids, tok, pos, out)
    dt = _embed_args("embed_rows", ids, tok, pos, out)
    B, L = ids.shape
    vocab, d = tok.shape
    if pos.shape[0] < L:
        raise ValueError(f"the position table has {pos.shape[0]} rows, fewer than the {L} ids of a row")
    if B * L == 0:
        return out
    _call(
        "b200enc_embed_rows", dict(rows=B * L, d=d), dev,
        ids.data_ptr(), B * L, L, tok.data_ptr(), pos.data_ptr(), dt, vocab, d, out.data_ptr(),
    )
    return out


def whisper_logmel(audio: Tensor, filters_t: Tensor, out: Tensor) -> Tensor:
    """audio: (N, L) fp32, filters_t: (201, n_mels) fp32 (mel filter bank transposed) -> out (N, n_mels, L // 160) fp32:
    the normalised log-mel spectrogram of ``WhisperPreprocessor`` (whisper.py:143-148)."""
    dev = _need_cuda(audio, filters_t, out)
    _need(audio, torch.float32, "audio"), _need(filters_t, torch.float32, "filters_t"), _need(out, torch.float32, "out")
    if audio.dim() != 2 or audio.stride(1) != 1 or not filters_t.is_contiguous() or not out.is_contiguous():
        raise ValueError("whisper_logmel expects (N, L) audio with unit inner stride and contiguous filters / output")
    N, L = audio.shape
    n_mels = filters_t.shape[1]
    if filters_t.shape[0] != 201 or out.shape != (N, n_mels, L // 160):
        raise ValueError(f"shape mismatch: filters_t {tuple(filters_t.shape)}, out {tuple(out.shape)}, L={L}")
    if N == 0:
        return out
    scratch = torch.empty(N, device=audio.device, dtype=torch.int32)
    _call(
        "b200enc_whisper_logmel", dict(N=N, L=L, n_mels=n_mels), dev,
        audio.data_ptr(), audio.stride(0), N, L, filters_t.data_ptr(), n_mels, out.data_ptr(), scratch.data_ptr(),
    )
    return out


def _per_sequence(length: Tensor | None, B: int, name: str) -> bool:
    """True if a device length tensor holds one length per sequence (B > 1 elements), False if it holds one shared
    length; anything else is refused."""
    if length is None or length.numel() == 1:
        return False
    if length.dim() != 1 or length.numel() != B or not length.is_contiguous():
        raise ValueError(f"{name} must be a contiguous int32 tensor of 1 or {B} elements, got {tuple(length.shape)}")
    return True


def decode_workspace_bytes(B: int, n_heads: int, head_dim: int, keys: int) -> int:
    """Bytes of fp32 workspace `attention_decode` needs (keys = cache capacity, or Lkv in cross mode)."""
    return int(_lib.load().b200enc_attention_decode_workspace_bytes(B, n_heads, head_dim, keys))


def attention_decode(q: Tensor, k_cache: Tensor, v_cache: Tensor, out: Tensor, n_heads: int, scale: float,
                     workspace: Tensor, *, k_new: Tensor | None = None, v_new: Tensor | None = None,
                     length: Tensor | None = None, Lkv: int = 0) -> Tensor:
    """One query row per sequence against a KV cache (csrc/attention_decode.cuh).

    q, out: (B, H*hd) views with unit inner stride; k_cache / v_cache: (B, capacity, H*hd) views sharing strides;
    workspace: fp32, at least `decode_workspace_bytes` bytes.
    Append mode (``length`` = int32 device tensor of one element): attends over cache rows [0, length) plus the new row
    ``k_new`` / ``v_new`` ((B, H*hd) views) and writes the new row into cache row ``length``; ``length`` itself is not
    changed (`decode_advance`). A ``length`` of B elements gives each sequence its own length (a ragged batch,
    ``b200enc_attention_decode_ragged``). Cross mode (``length`` None): attends over cache rows [0, Lkv)."""
    dev = _need_cuda(q, k_cache, v_cache, out, workspace, k_new, v_new, length)
    for name, t in (("q", q), ("k_cache", k_cache), ("v_cache", v_cache), ("out", out), ("k_new", k_new),
                    ("v_new", v_new)):
        _need(t, torch.bfloat16, name)
    _need(workspace, torch.float32, "workspace"), _need(length, torch.int32, "length")
    B, D = q.shape
    if D % n_heads != 0:
        raise ValueError("width not divisible by n_heads")
    if (k_cache.dim() != 3 or k_cache.shape != v_cache.shape or k_cache.stride() != v_cache.stride()
            or k_cache.shape[0] != B or k_cache.shape[2] != D or k_cache.stride(2) != 1):
        raise ValueError(f"k_cache / v_cache must be (B, capacity, {D}) views sharing strides, got "
                         f"{tuple(k_cache.shape)} / {tuple(v_cache.shape)}")
    if out.shape != q.shape or q.stride(1) != 1 or out.stride(1) != 1:
        raise ValueError("q / out must be (B, H*head_dim) views with unit inner stride")
    if (k_new is None) != (length is None) or (v_new is None) != (length is None):
        raise ValueError("append mode takes k_new, v_new and length together; cross mode none of them")
    new_bs = 0
    if k_new is not None:
        if k_new.shape != q.shape or v_new.shape != q.shape or k_new.stride() != v_new.stride() or k_new.stride(1) != 1:
            raise ValueError("k_new / v_new must be (B, H*head_dim) views sharing strides")
        new_bs = k_new.stride(0)
    if not workspace.is_contiguous():
        raise ValueError("workspace must be contiguous")
    if _per_sequence(length, B, "length"):
        _call(
            "b200enc_attention_decode_ragged", dict(B=B, H=n_heads, keys=k_cache.shape[1], append=True), dev,
            q.data_ptr(), q.stride(0), k_new.data_ptr(), v_new.data_ptr(), new_bs, k_cache.data_ptr(),
            v_cache.data_ptr(), k_cache.stride(0), k_cache.stride(1), k_cache.shape[1], length.data_ptr(),
            out.data_ptr(), out.stride(0), B, n_heads, D // n_heads, float(scale), workspace.data_ptr(),
            workspace.numel() * 4,
        )
        return out
    _call(
        "b200enc_attention_decode", dict(B=B, H=n_heads, keys=k_cache.shape[1], append=length is not None), dev,
        q.data_ptr(), q.stride(0), _ptr(k_new), _ptr(v_new), new_bs, k_cache.data_ptr(), v_cache.data_ptr(),
        k_cache.stride(0), k_cache.stride(1), k_cache.shape[1], _ptr(length), int(Lkv), out.data_ptr(), out.stride(0),
        B, n_heads, D // n_heads, float(scale), workspace.data_ptr(), workspace.numel() * 4,
    )
    return out


def embed_rows_at(ids: Tensor, tok: Tensor, pos: Tensor, pos0: Tensor, out: Tensor) -> Tensor:
    """`embed_rows` at a device-side position: out[b, l] = tok[ids[b, l]] + pos[pos0 + l] with ``pos0`` an int32 device
    tensor of one element (a decode step's cache length), or of B elements, pos0[b] for sequence b (a ragged batch).
    A position past the table gives a NaN row."""
    dev = _need_cuda(ids, tok, pos, pos0, out)
    _need(pos0, torch.int32, "pos0")
    dt = _embed_args("embed_rows_at", ids, tok, pos, out)
    B, L = ids.shape
    vocab, d = tok.shape
    name = "b200enc_embed_rows_at_ragged" if _per_sequence(pos0, B, "pos0") else "b200enc_embed_rows_at"
    _call(
        name, dict(rows=B * L, d=d), dev,
        ids.data_ptr(), B * L, L, tok.data_ptr(), pos.data_ptr(), pos.shape[0], pos0.data_ptr(), dt, vocab, d,
        out.data_ptr(),
    )
    return out


def decode_advance(length: Tensor, delta: int = 1) -> Tensor:
    """length += delta on the device (int32, one element, or one per sequence of a ragged batch): issued at the end of
    a decode step's decoder stack."""
    dev = _need_cuda(length)
    _need(length, torch.int32, "length")
    n = length.numel()
    if _per_sequence(length, n, "length"):
        _call("b200enc_decode_advance_ragged", dict(n=n, delta=delta), dev, length.data_ptr(), n, int(delta))
    else:
        _call("b200enc_decode_advance", dict(delta=delta), dev, length.data_ptr(), int(delta))
    return length


def _cache_view(name: str, t: Tensor, B: int, W: int) -> None:
    if t.dim() != 3 or t.shape[0] != B or t.shape[2] != W or t.stride(2) != 1:
        raise ValueError(f"{name} must be a (B={B}, capacity, {W}) view with unit inner stride, got {tuple(t.shape)}")


def kv_append(src: Tensor, cache: Tensor, length: Tensor) -> Tensor:
    """cache[b, length_b + r] = src[b, r] for r < P on the device: src (B, P, W) view (the k|v columns of the q|k|v
    rows), cache (B, capacity, W) view, ``length`` an int32 device tensor of 1 element (one length for the batch) or B
    (one per sequence). A row that would land at or past the capacity is not written; ``length`` is not changed."""
    dev = _need_cuda(src, cache, length)
    _need(src, torch.bfloat16, "src"), _need(cache, torch.bfloat16, "cache"), _need(length, torch.int32, "length")
    if src.dim() != 3 or src.stride(2) != 1:
        raise ValueError(f"src must be a (B, P, W) view with unit inner stride, got {tuple(src.shape)}")
    B, P, W = src.shape
    _cache_view("cache", cache, B, W)
    _call(
        "b200enc_kv_append", dict(B=B, P=P, W=W), dev,
        src.data_ptr(), src.stride(0), src.stride(1), cache.data_ptr(), cache.stride(0), cache.stride(1),
        cache.shape[1], length.data_ptr(), int(_per_sequence(length, B, "length")), B, P, W,
    )
    return cache


def attention_extend(q: Tensor, k_cache: Tensor, v_cache: Tensor, out: Tensor, n_heads: int, scale: float,
                     length: Tensor) -> Tensor:
    """Causal attention of P new query rows per sequence against a KV cache, the rows of sequence b at positions
    length_b + i (query i sees cache rows [0, length_b + i]): q, out (B, P, H*hd) views, k_cache / v_cache
    (B, capacity, H*hd) views sharing strides that already hold the new rows (`kv_append`), ``length`` as in
    `kv_append`. With every length 0 this is `attention(q, k, v, out, n_heads, scale, causal=True)` bit for bit."""
    dev = _need_cuda(q, k_cache, v_cache, out, length)
    for name, t in (("q", q), ("k_cache", k_cache), ("v_cache", v_cache), ("out", out)):
        _need(t, torch.bfloat16, name)
    _need(length, torch.int32, "length")
    if q.dim() != 3 or q.stride(2) != 1 or out.shape != q.shape or out.stride(2) != 1:
        raise ValueError("q / out must be (B, P, H*head_dim) views with unit inner stride")
    B, P, D = q.shape
    if D % n_heads != 0:
        raise ValueError("width not divisible by n_heads")
    _cache_view("k_cache", k_cache, B, D)
    if k_cache.shape != v_cache.shape or k_cache.stride() != v_cache.stride():
        raise ValueError("k_cache / v_cache must share shape and strides")
    _call(
        "b200enc_attention_extend", dict(B=B, H=n_heads, P=P, keys=k_cache.shape[1]), dev,
        q.data_ptr(), q.stride(0), q.stride(1), k_cache.data_ptr(), v_cache.data_ptr(), k_cache.stride(0),
        k_cache.stride(1), k_cache.shape[1], length.data_ptr(), int(_per_sequence(length, B, "length")),
        out.data_ptr(), out.stride(0), out.stride(1), B, n_heads, P, D // n_heads, float(scale),
    )
    return out
