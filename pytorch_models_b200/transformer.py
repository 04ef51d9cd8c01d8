"""B200-native drop-in for ``pytorch_models/transformer.py`` (reference lines cited inline).

Same class names, constructor signatures, attribute names and ``state_dict`` keys as the reference, so
``new.load_state_dict(ref.state_dict())`` is strict-clean and the reference's weight loaders (which write in place
into ``layer.sa.q_proj.weight`` etc.) keep working. The arithmetic does not run in PyTorch: ``forward`` sequences
hand-written sm_100a kernels from ``libb200enc.so``:

    pre-norm layer (transformer.py:125-126), 5 launches (+1 row_stats for the first layer of a stack whose input
    did not come with statistics; ViT's patch-embedding GEMM provides them)
        linear [3·inner, d], LayerNorm folded -> fused q|k|v                  (transformer.py:87,47-49)
        attention                             -> softmax(q kᵀ/√head_dim) v    (transformer.py:52)
        linear out_proj + bias + residual     -> x1 (+ partial LN statistics) (transformer.py:53,125)
        linear1, LayerNorm folded, erf-GELU   -> hidden                       (transformer.py:93,59-61)
        linear2 + bias + residual             -> x2 (+ partial LN statistics) (transformer.py:66,126)

    The row statistics (mean, rstd) a folded LayerNorm needs are produced by the epilogue of the GEMM that wrote
    its input (per-128-column (mean, M2) partials, combined in a fixed order by the consumer), so no separate pass
    over the residual stream is needed after the first layer.

Only what the kernels implement is accepted (self/cross attention, optionally causal and/or with attn_bias; head_dim 64,
80, 96, 112 or 128; GELU (erf / tanh), ReLU, SiLU; eval mode);
anything else raises ``NotImplementedError`` — there is no PyTorch fallback.
"""
from __future__ import annotations

import math
from types import SimpleNamespace

import torch
from torch import Tensor, nn

from . import ops, plans
from .compile import compilable, compilable_module

_SUPPORTED_HEAD_DIMS = (64, 80, 96, 112, 128)  # 64: attention_stream / attention_short, wider: attention_wide
_MAX_STAT_PARTS = 12  # libb200enc combines at most 12 partial statistics per row (d <= 1536)


# ----------------------------------------------------------------------------------------------- weight packing
_PACK_EPOCH = 0  # bumped by invalidate_packed(): every kernel-ready copy made before is rebuilt on next use


def invalidate_packed() -> None:
    """Forget every packed (kernel-ready) copy of module parameters in this process.

    The caches key on ``(data_ptr, _version, dtype, device, shape)`` of the source parameters, which sees parameter
    replacement, ``load_state_dict``, ``copy_`` / ``mul_`` on the parameter (what the reference loaders do,
    vit.py:172-197,290-304), dtype / device moves and ``resize_pe``. PyTorch keeps NO record of writes made through
    ``param.data`` (``p.data.copy_(ema)``: ``.data`` carries its own version counter), so after such a write call
    this function — otherwise the forward keeps using the stale bf16 copies, silently."""
    global _PACK_EPOCH
    _PACK_EPOCH += 1
    plans.invalidate_all()  # recorded launch plans hold pointers to the packed copies


def _version(p: Tensor) -> int:
    try:
        return p._version
    except RuntimeError:  # "Inference tensors do not track version counter" (created under torch.inference_mode)
        return -1


def _key(*params: Tensor | None) -> tuple:
    return (_PACK_EPOCH,) + tuple(
        None if p is None else (p.data_ptr(), _version(p), p.dtype, p.device, tuple(p.shape)) for p in params)


class _Packed:
    """Kernel-ready copies of a module's parameters, rebuilt whenever a source tensor is replaced or mutated in place
    (the reference loaders do both: vit.py:172-197 copy_, vit.py:290-304 mul_); see `invalidate_packed` for the one
    kind of write that cannot be seen (through ``.data``)."""

    def __init__(self) -> None:
        self.key: tuple | None = None
        self.t: SimpleNamespace | None = None

    def get(self, params: tuple, build) -> SimpleNamespace:
        key = _key(*params)
        if key != self.key:
            with torch.no_grad():
                self.t = build()
            self.key = key
        return self.t


def _cat_bias(linears: list[nn.Linear]) -> Tensor:
    parts = []
    for lin in linears:
        if lin.bias is None:
            parts.append(torch.zeros(lin.out_features, device=lin.weight.device, dtype=torch.float32))
        else:
            parts.append(lin.bias.detach().float())
    return torch.cat(parts)


def pack_plain(linears: list[nn.Linear]) -> SimpleNamespace:
    """bf16 [sum N, K] weight + fp32 bias of one or more linears that share their input."""
    w = torch.cat([lin.weight.detach() for lin in linears]).to(torch.bfloat16).contiguous()
    return SimpleNamespace(w=w, bias=_cat_bias(linears).contiguous(), colsum=None)


def pack_folded(linears: list[nn.Linear], norm: nn.LayerNorm) -> SimpleNamespace:
    """LayerNorm folded into the following linear:  LN(x) Wᵀ + b = rstd·(x W'ᵀ − mean·s) + c  with
    W' = W ⊙ gamma (bf16), s = row sums of the *rounded* W' (so the mean term cancels exactly against what the
    tensor cores accumulate) and c = W beta + b."""
    w32 = torch.cat([lin.weight.detach().float() for lin in linears])
    gamma, beta = norm.weight.detach().float(), norm.bias.detach().float()
    wg = (w32 * gamma[None, :]).to(torch.bfloat16).contiguous()
    colsum = wg.float().sum(dim=1).contiguous()
    c = (w32 @ beta + _cat_bias(linears)).contiguous()
    return SimpleNamespace(w=wg, bias=c, colsum=colsum)


def _as_tokens(x: Tensor, d: int) -> tuple[Tensor, tuple]:
    """(*, L, d) any dtype/strides -> contiguous bf16 (B, L, d) plus what is needed to restore the caller's view."""
    if not x.is_cuda:
        raise RuntimeError(
            "pytorch_models_b200 runs only on CUDA (sm_100a) tensors; there is no CPU fallback "
            f"(got a {x.device} tensor)"
        )
    if x.dim() < 2 or x.shape[-1] != d:
        raise ValueError(f"expected (*, L, {d}) input, got {tuple(x.shape)}")
    lead = x.shape[:-2]
    x3 = x.reshape(-1, x.shape[-2], d) if x.dim() != 3 else x
    if x3.dtype != torch.bfloat16 or not x3.is_contiguous():
        x3 = x3.to(torch.bfloat16).contiguous()
    return x3, (lead, x.dtype)


def _restore(y3: Tensor, meta: tuple) -> Tensor:
    lead, dtype = meta
    y = y3 if len(lead) == 1 else y3.reshape(*lead, y3.shape[-2], y3.shape[-1])
    return y if dtype == torch.bfloat16 else y.to(dtype)


# ----------------------------------------------------------------------------------------------- modules
class MHA(nn.Module):
    """Multi-head attention, reference ``MHA`` (transformer.py:9-53)."""

    def __init__(
        self,
        d_model: int,
        n_heads: int | None = None,
        head_dim: int | None = None,
        bias: bool = True,
        dropout: float = 0.0,
    ) -> None:
        super().__init__()
        # same defaulting rule as transformer.py:20-26
        if n_heads is None and head_dim is None:
            head_dim = 64
        if head_dim is None:
            head_dim = d_model // n_heads
        if n_heads is None:
            n_heads = d_model // head_dim
        inner = n_heads * head_dim
        self.q_proj = nn.Linear(d_model, inner, bias)
        self.k_proj = nn.Linear(d_model, inner, bias)
        self.v_proj = nn.Linear(d_model, inner, bias)
        self.out_proj = nn.Linear(inner, d_model, bias)
        self.n_heads = n_heads
        self.head_dim = head_dim
        self.dropout = dropout
        self._packs = {name: _Packed() for name in ("qkv", "q", "kv", "k", "v", "out")}

    # -- packing -------------------------------------------------------------------------------
    def _pack(self, name: str, linears: list[nn.Linear]) -> SimpleNamespace:
        params = tuple(p for lin in linears for p in (lin.weight, lin.bias))
        return self._packs[name].get(params, lambda: pack_plain(linears))

    def check_supported(self, attn_bias: Tensor | None = None, causal: bool = False) -> None:
        if self.head_dim not in _SUPPORTED_HEAD_DIMS:
            raise NotImplementedError(
                f"head_dim={self.head_dim}: the sm_100a attention kernels take head_dim 64, 80, 96, 112 or 128")
        if self.training and self.dropout > 0.0:
            raise NotImplementedError("attention dropout (training mode) is not supported; call .eval()")

    def _bias_view(self, attn_bias: Tensor | None, B: int, Lq: int, Lkv: int) -> Tensor | None:
        """``attn_bias`` as SDPA takes it (transformer.py:52: float added to the scores, or bool with True = attend),
        broadcast to (B, H, Lq, Lkv) without materialising the broadcast dimensions."""
        if attn_bias is None:
            return None
        b = attn_bias
        if b.dtype == torch.bool:
            b = torch.zeros(b.shape, device=b.device, dtype=torch.float32).masked_fill_(~b, float("-inf"))
        b = b.to(torch.float32)
        if b.dim() > 4:
            b = b.reshape(-1, *b.shape[-3:])
        if b.shape[-1] == 1 and Lkv > 1:  # broadcast over the keys: the kernel reads consecutive keys, materialise them
            b = b.expand(*b.shape[:-1], Lkv)
        if b.stride(-1) != 1 and b.shape[-1] > 1:
            b = b.contiguous()
        return b.expand(B, self.n_heads, Lq, Lkv)

    @property
    def scale(self) -> float:
        return 1.0 / math.sqrt(self.head_dim)  # F.scaled_dot_product_attention default (transformer.py:52)

    def forward(
        self,
        q: Tensor,
        k: Tensor | None = None,
        v: Tensor | None = None,
        attn_bias: Tensor | None = None,
        causal: bool = False,
    ) -> Tensor:
        self.check_supported(attn_bias, causal)
        q3, meta = _as_tokens(q, self.q_proj.in_features)
        out = self.run(q3, k, v, attn_bias, causal)
        if out.shape[0] != q3.shape[0]:
            meta = ((out.shape[0],), meta[1])
        return _restore(out, meta)

    def run(self, q3: Tensor, k: Tensor | None = None, v: Tensor | None = None, attn_bias: Tensor | None = None,
            causal: bool = False) -> Tensor:
        """`forward` on kernel-ready tokens: q3 bf16 contiguous (B, Lq, d) -> bf16 (B, Lq, d_out), no dtype round trip
        (what `MHAPooling` calls, so that the pooling head consists of library launches only)."""
        self.check_supported(attn_bias, causal)
        d_in = self.q_proj.in_features
        inner = self.n_heads * self.head_dim
        B, Lq, _ = q3.shape
        dev = q3.device
        if k is None and v is None:
            pk = self._pack("qkv", [self.q_proj, self.k_proj, self.v_proj])
            qkv = torch.empty(B, Lq, 3 * inner, device=dev, dtype=torch.bfloat16)
            ops.linear(q3.view(B * Lq, d_in), pk.w, pk.bias, qkv.view(B * Lq, 3 * inner))
            qv, kv_k, kv_v = qkv[:, :, :inner], qkv[:, :, inner:2 * inner], qkv[:, :, 2 * inner:]
        else:
            k = q3 if k is None else k
            k3, _ = _as_tokens(k, d_in)
            Bk, Lkv, _ = k3.shape
            pq = self._pack("q", [self.q_proj])
            qv = torch.empty(B, Lq, inner, device=dev, dtype=torch.bfloat16)
            ops.linear(q3.view(B * Lq, d_in), pq.w, pq.bias, qv.view(B * Lq, inner))
            if v is None or v is k:
                pkv = self._pack("kv", [self.k_proj, self.v_proj])
                kvbuf = torch.empty(Bk, Lkv, 2 * inner, device=dev, dtype=torch.bfloat16)
                ops.linear(k3.view(Bk * Lkv, d_in), pkv.w, pkv.bias, kvbuf.view(Bk * Lkv, 2 * inner))
            else:
                v3, _ = _as_tokens(v, d_in)
                kvbuf = torch.empty(Bk, Lkv, 2 * inner, device=dev, dtype=torch.bfloat16)
                pkk, pvv = self._pack("k", [self.k_proj]), self._pack("v", [self.v_proj])
                ops.linear(k3, pkk.w, pkk.bias, kvbuf[:, :, :inner])
                ops.linear(v3, pvv.w, pvv.bias, kvbuf[:, :, inner:])
            kv_k, kv_v = kvbuf[:, :, :inner], kvbuf[:, :, inner:]
            if B != Bk:  # broadcast query (the MAP-pooling probe, vit.py:35,41)
                if B != 1:
                    raise ValueError("query batch must be 1 or match the key batch")
                qv = qv.expand(Bk, Lq, inner).contiguous()
                B = Bk
        att = torch.empty(B, Lq, inner, device=dev, dtype=torch.bfloat16)
        ops.attention(qv, kv_k, kv_v, att, self.n_heads, self.scale, causal, self._bias_view(attn_bias, B, Lq, kv_k.shape[1]))
        po = self._pack("out", [self.out_proj])
        out = torch.empty(B, Lq, self.out_proj.out_features, device=dev, dtype=torch.bfloat16)
        ops.linear(att.view(B * Lq, inner), po.w, po.bias, out.view(B * Lq, -1))
        return out


_ACTS = dict(
    gelu=nn.GELU,
    approximate_gelu=lambda: nn.GELU(approximate="tanh"),
    relu=lambda: nn.ReLU(inplace=True),
    silu=nn.SiLU,
)


class MLP(nn.Sequential):
    """``linear1 -> act -> linear2 -> dropout`` with the reference's child names/order (transformer.py:56-67)."""

    def __init__(self, in_dim: int, hidden_dim: float, dropout: float = 0.0, act: str = "gelu") -> None:
        super().__init__()
        self.linear1 = nn.Linear(in_dim, hidden_dim)
        self.act = _ACTS[act]()
        self.linear2 = nn.Linear(hidden_dim, in_dim)
        self.dropout = nn.Dropout(dropout)
        self._act_name = act
        self._p1, self._p2 = _Packed(), _Packed()

    def check_supported(self) -> None:
        if self.training and self.dropout.p > 0.0:
            raise NotImplementedError("MLP dropout (training mode) is not supported; call .eval()")

    @property
    def gelu_mode(self) -> bool | str:
        """Epilogue selector of `ops.linear` for the reference's four activations (transformer.py:60-65)."""
        return {"gelu": True, "approximate_gelu": "tanh", "relu": "relu", "silu": "silu"}[self._act_name]

    def pack1(self, norm: nn.LayerNorm | None) -> SimpleNamespace:
        lin = self.linear1
        if norm is None:
            return self._p1.get((lin.weight, lin.bias), lambda: pack_plain([lin]))
        return self._p1.get((lin.weight, lin.bias, norm.weight, norm.bias), lambda: pack_folded([lin], norm))

    def pack2(self) -> SimpleNamespace:
        lin = self.linear2
        return self._p2.get((lin.weight, lin.bias), lambda: pack_plain([lin]))

    def forward(self, x: Tensor) -> Tensor:
        self.check_supported()
        d = self.linear1.in_features
        x3, meta = _as_tokens(x.unsqueeze(0) if x.dim() == 2 else x, d)
        B, L, _ = x3.shape
        p1, p2 = self.pack1(None), self.pack2()
        hidden = torch.empty(B * L, self.linear1.out_features, device=x3.device, dtype=torch.bfloat16)
        out = torch.empty(B, L, d, device=x3.device, dtype=torch.bfloat16)
        ops.linear(x3.view(B * L, d), p1.w, p1.bias, hidden, gelu=self.gelu_mode)
        ops.linear(hidden, p2.w, p2.bias, out.view(B * L, d))
        y = _restore(out, meta)
        return y.squeeze(0) if x.dim() == 2 else y


class DecoderLayer(nn.Module):
    """Reference ``DecoderLayer`` (transformer.py:70-105): causal self-attention, optional cross-attention to an
    encoder ``memory``, MLP; pre-norm (:97-99) or post-norm (:101-103). ``EncoderLayer`` is the same sequence without
    the mask and without cross-attention, exactly as in the reference (transformer.py:108).

    Launch sequence, pre-norm (one row per launch; LayerNorms never run as separate passes):
        linear [3·inner, d], sa_norm folded        -> q|k|v
        attention (causal for the decoder)         -> att
        linear sa.out_proj + bias + x              -> x1, partial statistics of x1
        [cross-attention only]
        linear ca.q_proj, ca_norm folded (on x1)   -> qc
        linear [ca.k_proj; ca.v_proj] on memory    -> k|v of the memory (memory is not normalised, :98)
        attention                                  -> att
        linear ca.out_proj + bias + x1             -> x2, partial statistics of x2
        linear1, mlp_norm folded, GELU             -> hidden
        linear2 + bias + x2                        -> out, partial statistics of out for the next layer
    """

    _causal = True

    def __init__(
        self,
        d_model: int,
        n_heads: int | None = None,
        head_dim: int | None = None,
        cross_attn: bool = False,
        bias: bool = True,
        mlp_ratio: float = 4.0,
        dropout: float = 0.0,
        act: str = "gelu",
        pre_norm: bool = True,
        norm_eps: float = 1e-5,
    ) -> None:
        super().__init__()
        self.pre_norm = pre_norm
        self.sa_norm = nn.LayerNorm(d_model, norm_eps)
        self.sa = MHA(d_model, n_heads, head_dim, bias, dropout)
        self.ca_norm = nn.LayerNorm(d_model, norm_eps) if cross_attn else None
        self.ca = MHA(d_model, n_heads, head_dim, bias, dropout) if cross_attn else None
        self.mlp_norm = nn.LayerNorm(d_model, norm_eps)
        self.mlp = MLP(d_model, int(d_model * mlp_ratio), dropout, act)
        self._pqkv, self._pcq, self._pcqkv = _Packed(), _Packed(), _Packed()

    # -- packing -------------------------------------------------------------------------------
    def _pack_proj(self, slot: _Packed, lins: list[nn.Linear], norm: nn.LayerNorm) -> SimpleNamespace:
        params = tuple(p for lin in lins for p in (lin.weight, lin.bias))
        if self.pre_norm:
            return slot.get(params + (norm.weight, norm.bias), lambda: pack_folded(lins, norm))
        return slot.get(params, lambda: pack_plain(lins))

    def _pack_qkv(self) -> SimpleNamespace:
        sa = self.sa
        return self._pack_proj(self._pqkv, [sa.q_proj, sa.k_proj, sa.v_proj], self.sa_norm)

    def workspace(self, B: int, L: int, device: torch.device, Lm: int = 0) -> SimpleNamespace:
        d = self.sa_norm.normalized_shape[0]
        inner = self.sa.n_heads * self.sa.head_dim
        M = B * L
        e = lambda *s, dt=torch.bfloat16: torch.empty(*s, device=device, dtype=dt)  # noqa: E731
        parts = (d + 127) // 128
        fused = self.pre_norm and parts <= _MAX_STAT_PARTS
        ws = SimpleNamespace(
            qkv=e(B, L, 3 * inner), att=e(B, L, inner), hidden=e(M, self.mlp.linear1.out_features), mid=e(M, d),
            tmp=None if self.pre_norm else e(M, d), stats=e(M, 2, dt=torch.float32),
            parts_mid=e(M, parts, 2, dt=torch.float32) if fused else None,
            parts_out=e(M, parts, 2, dt=torch.float32) if fused else None,
            Lm=Lm,
        )
        if self.ca is not None:
            ci = self.ca.n_heads * self.ca.head_dim
            ws.catt, ws.mid2 = e(B, L, ci), e(M, d)
            if Lm > 0:
                ws.cq, ws.ckv = e(B, L, ci), e(B, Lm, 2 * ci)
            else:  # no memory: the reference's MHA falls back to k = v = q (transformer.py:44-45)
                ws.cqkv = e(B, L, 3 * ci)
            ws.parts_mid2 = e(M, parts, 2, dt=torch.float32) if fused else None
        return ws

    def run(self, x3: Tensor, out3: Tensor, ws: SimpleNamespace, stats_in: Tensor | None = None,
            want_stats: bool = False, memory3: Tensor | None = None) -> Tensor | None:
        """x3 (B, L, d) bf16 contiguous -> out3 (same shape, must not alias x3); memory3 (B, Lm, d) bf16 contiguous.

        ``stats_in``: partial LayerNorm statistics of x3 written by the producing GEMM (else a row_stats pass runs).
        Returns the partial statistics of out3 when ``want_stats`` (for the next layer's sa_norm), else None."""
        sa, ca = self.sa, self.ca
        sa.check_supported()
        self.mlp.check_supported()
        B, L, d = x3.shape
        inner = sa.n_heads * sa.head_dim
        qkv = ws.qkv

        def attend_self(_qkv2: Tensor, _att2: Tensor) -> None:  # takes the (B, L, ·) views of the same buffers
            ops.attention(qkv[:, :, :inner], qkv[:, :, inner:2 * inner], qkv[:, :, 2 * inner:], ws.att, sa.n_heads,
                          sa.scale, self._causal)

        cross = None
        if ca is not None:
            ca.check_supported()
            ci = ca.n_heads * ca.head_dim
            if memory3 is None:
                # memory=None: MHA.forward(q, None) takes k = v = q (transformer.py:44-45), i.e. the cross-attention
                # block degenerates to un-masked self-attention with the ca weights on ca_norm(x) (pre-norm) / x
                if ws.Lm != 0:
                    raise ValueError("workspace was sized for a memory but none was given")
                pcq = self._pack_proj(self._pcqkv, [ca.q_proj, ca.k_proj, ca.v_proj], self.ca_norm)
                cq_out = ws.cqkv.view(B * L, 3 * ci)
                cq, ck, cv = ws.cqkv[:, :, :ci], ws.cqkv[:, :, ci:2 * ci], ws.cqkv[:, :, 2 * ci:]
            else:
                if memory3.shape[0] != B or memory3.shape[2] != d or memory3.shape[1] != ws.Lm:
                    raise ValueError(f"memory {tuple(memory3.shape)} does not match the workspace / batch")
                Mm = B * ws.Lm
                pcq = self._pack_proj(self._pcq, [ca.q_proj], self.ca_norm)
                pckv = ca._pack("kv", [ca.k_proj, ca.v_proj])
                cq_out = ws.cq.view(B * L, ci)
                cq, ck, cv = ws.cq, ws.ckv[:, :, :ci], ws.ckv[:, :, ci:]

            def attend_cross(_catt2: Tensor) -> None:
                if memory3 is not None:  # the memory is not normalised (transformer.py:98)
                    ops.linear(memory3.view(Mm, d), pckv.w, pckv.bias, ws.ckv.view(Mm, 2 * ci))
                ops.attention(cq, ck, cv, ws.catt, ca.n_heads, ca.scale)

            cross = (pcq, cq_out, attend_cross)
        return self._launch(x3.view(B * L, d), out3.view(B * L, d), ws, stats_in, want_stats, attend_self, cross)

    def step(self, x2: Tensor, out2: Tensor, ws: SimpleNamespace, cache: "KVCache", i: int,
             stats_in: Tensor | None = None, want_stats: bool = False) -> Tensor | None:
        """`run` for one new token per sequence against layer ``i`` of a KV cache: x2 (B, d) -> out2 (B, d).

        Each attention is `ops.attention_decode` over the cache (the self-attention appends this token's k|v row); the
        memory's [k; v] projection is not recomputed (it lives in the cache)."""
        sa, ca = self.sa, self.ca
        B = x2.shape[0]
        inner = sa.n_heads * sa.head_dim
        kv = cache.kv[i]

        def attend_self(qkv: Tensor, att: Tensor) -> None:
            ops.attention_decode(qkv[:, :inner], kv[:, :, :inner], kv[:, :, inner:], att, sa.n_heads, sa.scale,
                                 cache.work, k_new=qkv[:, inner:2 * inner], v_new=qkv[:, 2 * inner:],
                                 length=cache.length)

        cross = None
        if ca is not None:
            ci = ca.n_heads * ca.head_dim
            cq, mkv = ws.cqkv.view(B, 3 * ci)[:, :ci], cache.memory_kv[i]

            def attend_cross(catt: Tensor) -> None:
                ops.attention_decode(cq, mkv[:, :, :ci], mkv[:, :, ci:], catt, ca.n_heads, ca.scale, cache.work,
                                     Lkv=mkv.shape[1])

            cross = (self._pack_proj(self._pcq, [ca.q_proj], self.ca_norm), cq, attend_cross)
        return self._launch(x2, out2, ws, stats_in, want_stats, attend_self, cross)

    def extend(self, x2: Tensor, out2: Tensor, ws: SimpleNamespace, cache: "KVCache", i: int,
               stats_in: Tensor | None = None, want_stats: bool = False) -> Tensor | None:
        """`run` for P new tokens per sequence against layer ``i`` of a KV cache: x2 (B*P, d) -> out2 (B*P, d), with
        ``ws`` the workspace of (B, P) rows (and the memory's length, for its cross-attention buffers).

        The self-attention writes the new k|v rows into the cache at each sequence's length (`ops.kv_append`), then
        attends causally from there over the cache (`ops.attention_extend`); the cross-attention reads the memory's
        [k; v] from the cache."""
        sa, ca = self.sa, self.ca
        inner = sa.n_heads * sa.head_dim
        kv = cache.kv[i]

        def attend_self(_qkv2: Tensor, _att2: Tensor) -> None:  # takes the (B, P, ·) views of the same buffers
            ops.kv_append(ws.qkv[:, :, inner:], kv, cache.length)
            ops.attention_extend(ws.qkv[:, :, :inner], kv[:, :, :inner], kv[:, :, inner:], ws.att, sa.n_heads,
                                 sa.scale, cache.length)

        cross = None
        if ca is not None:
            ci = ca.n_heads * ca.head_dim
            mkv = cache.memory_kv[i]

            def attend_cross(_catt2: Tensor) -> None:
                ops.attention(ws.cq, mkv[:, :, :ci], mkv[:, :, ci:], ws.catt, ca.n_heads, ca.scale)

            cross = (self._pack_proj(self._pcq, [ca.q_proj], self.ca_norm), ws.cq.view(-1, ci), attend_cross)
        return self._launch(x2, out2, ws, stats_in, want_stats, attend_self, cross)

    def _launch(self, x2: Tensor, out2: Tensor, ws: SimpleNamespace, stats_in: Tensor | None, want_stats: bool,
                attend_self, cross: tuple | None) -> Tensor | None:
        """The layer's launches on M token rows, x2 (M, d) -> out2 (M, d), for `run`, `step` and `extend`.

        ``attend_self(qkv, att)`` fills ``ws.att`` from the q|k|v rows in ``ws.qkv``; it is given their (M, ·) views.
        With cross-attention, ``cross`` is ``(pack, q_out, attend_cross)``: the cross-attention query projection (with
        ca_norm folded in pre-norm) writes ``q_out``, then ``attend_cross(catt)`` fills ``ws.catt``, given its (M, ·)
        view."""
        sa, mlp = self.sa, self.mlp
        M = x2.shape[0]
        pq = self._pack_qkv()
        po = sa._pack("out", [sa.out_proj])
        p1 = mlp.pack1(self.mlp_norm if self.pre_norm else None)
        p2 = mlp.pack2()
        qkv, att = ws.qkv.view(M, -1), ws.att.view(M, -1)
        if cross is not None:
            pc, cq, attend_cross = cross
            pco = self.ca._pack("out", [self.ca.out_proj])
            catt = ws.catt.view(M, -1)
        if self.pre_norm:
            if stats_in is None:
                stats_in = ops.row_stats(x2, self.sa_norm.eps, ws.stats)
            ops.linear(x2, pq.w, pq.bias, qkv, colsum=pq.colsum, rowstats=stats_in, ln_eps=self.sa_norm.eps)
            attend_self(qkv, att)
            ops.linear(att, po.w, po.bias, ws.mid, residual=x2, stats_out=ws.parts_mid)
            mid, mid_stats = ws.mid, ws.parts_mid
            if cross is not None:
                if mid_stats is None:
                    mid_stats = ops.row_stats(mid, self.ca_norm.eps, ws.stats)
                ops.linear(mid, pc.w, pc.bias, cq, colsum=pc.colsum, rowstats=mid_stats, ln_eps=self.ca_norm.eps)
                attend_cross(catt)
                ops.linear(catt, pco.w, pco.bias, ws.mid2, residual=mid, stats_out=ws.parts_mid2)
                mid, mid_stats = ws.mid2, ws.parts_mid2
            if mid_stats is None:
                mid_stats = ops.row_stats(mid, self.mlp_norm.eps, ws.stats)
            ops.linear(mid, p1.w, p1.bias, ws.hidden, colsum=p1.colsum, rowstats=mid_stats,
                       ln_eps=self.mlp_norm.eps, gelu=mlp.gelu_mode)
            out_stats = ws.parts_out if want_stats else None
            ops.linear(ws.hidden, p2.w, p2.bias, out2, residual=mid, stats_out=out_stats)
            return out_stats
        # post-norm (BERT, GPT): transformer.py:101-103,128-129
        g1, b1 = norm_vectors(self.sa_norm)
        g2, b2 = norm_vectors(self.mlp_norm)
        ops.linear(x2, pq.w, pq.bias, qkv)
        attend_self(qkv, att)
        ops.linear(att, po.w, po.bias, ws.tmp, residual=x2)
        ops.layernorm(ws.tmp, g1, b1, self.sa_norm.eps, ws.mid)
        mid = ws.mid
        if cross is not None:
            gc, bc = norm_vectors(self.ca_norm)
            ops.linear(mid, pc.w, pc.bias, cq)
            attend_cross(catt)
            ops.linear(catt, pco.w, pco.bias, ws.tmp, residual=mid)
            ops.layernorm(ws.tmp, gc, bc, self.ca_norm.eps, ws.mid2)
            mid = ws.mid2
        ops.linear(mid, p1.w, p1.bias, ws.hidden, gelu=mlp.gelu_mode)
        ops.linear(ws.hidden, p2.w, p2.bias, ws.tmp, residual=mid)
        ops.layernorm(ws.tmp, g2, b2, self.mlp_norm.eps, out2)
        return None

    def forward(self, x: Tensor, memory: Tensor | None = None) -> Tensor:
        d = self.sa_norm.normalized_shape[0]
        x3, meta = _as_tokens(x, d)
        m3 = None
        if self.ca is not None and memory is not None:
            m3, _ = _as_tokens(memory, d)
        out3 = torch.empty_like(x3)
        if x3.numel():
            ws = self.workspace(x3.shape[0], x3.shape[1], x3.device, 0 if m3 is None else m3.shape[1])
            self.run(x3, out3, ws, memory3=m3)
        return _restore(out3, meta)


class EncoderLayer(DecoderLayer):
    """Reference ``EncoderLayer`` (transformer.py:108-130): a ``DecoderLayer`` without cross-attention whose
    self-attention is not masked."""

    _causal = False

    def __init__(
        self,
        d_model: int,
        n_heads: int | None = None,
        head_dim: int | None = None,
        bias: bool = True,
        mlp_ratio: float = 4.0,
        dropout: float = 0.0,
        act: str = "gelu",
        pre_norm: bool = True,
        norm_eps: float = 1e-5,
    ) -> None:
        super().__init__(d_model, n_heads, head_dim, False, bias, mlp_ratio, dropout, act, pre_norm, norm_eps)

    def forward(self, x: Tensor) -> Tensor:
        return super().forward(x)


def norm_vectors(norm: nn.LayerNorm) -> tuple[Tensor, Tensor]:
    """fp32 contiguous (gamma, beta) of a LayerNorm, cached on the module until the parameters change."""
    key = _key(norm.weight, norm.bias)
    hit = norm.__dict__.get("_b200_vectors")
    if hit is None or hit[0] != key:
        with torch.no_grad():
            hit = (key, (norm.weight.detach().float().contiguous(), norm.bias.detach().float().contiguous()))
        norm.__dict__["_b200_vectors"] = hit
    return hit[1]


@compilable_module
class Encoder(nn.Sequential):
    """Reference ``Encoder`` (transformer.py:133-149): an ``nn.Sequential`` of ``EncoderLayer`` — iteration, ``len``
    and indexing behave the same; ``forward`` additionally shares one workspace across the layers."""

    def __init__(
        self,
        n_layers: int,
        d_model: int,
        n_heads: int | None = None,
        head_dim: int | None = None,
        bias: bool = True,
        mlp_ratio: float = 4.0,
        dropout: float = 0.0,
        act: str = "gelu",
        pre_norm: bool = True,
        norm_eps: float = 1e-5,
    ) -> None:
        super().__init__()
        for _ in range(n_layers):
            self.append(EncoderLayer(d_model, n_heads, head_dim, bias, mlp_ratio, dropout, act, pre_norm, norm_eps))
        self.d_model = d_model

    def run(self, x3: Tensor, stats: Tensor | None = None) -> Tensor:
        """bf16 contiguous (B, L, d) -> new tensor of the same shape; x3 is left untouched. ``stats``: partial
        LayerNorm statistics of x3's rows, (B*L, ceil(d/128), 2), if the kernel that produced x3 emitted them."""
        return _run_stack(list(self), x3, None, stats0=stats)

    def wants_stats(self) -> bool:
        """True if the first layer can consume partial statistics written by the producer of its input."""
        layers = list(self)
        return bool(layers) and layers[0].pre_norm and (self.d_model + 127) // 128 <= _MAX_STAT_PARTS

    @compilable(lambda self, x, extra: (x.shape, x.dtype))
    def forward(self, x: Tensor) -> Tensor:
        x3, meta = _as_tokens(x, self.d_model)
        if len(self) == 0 or x3.numel() == 0:
            return _restore(self.run(x3), meta)
        return _restore(plans.run(self, (x3,), self.run), meta)  # recorded once, replayed by one C-ABI call


def partial_stats_of(row: Tensor) -> Tensor:
    """(parts, 2) fp32 per-128-column (mean, M2) of one stored bf16 row — what the GEMM epilogue writes for the rows it
    produces; used for rows that no GEMM produces (the class token)."""
    v = row.detach().to(torch.bfloat16).float().flatten()
    out = []
    for c0 in range(0, v.numel(), 128):
        sl = v[c0:c0 + 128]
        mean = sl.mean()
        out.append(torch.stack([mean, ((sl - mean) ** 2).sum()]))
    return torch.stack(out).contiguous()


def _run_stack(layers: list, x3: Tensor, memory3: Tensor | None, final_stats: bool = False,
               stats0: Tensor | None = None, after_layer=None):
    """Run a list of layers over bf16 contiguous (B, L, d) tokens with one shared workspace and two ping-pong output
    buffers; the LayerNorm statistics travel from each layer's last GEMM to the next layer's first.

    With ``final_stats`` returns ``(tokens, stats)`` where stats are the partial LayerNorm statistics of the output
    rows (None when the stack cannot produce them) for a LayerNorm folded into whatever consumes the tokens.
    ``stats0``: partial statistics of x3's rows if its producer wrote them (saves the first layer's row_stats pass).
    ``after_layer(i, ws)`` runs after layer ``i``, before the next layer overwrites the workspace."""
    if not layers or x3.numel() == 0:
        return (x3.clone(), None) if final_stats else x3.clone()
    B, L, _ = x3.shape
    ws = layers[0].workspace(B, L, x3.device, 0 if memory3 is None else memory3.shape[1])
    bufs = [torch.empty_like(x3), torch.empty_like(x3) if len(layers) > 1 else None]
    cur, stats = x3, stats0
    for i, layer in enumerate(layers):
        want = final_stats or i + 1 < len(layers)
        stats = layer.run(cur, bufs[i % 2], ws, stats_in=stats, want_stats=want, memory3=memory3)
        if after_layer is not None:
            after_layer(i, ws)
        cur = bufs[i % 2]
    return (cur, stats) if final_stats else cur


@compilable_module
class Decoder(nn.ModuleList):
    """Reference ``Decoder`` (transformer.py:152-176): an ``nn.ModuleList`` of ``DecoderLayer`` called as
    ``decoder(x, memory)``; ``forward`` additionally shares one workspace across the layers."""

    def __init__(
        self,
        n_layers: int,
        d_model: int,
        n_heads: int | None = None,
        head_dim: int | None = None,
        cross_attn: bool = False,
        bias: bool = True,
        mlp_ratio: float = 4.0,
        dropout: float = 0.0,
        act: str = "gelu",
        pre_norm: bool = True,
        norm_eps: float = 1e-5,
    ) -> None:
        super().__init__()
        for _ in range(n_layers):
            self.append(
                DecoderLayer(d_model, n_heads, head_dim, cross_attn, bias, mlp_ratio, dropout, act, pre_norm, norm_eps)
            )
        self.d_model = d_model

    def run(self, x3: Tensor, memory3: Tensor | None = None, final_stats: bool = False):
        """bf16 contiguous (B, L, d) [+ memory (B, Lm, d)] -> new tensor of x3's shape; inputs are left untouched.
        ``final_stats``: also return the output rows' partial LayerNorm statistics (see `_run_stack`)."""
        return _run_stack(list(self), x3, memory3, final_stats)

    @compilable(lambda self, x, extra: (x.shape, x.dtype))
    def forward(self, x: Tensor, memory: Tensor | None = None) -> Tensor:
        x3, meta = _as_tokens(x, self.d_model)
        m3 = None
        if memory is not None and len(self) and self[0].ca is not None:
            m3, _ = _as_tokens(memory, self.d_model)
        if len(self) == 0 or x3.numel() == 0:
            return _restore(self.run(x3, m3), meta)
        return _restore(plans.run(self, (x3,) if m3 is None else (x3, m3), self.run), meta)

    # -- incremental decoding ------------------------------------------------------------------
    def _check_decodable(self) -> None:
        for layer in self:
            layer.sa.check_supported()
            layer.mlp.check_supported()
            if layer.ca is not None:
                layer.ca.check_supported()

    def new_kv_cache(self, batch: int, capacity: int, memory: Tensor | None = None) -> "KVCache":
        """An empty `KVCache` for ``batch`` sequences of up to ``capacity`` tokens. A decoder with cross-attention
        needs its encoder ``memory`` (batch, Lm, d): the [k; v] projection of every layer runs on it here, once."""
        if not len(self):
            raise ValueError("a decoder without layers has nothing to cache")
        self._check_decodable()
        if batch < 1 or capacity < 1:
            raise ValueError(f"batch={batch} and capacity={capacity} must be >= 1")
        m3 = None
        if self[0].ca is not None:
            if memory is None:
                # without memory the block attends k = v = q over the current tokens without a mask
                # (transformer.py:44-45, `DecoderLayer.run` here): every token changes every earlier output
                raise NotImplementedError("a cross-attention decoder without memory cannot be decoded incrementally")
            if memory.dim() != 3 or memory.shape[0] != batch or memory.shape[2] != self.d_model or memory.shape[1] < 1:
                raise ValueError(f"memory {tuple(memory.shape)} does not match (batch={batch}, Lm, d={self.d_model})")
            m3, _ = _as_tokens(memory, self.d_model)
        return KVCache(self, batch, capacity, m3)

    def prefill(self, x3: Tensor, cache: "KVCache", lengths=None) -> tuple[Tensor, Tensor | None]:
        """`run` (``final_stats=True``) on the first P tokens of an EMPTY cache, keeping every layer's k|v rows in it:
        x3 bf16 contiguous (B, P, d) -> (tokens, partial statistics or None). Sets the cache length to P.

        ``lengths``: B host ints in [1, P] for a ragged batch of right-padded sequences; sequence b then holds
        ``lengths[b]`` tokens. Causal attention keeps every real token away from the padding rows after it, so the
        stack runs unchanged; the padding rows' k|v land in cache rows at or past each sequence's length, which no step
        reads and the steps overwrite. The output rows of padding positions are not meaningful."""
        self._check_decodable()
        B, P, _ = x3.shape
        cache.check_prefill(B, P)
        lengths = cache.check_lengths(lengths, P)

        def keep_kv(i: int, ws: SimpleNamespace) -> None:
            cache.kv[i][:, :P].copy_(ws.qkv[:, :, ws.qkv.shape[2] // 3:])  # the k|v of the layer's q|k|v rows

        out = _run_stack(list(self), x3, cache.memory3, final_stats=True, after_layer=keep_kv)
        cache.set_lengths(P, lengths)
        return out

    def step(self, x3: Tensor, cache: "KVCache") -> tuple[Tensor, Tensor | None]:
        """One token per sequence: x3 bf16 contiguous (B, 1, d) at position ``cache.n`` -> (tokens (B, 1, d), partial
        statistics or None). Appends every layer's k|v row to the cache and advances its length by one, on the device
        (the launches are the same at every position, so `graphs.GraphedStep` can capture them). The returned tokens
        live in a buffer of the cache that the next step overwrites."""
        self._check_decodable()
        B = x3.shape[0]
        cache.check_step(B)
        ws = cache.ws
        cur, stats = x3.view(B, self.d_model), None
        for i, layer in enumerate(self):
            out = cache.bufs[i % 2]
            stats = layer.step(cur, out, ws, cache, i, stats_in=stats, want_stats=True)
            cur = out
        ops.decode_advance(cache.length)
        cache.n += 1
        return cur.view(B, 1, self.d_model), stats

    def extend(self, x3: Tensor, cache: "KVCache", lengths=None) -> tuple[Tensor, Tensor | None]:
        """P more tokens per sequence on a cache that may already hold some: x3 bf16 contiguous (B, P, d), the tokens
        at positions ``seq_lengths[b] + i`` -> (tokens (B, P, d), partial statistics or None). The launches of
        `prefill`, except that each layer writes its k|v rows into the cache at each sequence's length and attends
        causally from there over the cache (and reads the memory's [k; v] from it); on an empty cache the result equals
        `prefill`'s bit for bit. Each sequence grows by P tokens, or by ``lengths[b]`` (B host ints in [1, P], rows
        right-padded as in a ragged `prefill`); a shared-length cache extended by unequal ``lengths`` becomes ragged."""
        self._check_decodable()
        B, P, d = x3.shape
        cache.check_extend(B, P)
        lengths = cache.check_lengths(lengths, P)
        Lm = 0 if cache.memory3 is None else cache.memory3.shape[1]
        ws = self[0].workspace(B, P, x3.device, Lm)
        bufs = [torch.empty_like(x3), torch.empty_like(x3) if len(self) > 1 else None]
        cur, stats = x3.view(B * P, d), None
        for i, layer in enumerate(self):
            out = bufs[i % 2].view(B * P, d)
            stats = layer.extend(cur, out, ws, cache, i, stats_in=stats, want_stats=True)
            cur = out
        cache.extend_lengths(P, lengths)
        return cur.view(B, P, d), stats


class KVCache:
    """Keys and values of the tokens a `Decoder` has seen, for incremental decoding (`Decoder.new_kv_cache`).

    Per layer: ``kv[i]`` (batch, capacity, 2·inner) bf16, the self-attention k|v rows of positions [0, n); with
    cross-attention ``memory_kv[i]`` (batch, Lm, 2·inner), the projected memory. ``length`` is the device-side int32
    length the decode kernels read and the step advances; ``n`` is its host mirror, used for the argument checks. Also
    holds the step's scratch buffers and the fp32 workspace of the decode kernel.

    All sequences of a batch have the same length, unless the cache was filled by a ragged prefill (``lengths``): then
    ``length`` is the cache's (batch,) int32 tensor of per-sequence lengths, which the step's launches read and advance
    instead; ``n`` is the longest sequence's length and ``pad[b]`` how many tokens sequence b is shorter, fixed for the
    whole fill. `seq_lengths` reads the per-sequence lengths on the host. A cache is valid for the weights it was
    filled with: after changing the model's parameters, start a new cache (this is not detected)."""

    def __init__(self, decoder: Decoder, batch: int, capacity: int, memory3: Tensor | None) -> None:
        layers = list(decoder)
        p = next(decoder.parameters())
        dev = p.device
        self.batch, self.capacity = batch, capacity
        self.n = 0
        self.pad = None
        self.shared_length = torch.zeros(1, device=dev, dtype=torch.int32)
        # allocated once, so that a step captured on a ragged fill keeps reading the same tensor after later fills
        self.seq_length = torch.zeros(batch, device=dev, dtype=torch.int32)
        self.length = self.shared_length
        self.memory3 = memory3
        e = lambda *s: torch.empty(*s, device=dev, dtype=torch.bfloat16)  # noqa: E731
        self.kv = [e(batch, capacity, 2 * layer.sa.n_heads * layer.sa.head_dim) for layer in layers]
        self.memory_kv = None
        ws_bytes = max(ops.decode_workspace_bytes(batch, layer.sa.n_heads, layer.sa.head_dim, capacity)
                       for layer in layers)
        if memory3 is not None:
            Lm, d = memory3.shape[1], memory3.shape[2]
            self.memory_kv = []
            for layer in layers:
                ca = layer.ca
                ci = ca.n_heads * ca.head_dim
                pkv = ca._pack("kv", [ca.k_proj, ca.v_proj])
                mkv = e(batch, Lm, 2 * ci)
                ops.linear(memory3.view(batch * Lm, d), pkv.w, pkv.bias, mkv.view(batch * Lm, 2 * ci))
                self.memory_kv.append(mkv)
                ws_bytes = max(ws_bytes, ops.decode_workspace_bytes(batch, ca.n_heads, ca.head_dim, Lm))
        self.work = torch.empty((ws_bytes + 3) // 4, device=dev, dtype=torch.float32)
        self.ws = layers[0].workspace(batch, 1, dev, 0)
        self.bufs = [e(batch, decoder.d_model), e(batch, decoder.d_model)]

    def reset(self) -> None:
        """Empty the cache (for a new prefill); the buffers are kept."""
        self.length = self.shared_length
        self.length.zero_()
        self.n = 0
        self.pad = None

    @property
    def ragged(self) -> bool:
        """True when the sequences have their own lengths (the cache was filled by a prefill with ``lengths``)."""
        return self.pad is not None

    @property
    def seq_lengths(self) -> list[int]:
        """The number of tokens each sequence holds, from the host mirror (no device synchronisation)."""
        return [self.n] * self.batch if self.pad is None else [self.n - p for p in self.pad]

    def check_lengths(self, lengths, P: int) -> list[int] | None:
        """Validate the ``lengths`` of a ragged prefill of P tokens per row: None, or B host ints in [1, P]."""
        if lengths is None:
            return None
        if isinstance(lengths, Tensor):
            if lengths.is_cuda:
                raise ValueError("lengths must be host ints (a list or a CPU tensor), not a CUDA tensor: the checks "
                                 "and the host mirror of the cache need them without a device synchronisation")
            lengths = lengths.reshape(-1).tolist()
        lengths = [int(n) for n in lengths]
        if len(lengths) != self.batch:
            raise ValueError(f"lengths has {len(lengths)} entries for a batch of {self.batch}")
        bad = [n for n in lengths if not 1 <= n <= P]
        if bad:
            raise ValueError(f"length {bad[0]} is outside [1, {P}] (the prompts are right-padded to {P} tokens)")
        return lengths

    def set_lengths(self, P: int, lengths: list[int] | None) -> None:
        """After a prefill of P tokens per row: every sequence holds P tokens, or ``lengths[b]`` (ragged)."""
        if lengths is None:
            self.length = self.shared_length
            self.length.fill_(P)
            self.pad = None
        else:
            self.length = self.seq_length
            self.length.copy_(torch.tensor(lengths, dtype=torch.int32))
            self.pad = [P - n for n in lengths]
        self.n = P

    def check_prefill(self, batch: int, P: int) -> None:
        if batch != self.batch:
            raise ValueError(f"batch {batch} does not match the cache's batch {self.batch}")
        if self.n != 0:
            raise ValueError(f"prefill needs an empty cache (it holds {self.n} tokens; call reset())")
        if not 1 <= P <= self.capacity:
            raise ValueError(f"prefill of {P} tokens into a cache of capacity {self.capacity}")

    def extend_lengths(self, P: int, lengths: list[int] | None) -> None:
        """After an extend of P tokens per row: sequence b grows by ``lengths[b]`` (or P), on the host mirror and on
        the device. The cache stays shared-length while every sequence has the same length, else it becomes ragged."""
        new = [n + k for n, k in zip(self.seq_lengths, lengths or [P] * self.batch)]
        if not self.ragged and len(set(new)) == 1:
            self.length.fill_(new[0])
        else:
            self.length = self.seq_length
            self.length.copy_(torch.tensor(new, dtype=torch.int32))
            self.pad = [max(new) - n for n in new]
        self.n = max(new)

    def check_extend(self, batch: int, P: int) -> None:
        if batch != self.batch:
            raise ValueError(f"batch {batch} does not match the cache's batch {self.batch}")
        if P < 1 or self.n + P > self.capacity:
            raise ValueError(f"extend of {P} tokens onto {self.n} held tokens overflows a cache of capacity "
                             f"{self.capacity}")

    def check_step(self, batch: int) -> None:
        if batch != self.batch:
            raise ValueError(f"batch {batch} does not match the cache's batch {self.batch}")
        if self.n >= self.capacity:
            raise ValueError(f"the cache is full ({self.n} of {self.capacity} tokens)")


# ----------------------------------------------------------------------------------------------- language-model ends
def _embedding_tables(ids: Tensor, token_embs: nn.Embedding, pos_embs: Tensor) -> tuple[Tensor, Tensor]:
    """Refuse ids that are not on a CUDA device; the token and position tables as contiguous tensors of the one dtype
    (fp32 or bf16) the gather kernels take."""
    if not ids.is_cuda:
        raise RuntimeError(
            "pytorch_models_b200 runs only on CUDA (sm_100a) tensors; there is no CPU fallback "
            f"(got a {ids.device} tensor)"
        )
    tok = token_embs.weight.detach()
    pos = pos_embs.detach()
    if tok.dtype not in (torch.float32, torch.bfloat16):
        tok = tok.float()
    if pos.dtype != tok.dtype:
        pos = pos.to(tok.dtype)
    return tok.contiguous(), pos.contiguous()


def embed_tokens(ids: Tensor, token_embs: nn.Embedding, pos_embs: Tensor) -> Tensor:
    """``token_embs(ids) + pos_embs[:L]`` (bert.py:35-36, gpt2.py:22-23, gpt.py:25-26, whisper.py:47-48):
    (*, L) int64 -> contiguous bf16 (B, L, d) in one gather kernel."""
    tok, pos = _embedding_tables(ids, token_embs, pos_embs)
    L = ids.shape[-1]
    if L > pos.shape[0]:
        raise ValueError(f"sequence length {L} exceeds the {pos.shape[0]} rows of the position table")
    ids2 = ids.reshape(-1, L).to(torch.int64).contiguous()
    out = torch.empty(ids2.shape[0], L, tok.shape[1], device=ids.device, dtype=torch.bfloat16)
    return ops.embed_rows(ids2, tok, pos, out)


def embed_tokens_at(ids: Tensor, token_embs: nn.Embedding, pos_embs: Tensor, cache: KVCache) -> Tensor:
    """`embed_tokens` of new tokens at each sequence's cache length: (B,) or (B, 1) int64 (a step) or (B, P) (an
    extend) -> contiguous bf16 (B, L, d), row l of sequence b at position ``length_b + l``. The position is read on
    the device (the cache length), so a step's launch is the same at every position."""
    tok, pos = _embedding_tables(ids, token_embs, pos_embs)
    ids2 = ids.reshape(ids.shape[0] if ids.dim() else 1, -1).to(torch.int64).contiguous()
    out = torch.empty(*ids2.shape, tok.shape[1], device=ids.device, dtype=torch.bfloat16)
    return ops.embed_rows_at(ids2, tok, pos, cache.length, out)


def step_ids_batch(ids: Tensor) -> int:
    """Batch of a decode step's token ids: (B,) or (B, 1)."""
    if ids.dim() > 2 or (ids.dim() == 2 and ids.shape[1] != 1):
        raise ValueError(f"a decode step takes one token per sequence, (B,) or (B, 1) ids; got {tuple(ids.shape)}")
    return ids.shape[0] if ids.dim() else 1


class TiedLogits:
    """``norm(x) @ token_embs.weight.T`` (gpt2.py:25-26, whisper.py:50-51) or without the norm (gpt.py:28) as one
    GEMM: the final LayerNorm is folded into a cached bf16 copy of the embedding table (rows padded to a multiple of
    8 so that every logits row is 16-byte aligned; the padding columns are sliced off the returned view)."""

    def __init__(self) -> None:
        self._slot = _Packed()

    def _pack(self, emb: nn.Embedding, norm: nn.LayerNorm | None) -> SimpleNamespace:
        def build() -> SimpleNamespace:
            w32 = emb.weight.detach().float()
            V, d = w32.shape
            V8 = (V + 7) // 8 * 8
            if norm is None:
                w = torch.zeros(V8, d, device=w32.device, dtype=torch.bfloat16)
                w[:V] = w32
                return SimpleNamespace(w=w, bias=None, colsum=None, V=V)
            gamma, beta = norm.weight.detach().float(), norm.bias.detach().float()
            w = torch.zeros(V8, d, device=w32.device, dtype=torch.bfloat16)
            w[:V] = w32 * gamma[None, :]
            c = torch.zeros(V8, device=w32.device, dtype=torch.float32)
            c[:V] = w32 @ beta
            return SimpleNamespace(w=w, bias=c, colsum=w.float().sum(dim=1).contiguous(), V=V)

        params = (emb.weight,) if norm is None else (emb.weight, norm.weight, norm.bias)
        return self._slot.get(params, build)

    def __call__(self, x3: Tensor, emb: nn.Embedding, norm: nn.LayerNorm | None = None,
                 stats: Tensor | None = None) -> Tensor:
        """x3: bf16 contiguous (B, L, d); ``stats``: partial LayerNorm statistics of its rows if the producer wrote
        them (else one row_stats pass runs). Returns bf16 (B, L, vocab) — a view into rows of ceil8(vocab) columns."""
        B, L, d = x3.shape
        pk = self._pack(emb, norm)
        V8 = pk.w.shape[0]
        out = torch.empty(B, L, V8, device=x3.device, dtype=torch.bfloat16)
        if B * L:
            x2 = x3.view(B * L, d)
            if norm is None:
                ops.linear(x2, pk.w, None, out.view(B * L, V8))
            else:
                if stats is None:
                    stats = ops.row_stats(x2, norm.eps, torch.empty(B * L, 2, device=x3.device, dtype=torch.float32))
                ops.linear(x2, pk.w, pk.bias, out.view(B * L, V8), colsum=pk.colsum, rowstats=stats, ln_eps=norm.eps)
        return out[:, :, :pk.V]


class DecoderLM:
    """What ``GPT2``, ``GPT`` and ``WhisperDecoder`` share: token + position embedding, a `Decoder`, logits against the
    tied token table, and cached decoding on top of it. Holds no parameters; the model defines ``token_embs``,
    ``pos_embs``, ``layers`` (the `Decoder`), ``_logits`` (a `TiedLogits`) and, except for GPT, the final ``norm``."""

    def _logits_as(self, h: Tensor, stats: Tensor | None, lead: tuple) -> Tensor:
        """bf16 tokens (B, L, d) -> logits (*lead, vocab) in the parameters' dtype; ``stats``: partial LayerNorm
        statistics of h's rows, if its producer wrote them."""
        logits = self._logits(h, self.token_embs, getattr(self, "norm", None), stats)
        logits = logits.reshape(*lead, logits.shape[-1])
        out_dtype = self.token_embs.weight.dtype
        return logits if out_dtype == torch.bfloat16 else logits.to(out_dtype)

    # -- incremental decoding (no reference counterpart: the reference recomputes the whole prefix) ----------------
    def _check_capacity(self, capacity: int) -> None:
        if capacity > self.pos_embs.shape[0]:
            raise ValueError(f"capacity {capacity} exceeds the {self.pos_embs.shape[0]} rows of the position table")

    def new_kv_cache(self, batch: int, capacity: int) -> KVCache:
        """An empty KV cache for ``batch`` sequences of up to ``capacity`` <= max_seq_len tokens (see `prefill`)."""
        self._check_capacity(capacity)
        return self.layers.new_kv_cache(batch, capacity)

    def prefill(self, x: Tensor, cache: KVCache, lengths=None) -> Tensor:
        """`forward` on the prompt, (B, P) or (P,) ids (against the cache's memory for ``WhisperDecoder``), that also
        fills an empty ``cache``: (*, P, vocab) logits.

        ``lengths``: B host ints in [1, P] (a list or a CPU tensor) for prompts of different lengths, right-padded to P
        tokens; prompt b is ``x[b, :lengths[b]]``, and the steps then continue each sequence at its own position. The
        padding ids are replaced by a valid id before the embedding; the logits of padding positions are not
        meaningful (those of prompt b's last token are at ``lengths[b] - 1``)."""
        P = x.shape[-1]
        cache.check_prefill(x.reshape(-1, P).shape[0], P)
        lengths = cache.check_lengths(lengths, P)
        if lengths is not None:
            pad = torch.arange(P)[None, :] >= torch.tensor(lengths)[:, None]
            x = x.masked_fill(pad.reshape(x.shape).to(x.device), 0)
        h, stats = self.layers.prefill(embed_tokens(x, self.token_embs, self.pos_embs), cache, lengths)
        return self._logits_as(h, stats, x.shape)

    def step(self, x: Tensor, cache: KVCache) -> Tensor:
        """The next token of every sequence, (B,) or (B, 1) ids at position ``cache.n`` -> (B, vocab) logits, equal
        to ``forward(prefix)[:, -1]`` within bf16 rounding. Appends to the cache."""
        cache.check_step(step_ids_batch(x))
        self.layers._check_decodable()
        h, stats = self.layers.step(embed_tokens_at(x, self.token_embs, self.pos_embs, cache), cache)
        return self._logits_as(h, stats, h.shape[:1])

    def extend(self, x: Tensor, cache: KVCache, lengths=None) -> Tensor:
        """P more tokens of every sequence, (B, P) or (P,) ids continuing a cache that may already hold some (the next
        turn of a conversation, the next chunk of a long prompt) -> (*, P, vocab) logits, equal within bf16 rounding
        to ``forward`` of the whole sequence at those positions. On an empty cache it is `prefill`.

        ``lengths``: B host ints in [1, P] when sequence b appends only ``x[b, :lengths[b]]`` (right-padded to P as in
        `prefill`); the logits of padding positions are not meaningful."""
        P = x.shape[-1]
        ids = x.reshape(-1, P)
        cache.check_extend(ids.shape[0], P)
        lengths = cache.check_lengths(lengths, P)
        self.layers._check_decodable()
        if lengths is not None:
            pad = torch.arange(P)[None, :] >= torch.tensor(lengths)[:, None]
            ids = ids.masked_fill(pad.to(ids.device), 0)
        h, stats = self.layers.extend(embed_tokens_at(ids, self.token_embs, self.pos_embs, cache), cache, lengths)
        return self._logits_as(h, stats, x.shape)
