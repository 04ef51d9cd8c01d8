"""B200-native drop-in for ``GPT2`` (reference ``pytorch_models/text/gpt2.py:11-99``).

Same constructor, ``state_dict`` keys (``token_embs``, ``pos_embs``, ``layers.*``, ``norm``) and call signature.
``forward`` is: one gather kernel (token + position embedding), the pre-norm ``Decoder`` stack (causal tcgen05
attention, tanh-GELU fused into linear1), and one GEMM against the tied embedding table with the final LayerNorm
folded in — its row statistics come out of the last layer's linear2 epilogue.
"""
from __future__ import annotations

import torch
from torch import Tensor, nn

from ..compile import compilable, compilable_module
from ..transformer import Decoder, KVCache, TiedLogits, embed_tokens, embed_tokens_at, step_ids_batch


@compilable_module
class GPT2(nn.Module):
    vocab_size = 50257
    max_seq_len: int = 1024

    def __init__(self, n_layers: int, d_model: int, dropout: float = 0.0) -> None:
        super().__init__()
        self.token_embs = nn.Embedding(self.vocab_size, d_model)
        self.pos_embs = nn.Parameter(torch.zeros(self.max_seq_len, d_model))
        self.layers = Decoder(n_layers, d_model, dropout=dropout, act="approximate_gelu")
        self.norm = nn.LayerNorm(d_model)
        self._logits = TiedLogits()

    @compilable(lambda self, x, extra: ((*x.shape, self.token_embs.weight.shape[0]), self.token_embs.weight.dtype))
    def forward(self, x: Tensor) -> Tensor:
        """(*, L) int64 token ids -> (*, L, vocab) logits in the parameters' dtype (gpt2.py:21-27)."""
        out_dtype = self.token_embs.weight.dtype
        h, stats = self.layers.run(embed_tokens(x, self.token_embs, self.pos_embs), final_stats=True)
        logits = self._logits(h, self.token_embs, self.norm, stats)
        logits = logits.reshape(*x.shape, logits.shape[-1])
        return logits if out_dtype == torch.bfloat16 else logits.to(out_dtype)

    # -- incremental decoding (no reference counterpart: the reference recomputes the whole prefix) ----------------
    def new_kv_cache(self, batch: int, capacity: int) -> KVCache:
        """An empty KV cache for ``batch`` sequences of up to ``capacity`` <= max_seq_len tokens (see `prefill`)."""
        if capacity > self.pos_embs.shape[0]:
            raise ValueError(f"capacity {capacity} exceeds the {self.pos_embs.shape[0]} rows of the position table")
        return self.layers.new_kv_cache(batch, capacity)

    def prefill(self, x: Tensor, cache: KVCache) -> Tensor:
        """`forward` on the prompt, (B, P) or (P,) ids, that also fills an empty ``cache``: (*, P, vocab) logits."""
        cache.check_prefill(x.reshape(-1, x.shape[-1]).shape[0], x.shape[-1])
        out_dtype = self.token_embs.weight.dtype
        h, stats = self.layers.prefill(embed_tokens(x, self.token_embs, self.pos_embs), cache)
        logits = self._logits(h, self.token_embs, self.norm, stats)
        logits = logits.reshape(*x.shape, logits.shape[-1])
        return logits if out_dtype == torch.bfloat16 else logits.to(out_dtype)

    def step(self, x: Tensor, cache: KVCache) -> Tensor:
        """The next token of every sequence, (B,) or (B, 1) ids at position ``cache.n`` -> (B, vocab) logits, equal
        to ``forward(prefix)[:, -1]`` within bf16 rounding. Appends to the cache."""
        cache.check_step(step_ids_batch(x))
        self.layers._check_decodable()
        out_dtype = self.token_embs.weight.dtype
        h, stats = self.layers.step(embed_tokens_at(x, self.token_embs, self.pos_embs, cache), cache)
        logits = self._logits(h, self.token_embs, self.norm, stats)[:, 0]
        return logits if out_dtype == torch.bfloat16 else logits.to(out_dtype)

    @staticmethod
    def from_hf(model_tag: str, *, pretrained: bool = False, **kwargs) -> "GPT2":
        """Sizes as gpt2.py:31-36; ``pretrained=True`` downloads the HuggingFace checkpoint (needs network)."""
        n_layers, d_model = {
            "gpt2": (12, 768),
            "gpt2-medium": (24, 1024),
            "gpt2-large": (36, 1280),
            "gpt2-xl": (48, 1600),
        }[model_tag]
        m = GPT2(n_layers, d_model, **kwargs)
        if pretrained:
            url = f"https://huggingface.co/{model_tag}/resolve/main/pytorch_model.bin"
            m.load_hf_state_dict(torch.hub.load_state_dict_from_url(url, file_name=model_tag))
        return m

    @torch.no_grad()
    def load_hf_state_dict(self, state_dict: dict) -> None:
        """HuggingFace GPT-2 checkpoint -> this layout (gpt2.py:48-99): Conv1D weights are stored (in, out) and are
        transposed; the fused ``c_attn`` splits into q/k/v."""
        sd = {k.removeprefix("transformer."): v for k, v in state_dict.items()}

        def take(module, key: str) -> None:
            w = sd.pop(f"{key}.weight")
            module.weight.copy_(w.T if w.ndim == 2 else w)
            if module.bias is not None:
                module.bias.copy_(sd.pop(f"{key}.bias"))

        tok = sd.pop("wte.weight")
        self.token_embs.weight[: tok.shape[0]] = tok
        self.pos_embs.copy_(sd.pop("wpe.weight"))
        for i, layer in enumerate(self.layers):
            pre = f"h.{i}"
            take(layer.sa_norm, f"{pre}.ln_1")
            take(layer.sa.out_proj, f"{pre}.attn.c_proj")
            wq, wk, wv = sd.pop(f"{pre}.attn.c_attn.weight").chunk(3, 1)
            bq, bk, bv = sd.pop(f"{pre}.attn.c_attn.bias").chunk(3, 0)
            for lin, w, b in ((layer.sa.q_proj, wq, bq), (layer.sa.k_proj, wk, bk), (layer.sa.v_proj, wv, bv)):
                lin.weight.copy_(w.T)
                lin.bias.copy_(b)
            take(layer.mlp_norm, f"{pre}.ln_2")
            take(layer.mlp.linear1, f"{pre}.mlp.c_fc")
            take(layer.mlp.linear2, f"{pre}.mlp.c_proj")
        take(self.norm, "ln_f")
