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
from ..transformer import Decoder, DecoderLM, TiedLogits, embed_tokens


@compilable_module
class GPT2(DecoderLM, nn.Module):
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
        h, stats = self.layers.run(embed_tokens(x, self.token_embs, self.pos_embs), final_stats=True)
        return self._logits_as(h, stats, x.shape)

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
