"""B200-native drop-in for ``GPT`` (reference ``pytorch_models/text/gpt.py:14-93``): post-norm causal ``Decoder`` with
tanh-GELU, no final LayerNorm, logits against the tied embedding table."""
from __future__ import annotations

import torch
from torch import Tensor, nn

from ..compile import compilable, compilable_module
from ..transformer import Decoder, DecoderLM, TiedLogits, embed_tokens


@compilable_module
class GPT(DecoderLM, nn.Module):
    vocab_size = 40478
    max_seq_len: int = 512

    def __init__(self, n_layers: int = 12, d_model: int = 768, dropout: float = 0.0) -> None:
        super().__init__()
        self.token_embs = nn.Embedding(self.vocab_size, d_model)
        self.pos_embs = nn.Parameter(torch.zeros(self.max_seq_len, d_model))
        self.layers = Decoder(n_layers, d_model, dropout=dropout, pre_norm=False, act="approximate_gelu")
        self._logits = TiedLogits()

    @compilable(lambda self, x, extra: ((*x.shape, self.token_embs.weight.shape[0]), self.token_embs.weight.dtype))
    def forward(self, x: Tensor) -> Tensor:
        """(*, L) int64 token ids -> (*, L, vocab) logits in the parameters' dtype (gpt.py:24-29)."""
        h = self.layers.run(embed_tokens(x, self.token_embs, self.pos_embs))
        return self._logits_as(h, None, x.shape)

    @staticmethod
    def from_openai(*, pretrained: bool = False, **kwargs) -> "GPT":
        m = GPT(**kwargs)
        if pretrained:
            m.load_openai_arrays(_download_openai_arrays())
        return m

    @torch.no_grad()
    def load_openai_arrays(self, params: list) -> None:
        """The flat parameter list of openai/finetune-transformer-lm (gpt.py:52-91): [pos, tok, then 12 arrays per
        layer: c_attn w/b, c_proj w/b, ln_1 g/b, c_fc w/b, c_proj w/b, ln_2 g/b]; weights are stored (1, in, out)."""
        t = [torch.as_tensor(p) for p in params]
        self.pos_embs.copy_(t[0])
        self.token_embs.weight[: t[1].shape[0]] = t[1]
        n = 12
        for i, layer in enumerate(self.layers):
            o = 2 + i * n
            wq, wk, wv = t[o].squeeze(0).chunk(3, -1)
            bq, bk, bv = t[o + 1].chunk(3, -1)
            for lin, w, b in ((layer.sa.q_proj, wq, bq), (layer.sa.k_proj, wk, bk), (layer.sa.v_proj, wv, bv)):
                lin.weight.copy_(w.T)
                lin.bias.copy_(b)
            layer.sa.out_proj.weight.copy_(t[o + 2].squeeze(0).T)
            layer.sa.out_proj.bias.copy_(t[o + 3])
            layer.sa_norm.weight.copy_(t[o + 4])
            layer.sa_norm.bias.copy_(t[o + 5])
            layer.mlp.linear1.weight.copy_(t[o + 6].squeeze(0).T)
            layer.mlp.linear1.bias.copy_(t[o + 7])
            layer.mlp.linear2.weight.copy_(t[o + 8].squeeze(0).T)
            layer.mlp.linear2.bias.copy_(t[o + 9])
            layer.mlp_norm.weight.copy_(t[o + 10])
            layer.mlp_norm.bias.copy_(t[o + 11])


def _download_openai_arrays() -> list:
    """Fetch and un-flatten the ten ``params_{i}.npy`` shards (gpt.py:36-50); needs network access."""
    import json
    import os

    import numpy as np
    import requests

    base = "https://github.com/openai/finetune-transformer-lm/raw/master/model"
    shapes = json.loads(requests.get(f"{base}/params_shapes.json").content)
    offsets = np.cumsum([np.prod(shape) for shape in shapes])
    cache = os.path.join(torch.hub.get_dir(), "openai_gpt")
    os.makedirs(cache, exist_ok=True)
    shards = []
    for i in range(10):
        path = os.path.join(cache, f"params_{i}.npy")
        if not os.path.exists(path):
            torch.hub.download_url_to_file(f"{base}/params_{i}.npy", path)
        shards.append(np.load(path))
    flat = np.split(np.concatenate(shards, axis=0), offsets)[:-1]
    return [p.reshape(shape) for p, shape in zip(flat, shapes)]
