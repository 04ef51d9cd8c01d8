"""B200-native drop-in for ``WhisperEncoder`` / ``WhisperDecoder`` / ``Whisper`` (reference
``pytorch_models/audio2text/whisper.py:11-135``).

Same constructor, ``state_dict`` keys (``stem.0/2``, ``pos_embs`` buffer, ``layers.*``, ``norm``) and call signature.
The conv stem runs as two GEMMs on the same tcgen05 kernel as the linears: the log-mel input is rewritten once as
zero-padded time-major rows, after which a k=3 convolution over time is a GEMM over an *overlapping* strided view
(row t starts at element stride·t·C and is 3·C long), with GELU — and for the second conv the positional embedding —
fused into the epilogue (whisper.py:16-21,30-31).

The decoder is one gather kernel (token + position embedding), the ``Decoder`` stack with causal self-attention and
cross-attention to the encoder output, and one GEMM against the tied token table with the final LayerNorm folded in.
"""
from __future__ import annotations

import math
from types import SimpleNamespace

import torch
from torch import Tensor, nn

from .. import ops, plans
from ..compile import compilable, compilable_module, float_like
from ..transformer import (Decoder, DecoderLM, Encoder, KVCache, TiedLogits, _as_tokens, _Packed, embed_tokens,
                           norm_vectors)


@compilable_module
class WhisperEncoder(nn.Module):
    max_seq_len = 3000

    def __init__(self, n_layers: int, d_model: int, n_mels: int = 80, dropout: float = 0.0) -> None:
        super().__init__()
        # parameter containers with the reference's layout; the arithmetic does not go through nn.Conv1d.forward
        self.stem = nn.Sequential(
            nn.Conv1d(n_mels, d_model, 3, 1, 1),
            nn.GELU(),
            nn.Conv1d(d_model, d_model, 3, 2, 1),
            nn.GELU(),
        )
        self.register_buffer("pos_embs", torch.zeros(self.max_seq_len // 2, d_model))
        self.pos_embs: Tensor
        self.layers = Encoder(n_layers, d_model, dropout=dropout)
        self.norm = nn.LayerNorm(d_model)
        self._pstem = _Packed()

    def _pack_stem(self) -> SimpleNamespace:
        c1, c2 = self.stem[0], self.stem[2]

        def conv_as_linear(conv: nn.Conv1d) -> tuple[Tensor, Tensor]:
            # w[n][k*C + c] = weight[n][c][k]: matches rows that concatenate time steps t-1, t, t+1
            w = conv.weight.detach().permute(0, 2, 1).reshape(conv.out_channels, -1).to(torch.bfloat16).contiguous()
            b = (conv.bias.detach().float() if conv.bias is not None
                 else torch.zeros(conv.out_channels, device=w.device)).contiguous()
            return w, b

        def build() -> SimpleNamespace:
            w1, b1 = conv_as_linear(c1)
            w2, b2 = conv_as_linear(c2)
            return SimpleNamespace(w1=w1, b1=b1, w2=w2, b2=b2, pos=self.pos_embs.detach().to(torch.bfloat16).contiguous())

        return self._pstem.get((c1.weight, c1.bias, c2.weight, c2.bias, self.pos_embs), build)

    def embed(self, x: Tensor, with_stats: bool = False):
        """(N, n_mels, T) log-mel -> contiguous bf16 tokens (N, ceil(T/2), d) incl. positional embedding.
        ``with_stats``: also return the rows' partial LayerNorm statistics from the second conv GEMM's epilogue."""
        if not x.is_cuda:
            raise RuntimeError("pytorch_models_b200 runs only on CUDA (sm_100a) tensors; there is no CPU fallback")
        if x.dtype not in (torch.bfloat16, torch.float32):
            x = x.float()
        x = x.contiguous()
        N, C, T = x.shape
        d = self.stem[0].out_channels
        if C % 8 != 0:
            raise NotImplementedError(f"n_mels={C} must be a multiple of 8 for 16-byte aligned rows")
        T2 = (T + 2 - 3) // 2 + 1  # Conv1d(k=3, stride=2, pad=1) output length
        if T2 > self.pos_embs.shape[0]:
            raise ValueError(f"{T} frames give {T2} tokens but pos_embs has {self.pos_embs.shape[0]} rows")
        pk = self._pack_stem()
        dev = x.device
        rows = torch.empty(N, T + 2, C, device=dev, dtype=torch.bfloat16)
        ops.time_rows(x, rows)
        # conv1 (stride 1): output step t reads rows[t : t+3]; written at rows 1..T of a zero-padded buffer
        h1 = torch.empty(N, T + 3, d, device=dev, dtype=torch.bfloat16)
        h1[:, 0].zero_()
        h1[:, T + 1:].zero_()
        a1 = rows.as_strided((N, T, 3 * C), ((T + 2) * C, C, 1))
        ops.linear(a1, pk.w1, pk.b1, h1[:, 1:T + 1, :], gelu=True)
        # conv2 (stride 2): output step t reads h1 rows[2t : 2t+3]  (= time steps 2t-1, 2t, 2t+1)
        a2 = h1.as_strided((N, T2, 3 * d), ((T + 3) * d, 2 * d, 1))
        tokens = torch.empty(N, T2, d, device=dev, dtype=torch.bfloat16)
        stats = None
        if with_stats and self.layers.wants_stats():
            stats = torch.empty(N * T2, (d + 127) // 128, 2, device=dev, dtype=torch.float32)
        ops.linear(a2, pk.w2, pk.b2, tokens, gelu=True, residual=pk.pos[:T2].unsqueeze(0), stats_out=stats)
        return (tokens, stats) if with_stats else tokens

    @compilable(lambda self, x, extra: ((x.shape[0], (x.shape[2] - 1) // 2 + 1, self.stem[0].out_channels), float_like(x)))
    def forward(self, x: Tensor) -> Tensor:
        out_dtype = x.dtype if x.dtype in (torch.bfloat16, torch.float32) else torch.float32
        if x.is_cuda and x.numel():
            if x.dtype not in (torch.bfloat16, torch.float32):
                x = x.float()
            # recorded once per (shape, dtype, stream, weights), then replayed by one C-ABI call (plans.py)
            out = plans.run(self, (x.contiguous(),), self._forward_launches)
        else:
            out = self._forward_launches(x)
        return out if out_dtype == torch.bfloat16 else out.to(out_dtype)

    def _forward_launches(self, x: Tensor) -> Tensor:
        """log-mel (N, n_mels, T) -> bf16 (N, ceil(T/2), d): libb200enc launches only (the two `zero_` calls of `embed`
        initialise padding rows that no kernel writes, so a replayed plan finds them as recorded)."""
        tokens, stats = self.embed(x, with_stats=True)
        h = self.layers.run(tokens, stats)
        N, L, d = h.shape
        gamma, beta = norm_vectors(self.norm)
        out = torch.empty_like(h)
        ops.layernorm(h.view(N * L, d), gamma, beta, self.norm.eps, out.view(N * L, d))
        return out

    @torch.no_grad()
    def load_openai_state_dict(self, state_dict: dict) -> None:
        """Encoder half of an openai-whisper checkpoint (``model_state_dict``), cf. whisper.py:97-135."""
        _load_openai(self, state_dict, "encoder")


def _load_openai(half: nn.Module, state_dict: dict, prefix: str) -> None:
    """Copy the ``encoder.*`` or ``decoder.*`` entries of an openai-whisper ``model_state_dict`` into ``half``
    (whisper.py:97-132). The key projections have no bias in the checkpoint: their bias is set to zero."""
    sd = {k[len(prefix) + 1:]: v for k, v in state_dict.items() if k.startswith(prefix + ".")}

    def take(module, key: str) -> None:
        module.weight.copy_(sd.pop(f"{key}.weight"))
        if module.bias is not None:
            module.bias.copy_(sd.pop(f"{key}.bias", 0))

    if prefix == "encoder":
        take(half.stem[0], "conv1")
        take(half.stem[2], "conv2")
    else:
        half.token_embs.weight.copy_(sd.pop("token_embedding.weight"))
    half.pos_embs.copy_(sd.pop("positional_embedding"))
    for i, layer in enumerate(half.layers):
        pre = f"blocks.{i}"
        for mha, norm, name in ((layer.sa, layer.sa_norm, "attn"), (layer.ca, layer.ca_norm, "cross_attn")):
            if mha is None:
                continue
            take(mha.q_proj, f"{pre}.{name}.query")
            take(mha.k_proj, f"{pre}.{name}.key")
            take(mha.v_proj, f"{pre}.{name}.value")
            take(mha.out_proj, f"{pre}.{name}.out")
            take(norm, f"{pre}.{name}_ln")
        take(layer.mlp.linear1, f"{pre}.mlp.0")
        take(layer.mlp.linear2, f"{pre}.mlp.2")
        take(layer.mlp_norm, f"{pre}.mlp_ln")
    take(half.norm, "ln_post" if prefix == "encoder" else "ln")


@compilable_module
class WhisperDecoder(DecoderLM, nn.Module):
    """Reference ``WhisperDecoder`` (whisper.py:37-53)."""

    max_seq_len = 448

    def __init__(self, vocab_size: int, n_layers: int, d_model: int, dropout: float = 0.0) -> None:
        super().__init__()
        self.token_embs = nn.Embedding(vocab_size, d_model)
        self.pos_embs = nn.Parameter(torch.zeros(self.max_seq_len, d_model))
        self.layers = Decoder(n_layers, d_model, cross_attn=True, dropout=dropout)
        self.norm = nn.LayerNorm(d_model)
        self._logits = TiedLogits()

    @compilable(lambda self, x, extra: ((*x.shape, self.token_embs.weight.shape[0]), self.token_embs.weight.dtype))
    def forward(self, x: Tensor, memory: Tensor) -> Tensor:
        """x: (N, L) int64 token ids, memory: (N, Lm, d) encoder output -> (N, L, vocab) logits (whisper.py:46-52)."""
        m3, _ = _as_tokens(memory, self.token_embs.weight.shape[1])
        h, stats = self.layers.run(embed_tokens(x, self.token_embs, self.pos_embs), m3, final_stats=True)
        return self._logits_as(h, stats, x.shape)

    def new_kv_cache(self, memory: Tensor, capacity: int) -> KVCache:
        """An empty KV cache for the (N, Lm, d) encoder output ``memory`` and up to ``capacity`` <= max_seq_len tokens.
        Every layer's cross-attention [k; v] projection of the memory runs here, once."""
        self._check_capacity(capacity)
        if memory.dim() != 3:
            raise ValueError(f"memory must be (N, Lm, d), got {tuple(memory.shape)}")
        return self.layers.new_kv_cache(memory.shape[0], capacity, memory)


_OPENAI_SIZES = {
    # tag: (n_layers, d_model, checkpoint hash) — whisper.py:66-78
    "tiny": (4, 384, "65147644a518d12f04e32d6f3b26facc3f8dd46e5390956a9424a650c0ce22b9"),
    "tiny.en": (4, 384, "d3dd57d32accea0b295c96e26691aa14d8822fac7d9d27d5dc00b4ca2826dd03"),
    "base": (8, 512, "ed3a0b6b1c0edf879ad9b11b1af5a0e6ab5db9205f891f668f8b0e6c6326e34e"),
    "base.en": (8, 512, "25a8566e1d0c1e2231d1c762132cd20e0f96a85d16145c3a00adf5d1ac670ead"),
    "small": (12, 768, "9ecf779972d90ba49c06d968637d720dd632c55bbf19d441fb42bf17a411e794"),
    "small.en": (12, 768, "f953ad0fd29cacd07d5a9eda5624af0f6bcf2258be67c92b79389873d91e0872"),
    "medium": (24, 1024, "345ae4da62f9b3d59415adc60127b97c714f32e89e936602e85993674d08dcb1"),
    "medium.en": (24, 1024, "d7440d1dc186f76616474e0ff0b3b6b879abc9d1a4926b7adfa41db2d497ab4f"),
    "large-v1": (32, 1280, "e4b87e7e0bf463eb8e6956e646f1e277e901512310def2c24bf0e11bd3c28e9a"),
    "large-v2": (32, 1280, "81f7c96c852ee8fc832187b0132e569d6c3065a3252ed18e56effd0b6a73e524"),
    "large-v3": (32, 1280, "e5b1a55b89c1367dacf97e3e19bfd829a01529dbfdeefa8caeb59b3f1b81dadb"),
}


@compilable_module
class Whisper(nn.Module):
    """Reference ``Whisper`` (whisper.py:56-135): ``decoder(targets, encoder(x))``."""

    def __init__(self, vocab_size: int, n_layers: int, d_model: int, n_mels: int = 80, dropout: float = 0.0) -> None:
        super().__init__()
        self.encoder = WhisperEncoder(n_layers, d_model, n_mels, dropout=dropout)
        self.decoder = WhisperDecoder(vocab_size, n_layers, d_model, dropout=dropout)

    @compilable(lambda self, x, extra: ((*extra.shape, self.decoder.token_embs.weight.shape[0]),
                                        self.decoder.token_embs.weight.dtype))
    def forward(self, x: Tensor, targets: Tensor) -> Tensor:
        return self.decoder(targets, self.encoder(x))

    @staticmethod
    def from_openai(model_tag: str, *, pretrained: bool = False, **kwargs) -> "Whisper":
        n_layers, d_model, ckpt_hash = _OPENAI_SIZES[model_tag]
        if model_tag == "large-v3":
            n_mels, vocab_size = 128, 51866
        else:
            n_mels, vocab_size = 80, 51864 if model_tag.endswith(".en") else 51865
        m = Whisper(vocab_size, n_layers, d_model, n_mels, **kwargs)
        if pretrained:  # needs network access
            url = f"https://openaipublic.azureedge.net/main/whisper/models/{ckpt_hash}/{model_tag}.pt"
            sd = torch.hub.load_state_dict_from_url(url, file_name=f"whisper_{model_tag}")["model_state_dict"]
            m.load_openai_state_dict(sd)
        return m

    @torch.no_grad()
    def load_openai_state_dict(self, state_dict: dict) -> None:
        _load_openai(self.encoder, state_dict, "encoder")
        _load_openai(self.decoder, state_dict, "decoder")


def mel_filters(n_mels: int, n_fft: int, sample_rate: float) -> Tensor:
    """Triangular Slaney-style mel filter bank, (n_mels, n_fft // 2 + 1), area-normalised — the same definition as the
    reference's ``get_mel_filters`` (audio/spectrogram.py:19-36): linear below 1 kHz (200/3 Hz per mel), logarithmic
    above (step 6.4^(1/27))."""
    f_max = sample_rate / 2
    mel_max = f_max * 3 / 200 if f_max < 1000 else 15 + 27 * math.log(f_max / 1000, 6.4)
    mels = torch.linspace(0, mel_max, n_mels + 2)
    hz = torch.where(mels < 15, mels * 200 / 3, 1000 * 6.4 ** ((mels - 15) / 27))
    fft_hz = torch.linspace(0, sample_rate / 2, n_fft // 2 + 1)
    width = hz.diff()
    ramp = hz.unsqueeze(1) - fft_hz.unsqueeze(0)
    rising = -ramp[:-2] / width[:-1, None]
    falling = ramp[2:] / width[1:, None]
    bank = rising.minimum(falling).clamp(0)
    bank *= 2 / (hz[2:, None] - hz[:-2, None])
    return bank


@compilable_module
class WhisperPreprocessor(nn.Module):
    """Reference ``WhisperPreprocessor`` (whisper.py:138-148): raw 16 kHz audio (N, L) -> normalised log-mel
    (N, n_mels, L // 160). Same buffers as the reference (``window`` non-persistent, ``filters`` persistent); the
    STFT, mel projection, log and dynamic-range normalisation run in one sm_100a kernel (fp32)."""

    def __init__(self, variant: str = "tiny") -> None:
        super().__init__()
        n_mels = 128 if variant == "large-v3" else 80
        self.n_fft, self.hop_length = 400, 160
        self.register_buffer("window", torch.hann_window(self.n_fft), False)
        self.register_buffer("filters", mel_filters(n_mels, self.n_fft, 16_000))
        self._pf = _Packed()

    @compilable(lambda self, x, extra: ((*x.shape[:-1], self.filters.shape[0], x.shape[-1] // 160), x.dtype))
    def forward(self, x: Tensor) -> Tensor:
        if not x.is_cuda:
            raise RuntimeError("pytorch_models_b200 runs only on CUDA (sm_100a) tensors; there is no CPU fallback")
        lead = x.shape[:-1]
        L = x.shape[-1]
        a = x.reshape(-1, L).float().contiguous()
        ft = self._pf.get((self.filters,), lambda: SimpleNamespace(t=self.filters.detach().float().t().contiguous())).t
        out = torch.empty(a.shape[0], ft.shape[1], L // self.hop_length, device=x.device, dtype=torch.float32)
        ops.whisper_logmel(a, ft, out)
        out = out.reshape(*lead, ft.shape[1], out.shape[-1])
        return out if x.dtype == torch.float32 else out.to(x.dtype)
