"""Pretrained-weight converters on synthetic checkpoints (no network): random tensors in the checkpoint layouts go
through our converters, and the resulting state_dicts must be identical (keys, order, shapes, dtypes, bytes) to what
the reference's own loaders produce from the same checkpoints.

The reference's results are stored in tests/golden/weight_loading.json as one SHA-256 per tensor (the state_dicts
themselves are several MB). They were recorded from this project's converters at a revision where this same test
compared them, state_dict against state_dict, with the reference loaders (download helper monkey-patched to a local
file) and passed; no converter or checkpoint builder below has changed since. Re-record only after such a comparison.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np
import pytest
import torch

import pytorch_models_b200 as pm

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "weight_loading.json")) as _f:
    REFERENCE = json.load(_f)["state_dicts"]


def digest(module: torch.nn.Module) -> list[list]:
    """[key, shape, dtype, sha256 of the tensor's bytes] per state_dict entry, in state_dict order."""
    out = []
    for k, v in module.state_dict().items():
        raw = v.detach().cpu().contiguous().reshape(-1).view(torch.uint8).numpy().tobytes()
        out.append([k, list(v.shape), str(v.dtype).replace("torch.", ""), hashlib.sha256(raw).hexdigest()])
    return out


def _same(case: str, module: torch.nn.Module) -> None:
    got, want = digest(module), REFERENCE[case]
    assert [g[0] for g in got] == [w[0] for w in want]
    for g, w in zip(got, want):
        assert g == w, g[0]


def _flax_tree(n_layers, d, h, p, n_patches, big_vision, rng):
    r = lambda *s: rng.standard_normal(s).astype(np.float32)  # noqa: E731
    attn, ln2, mlp = (("MultiHeadDotProductAttention_0", "LayerNorm_1", "MlpBlock_0") if big_vision
                      else ("MultiHeadDotProductAttention_1", "LayerNorm_2", "MlpBlock_3"))
    t = {"embedding/kernel": r(p, p, 3, d), "embedding/bias": r(d),
         "Transformer/encoder_norm/scale": r(d), "Transformer/encoder_norm/bias": r(d)}
    if big_vision:
        t["pos_embedding"] = r(1, n_patches, d)
    else:
        t["cls"] = r(1, 1, d)
        t["Transformer/posembed_input/pos_embedding"] = r(1, n_patches + 1, d)

    def mha(prefix):
        for name in ("query", "key", "value"):
            t[f"{prefix}/{name}/kernel"] = r(d, h, d // h)
            t[f"{prefix}/{name}/bias"] = r(h, d // h)
        t[f"{prefix}/out/kernel"] = r(h, d // h, d)
        t[f"{prefix}/out/bias"] = r(d)

    def block_mlp(prefix):
        t[f"{prefix}/Dense_0/kernel"] = r(d, 4 * d)
        t[f"{prefix}/Dense_0/bias"] = r(4 * d)
        t[f"{prefix}/Dense_1/kernel"] = r(4 * d, d)
        t[f"{prefix}/Dense_1/bias"] = r(d)

    for i in range(n_layers):
        b = f"Transformer/encoderblock_{i}"
        for ln in ("LayerNorm_0", ln2):
            t[f"{b}/{ln}/scale"], t[f"{b}/{ln}/bias"] = r(d), r(d)
        mha(f"{b}/{attn}")
        block_mlp(f"{b}/{mlp}")
    if big_vision:
        t["MAPHead_0/probe"] = r(1, 1, d)
        mha("MAPHead_0/MultiHeadDotProductAttention_0")
        t["MAPHead_0/LayerNorm_0/scale"], t["MAPHead_0/LayerNorm_0/bias"] = r(d), r(d)
        block_mlp("MAPHead_0/MlpBlock_0")
    return t


@pytest.mark.parametrize("big_vision", [False, True])
def test_flax_checkpoint_loader_matches_reference(big_vision):
    kw = dict(cls_token=False, pool_type="mha") if big_vision else {}
    tree = _flax_tree(2, 128, 2, 16, 16, big_vision, np.random.default_rng(0))
    ours = pm.ViT(2, 128, 2, 16, img_size=64, **kw)
    ours.load_flax_arrays(tree, big_vision=big_vision)
    _same(f"flax_big_vision={big_vision}", ours)


@pytest.mark.parametrize("style", ["deit3", "dino", "dinov2"])
def test_facebook_state_dict_loader_matches_reference(style):
    g = torch.Generator().manual_seed(1)
    r = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    d, n, p = 128, 2, 16
    with_cls_pos = style != "deit3"  # dino / dinov2 checkpoints carry a position embedding for the class token
    sd = {"patch_embed.proj.weight": r(d, 3, p, p), "patch_embed.proj.bias": r(d), "cls_token": r(1, 1, d),
          "pos_embed": r(1, 16 + int(with_cls_pos), d), "norm.weight": r(d), "norm.bias": r(d)}
    for i in range(n):
        b = f"blocks.{i}"
        sd.update({f"{b}.norm1.weight": r(d), f"{b}.norm1.bias": r(d), f"{b}.norm2.weight": r(d), f"{b}.norm2.bias": r(d),
                   f"{b}.attn.qkv.weight": r(3 * d, d), f"{b}.attn.qkv.bias": r(3 * d),
                   f"{b}.attn.proj.weight": r(d, d), f"{b}.attn.proj.bias": r(d),
                   f"{b}.mlp.fc1.weight": r(4 * d, d), f"{b}.mlp.fc1.bias": r(4 * d),
                   f"{b}.mlp.fc2.weight": r(d, 4 * d), f"{b}.mlp.fc2.bias": r(d)})
        if style == "deit3":
            sd.update({f"{b}.gamma_1": r(d), f"{b}.gamma_2": r(d)})
        if style == "dinov2":
            sd.update({f"{b}.ls1.gamma": r(d), f"{b}.ls2.gamma": r(d)})
    ours = pm.ViT(n, d, 2, p, img_size=64)
    ours.load_facebook_state_dict(sd)
    _same(f"facebook_{style}", ours)
    # the in-place LayerScale fold must invalidate the packed-weight cache of the kernels
    layer = ours.layers[0]
    before = layer.sa._pack("out", [layer.sa.out_proj])
    ours.load_facebook_state_dict(sd)
    assert layer.sa._pack("out", [layer.sa.out_proj]) is not before


@pytest.mark.parametrize("roberta", [False, True])
def test_hf_bert_loader_matches_reference(roberta):
    g = torch.Generator().manual_seed(2)
    r = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    d, n, vocab, max_len = 128, 2, 1000, 40
    pfx = "roberta." if roberta else "bert."
    sd = {f"{pfx}embeddings.word_embeddings.weight": r(vocab, d),
          f"{pfx}embeddings.position_embeddings.weight": r(max_len + (2 if roberta else 0), d),
          f"{pfx}embeddings.token_type_embeddings.weight": r(2, d),
          f"{pfx}embeddings.LayerNorm.weight": r(d), f"{pfx}embeddings.LayerNorm.bias": r(d)}
    for i in range(n):
        b = f"{pfx}encoder.layer.{i}"
        for name, (o, k) in {"attention.self.query": (d, d), "attention.self.key": (d, d), "attention.self.value": (d, d),
                             "attention.output.dense": (d, d), "intermediate.dense": (4 * d, d),
                             "output.dense": (d, 4 * d)}.items():
            sd[f"{b}.{name}.weight"], sd[f"{b}.{name}.bias"] = r(o, k), r(o)
        for name in ("attention.output.LayerNorm", "output.LayerNorm"):
            sd[f"{b}.{name}.weight"], sd[f"{b}.{name}.bias"] = r(d), r(d)
    torch.manual_seed(0)  # parameters the checkpoint does not carry keep the seeded init of both constructors
    ours = pm.BERT(vocab, n, d, max_len)
    with torch.no_grad():
        ours.load_hf_state_dict(dict(sd))
    _same(f"hf_bert_roberta={roberta}", ours)


def test_openai_whisper_encoder_loader_matches_reference():
    g = torch.Generator().manual_seed(3)
    sd = {}
    r = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    d = 128
    for side, n_ctx in (("encoder", 1500), ("decoder", 448)):
        sd[f"{side}.positional_embedding"] = r(n_ctx, d)
        for i in range(2):
            b = f"{side}.blocks.{i}"
            attns = ["attn"] + (["cross_attn"] if side == "decoder" else [])
            for a in attns:
                for name in ("query", "key", "value", "out"):
                    sd[f"{b}.{a}.{name}.weight"] = r(d, d)
                    if name != "key":
                        sd[f"{b}.{a}.{name}.bias"] = r(d)
                sd[f"{b}.{a}_ln.weight"], sd[f"{b}.{a}_ln.bias"] = r(d), r(d)
            sd[f"{b}.mlp.0.weight"], sd[f"{b}.mlp.0.bias"] = r(4 * d, d), r(4 * d)
            sd[f"{b}.mlp.2.weight"], sd[f"{b}.mlp.2.bias"] = r(d, 4 * d), r(d)
            sd[f"{b}.mlp_ln.weight"], sd[f"{b}.mlp_ln.bias"] = r(d), r(d)
    sd.update({"encoder.conv1.weight": r(d, 80, 3), "encoder.conv1.bias": r(d), "encoder.conv2.weight": r(d, d, 3),
               "encoder.conv2.bias": r(d), "encoder.ln_post.weight": r(d), "encoder.ln_post.bias": r(d),
               "decoder.token_embedding.weight": r(300, d), "decoder.ln.weight": r(d), "decoder.ln.bias": r(d)})
    ours = pm.WhisperEncoder(2, 128, 80)
    ours.load_openai_state_dict(sd)
    _same("openai_whisper_encoder", ours)
    # the full model (encoder + decoder with cross-attention)
    full = pm.Whisper(300, 2, 128, 80)
    full.load_openai_state_dict(sd)
    _same("openai_whisper", full)


def test_hf_gpt2_loader_matches_reference():
    g = torch.Generator().manual_seed(4)
    r = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    d, n_layers, vocab = 64, 2, 211
    sd = {"transformer.wte.weight": r(vocab, d), "transformer.wpe.weight": r(1024, d),
          "transformer.ln_f.weight": r(d), "transformer.ln_f.bias": r(d)}
    for i in range(n_layers):
        b = f"transformer.h.{i}"
        sd.update({f"{b}.ln_1.weight": r(d), f"{b}.ln_1.bias": r(d), f"{b}.ln_2.weight": r(d), f"{b}.ln_2.bias": r(d),
                   f"{b}.attn.c_attn.weight": r(d, 3 * d), f"{b}.attn.c_attn.bias": r(3 * d),
                   f"{b}.attn.c_proj.weight": r(d, d), f"{b}.attn.c_proj.bias": r(d),
                   f"{b}.mlp.c_fc.weight": r(d, 4 * d), f"{b}.mlp.c_fc.bias": r(4 * d),
                   f"{b}.mlp.c_proj.weight": r(4 * d, d), f"{b}.mlp.c_proj.bias": r(d)})
    torch.manual_seed(0)  # parameters the checkpoint does not carry keep the seeded init of both constructors
    ours = type("OS", (pm.GPT2,), dict(vocab_size=vocab))(n_layers, d)
    ours.load_hf_state_dict(dict(sd))
    _same("hf_gpt2", ours)


def test_openai_gpt_array_loader_matches_reference():
    """The reference inlines this conversion in GPT.from_openai (gpt.py:52-91, behind a download); restated here on
    the same flat parameter list."""
    rng = np.random.default_rng(5)
    d, n_layers, vocab, ctx = 64, 2, 97, 512
    r = lambda *s: rng.standard_normal(s).astype(np.float32)  # noqa: E731
    params = [r(ctx, d), r(vocab, d)]
    for _ in range(n_layers):
        params += [r(1, d, 3 * d), r(3 * d), r(1, d, d), r(d), r(d), r(d), r(1, d, 4 * d), r(4 * d), r(1, 4 * d, d),
                   r(d), r(d), r(d)]
    ours = type("OS", (pm.GPT,), dict(vocab_size=vocab))(n_layers, d)
    ours.load_openai_arrays(params)
    t = [torch.from_numpy(p) for p in params]
    sd = ours.state_dict()
    assert torch.equal(sd["pos_embs"], t[0]) and torch.equal(sd["token_embs.weight"], t[1])
    for i in range(n_layers):
        o = 2 + 12 * i
        wq, wk, wv = t[o].squeeze(0).chunk(3, -1)
        assert torch.equal(sd[f"layers.{i}.sa.q_proj.weight"], wq.T)
        assert torch.equal(sd[f"layers.{i}.sa.k_proj.weight"], wk.T)
        assert torch.equal(sd[f"layers.{i}.sa.v_proj.bias"], t[o + 1].chunk(3, -1)[2])
        assert torch.equal(sd[f"layers.{i}.sa.out_proj.weight"], t[o + 2].squeeze(0).T)
        assert torch.equal(sd[f"layers.{i}.sa_norm.weight"], t[o + 4])
        assert torch.equal(sd[f"layers.{i}.mlp.linear1.weight"], t[o + 6].squeeze(0).T)
        assert torch.equal(sd[f"layers.{i}.mlp.linear2.bias"], t[o + 9])
        assert torch.equal(sd[f"layers.{i}.mlp_norm.bias"], t[o + 11])
