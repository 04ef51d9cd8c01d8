"""CPU-side tests: module API / state_dict parity with the reference (recorded in tests/golden), packing logic,
argument validation, and that the C-ABI library loads and exports every symbol declared in include/b200enc.h."""
from __future__ import annotations

import ctypes
import os
import re

import numpy as np
import pytest
import torch

import pytorch_models_b200 as pm
from conftest import FIXTURES, ROOT, build_model
from pytorch_models_b200 import _lib
from pytorch_models_b200.transformer import pack_folded, pack_plain


@pytest.mark.parametrize("name", FIXTURES)
def test_state_dict_layout_matches_reference(golden, name):
    """Same keys, order, shapes and dtypes as the reference module that produced the fixture (strict load)."""
    g = golden(name)
    m = build_model(g)  # strict load_state_dict inside
    ours = m.state_dict()
    assert list(ours.keys()) == list(g.sd.keys())
    for k, v in g.sd.items():
        assert tuple(ours[k].shape) == v.shape and ours[k].numpy().dtype == v.dtype, k


def test_seeded_construction_reproduces_reference_weights(golden):
    """Parameters are created in the reference's order, so torch.manual_seed reproduces its random init exactly
    (this is what lets the C1 fixture store seeds instead of 22 MB of weights)."""
    g = golden("vit_cls")
    h = {k: v for k, v in g.hyper.items() if k != "kind"}
    torch.manual_seed(1)
    m = pm.ViT(**h)
    for k in ("patch_embed.weight", "layers.1.sa.v_proj.weight", "layers.0.mlp.linear2.bias"):
        np.testing.assert_array_equal(m.state_dict()[k].numpy(), g.sd[k])


def test_constructors_and_tags():
    m = pm.ViT.from_google("Ti/16")
    assert len(m.layers) == 12 and m.pe.shape == (1, 196, 192) and m.cls_token.shape == (1, 1, 192)
    assert len(m.state_dict()) == 198  # SURVEY §8(b)
    s = pm.ViT.from_google("B/16_siglip", img_size=256)
    assert s.cls_token is None and s.pe.shape == (1, 256, 768) and "pooler.probe" in s.state_dict()
    d = pm.ViT.from_facebook("S/14_dinov2")
    assert d.pe.shape == (1, 37 * 37, 384) and d.patch_embed.weight.shape == (384, 3, 14, 14)
    assert pm.ViT.from_facebook("B/16").pe.shape == (1, 196, 768)  # deit3 default, 224 px
    with pytest.raises(KeyError):
        pm.ViT.from_google("XL/16")
    with pytest.raises(ValueError):
        pm.ViT.from_facebook("B/16_mae")
    with pytest.raises(AssertionError):
        pm.ViT(1, 64, 1, 16, img_size=100)
    w = pm.WhisperEncoder(2, 128, 80)
    assert w.pos_embs.shape == (1500, 128) and "pos_embs" in w.state_dict() and "pos_embs" not in dict(w.named_parameters())
    b = pm.BERT(1000, 2, 128)
    assert b.token_embs.weight.shape == (1024, 128) and not b.layers[0].pre_norm and b.layers[0].sa_norm.eps == 1e-12
    enc = pm.Encoder(3, 256, n_heads=4)
    assert len(enc) == 3 and enc[0].sa.head_dim == 64 and enc[0].mlp[0] is enc[0].mlp.linear1 and enc[0].mlp[2] is enc[0].mlp.linear2
    assert pm.MHA(192).n_heads == 3 and pm.MHA(512, head_dim=32).n_heads == 16 and pm.MHA(512, n_heads=4).head_dim == 128


def test_resize_pe_shapes():
    m = pm.ViT.from_google("Ti/16")
    torch.nn.init.normal_(m.pe)
    m.resize_pe(256)  # tests/image/test_vit.py:21-26
    assert m.pe.shape == (1, 256, 192) and isinstance(m.pe, torch.nn.Parameter)
    m.resize_pe(224, "bilinear")
    assert m.pe.shape == (1, 196, 192)


def test_no_cpu_fallback():
    m = pm.ViT.from_google("Ti/16").eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 3, 224, 224))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.Encoder(1, 64)(torch.randn(1, 4, 64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.WhisperEncoder(1, 64)(torch.randn(1, 80, 16))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.BERT(100, 1, 64)(torch.randint(0, 100, (1, 8)))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.MHA(128).eval()(torch.randn(1, 4, 128), causal=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.MLP(128, 256, act="approximate_gelu").eval()(torch.randn(1, 4, 128))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.Decoder(1, 64, cross_attn=True)(torch.randn(1, 4, 64), torch.randn(1, 6, 64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.GPT2(1, 64)(torch.randint(0, 100, (1, 8)))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pm.Whisper(100, 1, 64)(torch.randn(1, 80, 16), torch.randint(0, 100, (1, 4)))


def test_unsupported_arguments_raise_not_implemented():
    x = torch.randn(1, 4, 128)
    mha = pm.MHA(128).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mha(x, attn_bias=torch.zeros(4, 4))
    with pytest.raises(NotImplementedError):
        pm.MHA(128, head_dim=32).eval()(x)
    with pytest.raises(NotImplementedError):
        pm.MHA(128, dropout=0.1).train()(x)
    for act in ("relu", "silu"):  # every activation of the reference is fused now: only the device check is left
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            pm.MLP(128, 256, act=act).eval()(x)
    with pytest.raises(NotImplementedError):
        pm.EncoderLayer(128, dropout=0.1).train().run(x, x, None)
    with pytest.raises(KeyError):
        pm.MLP(128, 256, act="tanh")


def test_layernorm_fold_identity_and_cache_invalidation():
    """pack_folded reproduces LN(x) W^T + b from raw x and (mean, rstd); the cache follows in-place edits."""
    torch.manual_seed(0)
    d, n = 64, 96
    lin, norm = torch.nn.Linear(d, n), torch.nn.LayerNorm(d, 1e-6)
    torch.nn.init.normal_(norm.weight, 1.0, 0.2)
    torch.nn.init.normal_(norm.bias, 0.0, 0.2)
    x = torch.randn(10, d) * 2 + 0.5
    pk = pack_folded([lin], norm)
    mean, var = x.mean(1, keepdim=True), x.var(1, unbiased=False, keepdim=True)
    rstd = (var + 1e-6).rsqrt()
    folded = rstd * (x @ pk.w.float().T - mean * pk.colsum[None]) + pk.bias
    torch.testing.assert_close(folded, lin(norm(x)), atol=2e-2, rtol=2e-2)  # bf16-rounded W'
    exact = rstd * (x @ (lin.weight * norm.weight).T - mean * (lin.weight * norm.weight).sum(1)[None]) + pk.bias
    torch.testing.assert_close(exact, lin(norm(x)), atol=1e-4, rtol=1e-4)
    assert pack_plain([lin, lin]).w.shape == (2 * n, d)

    layer = pm.EncoderLayer(64)
    a = layer._pack_qkv()
    assert layer._pack_qkv() is a
    with torch.no_grad():
        layer.sa.k_proj.weight.mul_(2.0)
    b = layer._pack_qkv()
    assert b is not a and not torch.equal(a.w, b.w)
    with torch.no_grad():
        layer.sa_norm.bias.add_(1.0)
    assert layer._pack_qkv() is not b
    layer.sa.q_proj.weight = torch.nn.Parameter(layer.sa.q_proj.weight.detach().clone())
    assert layer._pack_qkv() is not b


def _declared_symbols() -> list[str]:
    text = open(os.path.join(ROOT, "include", "b200enc.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200enc_[a-z_0-9]+)\s*\(", text)))


def test_cabi_library_exports_every_declared_symbol():
    """No compute here (no GPU): the library must load and export exactly what include/b200enc.h declares."""
    declared = _declared_symbols()
    assert declared, "header declares nothing?"
    assert set(declared) == set(_lib.EXPORTED_SYMBOLS)
    assert os.path.exists(_lib.LIB_PATH), "libb200enc.so is not built: run __graft_entry__.build()"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} not exported"
    assert _lib.load().b200enc_version() == 100
    assert isinstance(_lib.load().b200enc_last_error(), bytes)


def test_product_never_imports_the_oracle():
    """The CUDA path must not route through oracle/ (only tests, smoke() and bench.py's CPU arm may)."""
    pkg = os.path.join(ROOT, "pytorch_models_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports the oracle"


def test_tied_logits_pack_folds_final_norm_and_pads_vocabulary():
    """TiedLogits: norm(x) @ E^T as rstd*(x W'^T - mean*s) + c with the table padded to a multiple of 8 rows
    (gpt2.py:25-26, whisper.py:50-51); the cache follows in-place edits of the embedding table."""
    from pytorch_models_b200.transformer import TiedLogits

    torch.manual_seed(0)
    V, d = 101, 64
    emb, norm = torch.nn.Embedding(V, d), torch.nn.LayerNorm(d)
    torch.nn.init.normal_(norm.weight, 1.0, 0.2)
    torch.nn.init.normal_(norm.bias, 0.0, 0.2)
    tl = TiedLogits()
    pk = tl._pack(emb, norm)
    assert pk.w.shape == (104, d) and pk.V == V and pk.w.dtype == torch.bfloat16
    assert not pk.w[V:].any() and not pk.bias[V:].any() and not pk.colsum[V:].any()
    x = torch.randn(7, d) * 1.5 + 0.3
    mean, var = x.mean(1, keepdim=True), x.var(1, unbiased=False, keepdim=True)
    rstd = (var + norm.eps).rsqrt()
    got = rstd * (x @ pk.w.float().T - mean * pk.colsum[None]) + pk.bias
    want = norm(x) @ emb.weight.T
    torch.testing.assert_close(got[:, :V], want, atol=5e-2, rtol=2e-2)  # bf16-rounded table
    assert tl._pack(emb, norm) is pk
    with torch.no_grad():
        emb.weight.mul_(2.0)
    assert tl._pack(emb, norm) is not pk
    plain = TiedLogits()._pack(emb, None)
    assert plain.bias is None and plain.colsum is None and plain.w.shape == (104, d)


def test_decoder_modules_mirror_reference_structure():
    """DecoderLayer / Decoder keep the reference's attribute names, child order and call signatures
    (transformer.py:70-105,152-176); EncoderLayer derives from DecoderLayer as in the reference (:108)."""
    layer = pm.DecoderLayer(128, cross_attn=True)
    assert [n for n, _ in layer.named_children()] == ["sa_norm", "sa", "ca_norm", "ca", "mlp_norm", "mlp"]
    assert pm.DecoderLayer(128).ca is None and pm.DecoderLayer(128).ca_norm is None
    assert issubclass(pm.EncoderLayer, pm.DecoderLayer)
    dec = pm.Decoder(3, 128, cross_attn=True, pre_norm=False)
    assert isinstance(dec, torch.nn.ModuleList) and len(dec) == 3 and not dec[0].pre_norm
    assert len(dec.state_dict()) == 3 * (2 * 3 + 8 * 2 + 4)
    assert pm.GPT2.vocab_size == 50257 and pm.GPT2.max_seq_len == 1024 and pm.GPT.vocab_size == 40478
    assert pm.WhisperDecoder.max_seq_len == 448
    m = pm.Whisper.from_openai("tiny")
    assert m.decoder.token_embs.weight.shape == (51865, 384) and len(m.decoder.layers) == 4


def test_whisper_preprocessor_mirrors_reference_buffers(golden):
    """Same buffers as the reference (filters persistent, window not), identical filter bank values, CPU input raises."""
    g = golden("logmel_large_v3")
    m = pm.WhisperPreprocessor("large-v3")
    assert list(m.state_dict().keys()) == ["filters"] and m.window.shape == (400,)
    np.testing.assert_array_equal(m.filters.numpy(), g.sd["filters"])
    assert pm.WhisperPreprocessor().filters.shape == (80, 201)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 1600))


def test_torch_compile_fullgraph_traces_to_one_operator():
    """`torch.compile(m, fullgraph=True)` (reference tests: test_vit.py:14-18, test_gpt2.py:22, test_bert.py:22) must
    trace without a graph break: the whole forward is one b200enc::module_forward node. On this CPU-only box the node
    then raises the package's own 'no CPU fallback' error — a Dynamo `Unsupported` would mean a graph break."""
    import copy

    from pytorch_models_b200 import compile as pmc

    with torch.no_grad():
        for make, args in (
            (lambda: pm.ViT.from_google("Ti/16"), (torch.randn(1, 3, 224, 224),)),
            (lambda: pm.BERT(100, 1, 64), (torch.randint(0, 100, (1, 8)),)),
            (lambda: pm.GPT2(1, 64), (torch.randint(0, 100, (1, 8)),)),
            (lambda: pm.WhisperEncoder(1, 64), (torch.randn(1, 80, 16),)),
            (lambda: pm.Whisper(100, 1, 64), (torch.randn(1, 80, 16), torch.randint(0, 100, (1, 4)))),
            (lambda: pm.Encoder(1, 64), (torch.randn(1, 4, 64),)),
            (lambda: pm.Decoder(1, 64, cross_attn=True), (torch.randn(1, 4, 64), torch.randn(1, 6, 64))),
        ):
            m = make().eval()
            assert isinstance(m._b200_module_id, int) and "_b200_module_id" not in m.state_dict()
            compiled = torch.compile(m, fullgraph=True, backend="eager")
            with pytest.raises(RuntimeError, match="no CPU fallback"):
                compiled(*args)
    # the fake implementation describes the output without running anything
    m = pm.GPT2(1, 64)
    shape, dtype = type(m).forward._out_meta(m, torch.zeros(2, 5, dtype=torch.long), None)
    assert tuple(shape) == (2, 5, 50257) and dtype == torch.float32
    v = pm.ViT.from_google("Ti/16")
    assert type(v).forward._out_meta(v, torch.zeros(3, 3, 224, 224), None) == ((3, 192), torch.float32)
    # every instance has its own id; a deep copy has to be registered by hand before it is compiled
    a, b = pm.Encoder(1, 64), pm.Encoder(1, 64)
    assert a._b200_module_id != b._b200_module_id
    c = copy.deepcopy(a)
    assert c._b200_module_id == a._b200_module_id and pmc.register(c) != a._b200_module_id


def test_clock_sampler_windows_its_samples_to_the_timed_region():
    """bench.ClockSampler: samples are stamped on arrival; stop(t0, t1) reports those inside the timed region, and the
    warm-up + timed span (saying so) when the region is shorter than the sampling interval."""
    import bench

    s = bench.ClockSampler.__new__(bench.ClockSampler)

    class _Done:
        def terminate(self):
            pass

        def wait(self, timeout=None):
            return 0

    s.proc = _Done()
    s.lines = [(1.0, "1900, 1965, 300.0, Not Active, Not Active, Not Active, Not Active"),
               (2.0, "1200, 1965, 900.0, Not Active, Not Active, Not Active, Active"),
               (2.1, "1180, 1965, 950.0, Not Active, Not Active, Not Active, Active")]
    inside = s.stop(1.5, 2.5)
    assert inside["sm_mhz"] == 1190.0 and inside["samples"] == 2 and inside["reasons"] == ["sw_power_cap"]
    assert inside["window"] == "timed region" and inside["power_w_max"] == 950.0
    short = s.stop(3.0, 3.01)
    assert short["samples"] == 3 and short["window"].startswith("warm-up + timed region")


def test_bench_dump_outputs_is_float32_bounded_and_seeded(tmp_path, monkeypatch):
    """bench.dump_outputs: a small output is written whole as float32; a larger one is cut to the same seeded subset of
    samples, in batch order, on every call, within the byte limit."""
    import bench

    y = torch.arange(6 * 3 * 4, dtype=torch.bfloat16).reshape(6, 3, 4)
    bench.dump_outputs(str(tmp_path / "whole"), y, 0, 1)
    got = np.load(tmp_path / "whole" / "embeddings.npy")
    assert got.dtype == np.float32 and np.array_equal(got, y.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 3 * 4 * 4)  # room for two samples
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), y, 0, 1)
    a, b = np.load(tmp_path / "a" / "embeddings.npy"), np.load(tmp_path / "b" / "embeddings.npy")
    assert a.shape == (2, 3, 4) and np.array_equal(a, b)
    rows = [int(r[0, 0]) // 12 for r in a]
    assert rows == sorted(rows) and all(np.array_equal(r, y[i].float().numpy()) for r, i in zip(a, rows))
