"""How the `ops` wrappers pass device cache lengths to the C-ABI (no GPU needed).

Every entry point that reads the lengths takes (lens, len_stride): sequence b reads lens[b * len_stride]. These tests
record the calls `ops` makes into the library, with ``ops._need_cuda`` patched so that CPU tensors pass, and check for
a length tensor of 1 and of B elements which entry point is called, with which length pointer and which stride. The
arguments are matched to the parameter names declared in include/b200enc.h."""
from __future__ import annotations

import os
import re

import pytest
import torch

from pytorch_models_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, H, HD, CAPACITY = 3, 2, 64, 16


def _params(name: str) -> list[str]:
    """Parameter names of ``name`` in include/b200enc.h, without the trailing stream."""
    text = open(os.path.join(ROOT, "include", "b200enc.h")).read()
    decl = re.search(rf"\b{name}\(([^)]*)\);", text).group(1)
    names = [re.findall(r"\w+", p)[-1] for p in decl.split(",")]
    assert names[-1] == "stream"
    return names[:-1]


@pytest.fixture
def calls(monkeypatch):
    """The (entry point, {parameter: value}) of every library call `ops` makes; nothing is launched."""
    rec = []

    def record(name, meta, dev, *args):
        params = _params(name)
        assert len(args) == len(params) == len(_lib._SIGNATURES[name][1]) - 1, name
        rec.append((name, dict(zip(params, args))))

    monkeypatch.setattr(ops, "_need_cuda", lambda *ts: torch.device("cpu"))
    monkeypatch.setattr(ops, "_call", record)
    return rec


def _lengths(n: int) -> torch.Tensor:
    return torch.zeros(n, dtype=torch.int32)


def _decode_tensors():
    W = H * HD
    qkv = torch.zeros(B, 3 * W, dtype=torch.bfloat16)
    kv = torch.zeros(B, CAPACITY, 2 * W, dtype=torch.bfloat16)
    out = torch.zeros(B, W, dtype=torch.bfloat16)
    work = torch.zeros(1 << 16, dtype=torch.float32)
    return qkv[:, :W], kv[:, :, :W], kv[:, :, W:], out, work, qkv[:, W:2 * W], qkv[:, 2 * W:]


@pytest.mark.parametrize("n,stride", [(1, 0), (B, 1)])
def test_attention_decode_append(calls, n, stride):
    q, k, v, out, work, k_new, v_new = _decode_tensors()
    length = _lengths(n)
    ops.attention_decode(q, k, v, out, H, 0.125, work, k_new=k_new, v_new=v_new, length=length)
    [(name, a)] = calls
    assert name == "b200enc_attention_decode"
    assert a["lens"] == length.data_ptr() and a["len_stride"] == stride
    assert a["k_new"] == k_new.data_ptr() and a["v_new"] == v_new.data_ptr()


def test_attention_decode_cross(calls):
    q, k, v, out, work, _, _ = _decode_tensors()
    ops.attention_decode(q, k, v, out, H, 0.125, work, Lkv=7)
    [(name, a)] = calls
    assert name == "b200enc_attention_decode"
    assert a["lens"] is None and a["len_stride"] == 0 and a["Lkv"] == 7
    assert a["k_new"] is None and a["v_new"] is None


@pytest.mark.parametrize("n,stride", [(1, 0), (B, 1)])
def test_embed_rows_at(calls, n, stride):
    d = 64
    ids = torch.zeros(B, 1, dtype=torch.int64)
    tok, pos = torch.zeros(50, d), torch.zeros(CAPACITY, d)
    out = torch.zeros(B, 1, d, dtype=torch.bfloat16)
    pos0 = _lengths(n)
    ops.embed_rows_at(ids, tok, pos, pos0, out)
    [(name, a)] = calls
    assert name == "b200enc_embed_rows_at"
    assert a["pos0"] == pos0.data_ptr() and a["pos0_stride"] == stride
    assert a["rows"] == B and a["L"] == 1 and a["n_pos"] == CAPACITY


@pytest.mark.parametrize("n", [1, B])
def test_decode_advance(calls, n):
    length = _lengths(n)
    ops.decode_advance(length, 5)
    [(name, a)] = calls
    assert name == "b200enc_decode_advance"
    assert a["lens"] == length.data_ptr() and a["n"] == n and a["delta"] == 5
