"""Every attention entry point on inputs with exactly known outputs (tests/attention_inputs.py): ops.attention
(single-pass, streaming and wide kernels; causal, rectangular causal, 0 / -inf bias), kv_append + attention_extend,
and attention_decode (shared-length and ragged append, cross). Exact-count cases must be within 1 bf16 ulp of the
exact output (the module docstring of attention_inputs.py says why that bound holds); planted-maximum cases must meet
the suite's bound against fp64 SDPA. test_attention_inputs_host.py proves on the CPU that each mistake a kernel could
make on these inputs breaks the bound; the negative controls below show the same on the GPU with legal launches whose
arguments are wrong."""
from __future__ import annotations

import pytest
import torch

import attention_inputs as ai
from pytorch_models_b200 import ops

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", sorted(ai.EXACT_CASES))
def test_exact(name):
    case = ai.EXACT_CASES[name]()
    got = case.run(ops)
    torch.cuda.synchronize()
    ai.assert_exact(got.cpu(), case.expected(), case.zero_tol, name)
    if isinstance(case, ai.DecodeExact) and case.append:
        case.check_cache()


@pytest.mark.parametrize("name", sorted(ai.PLANTED_CASES))
def test_planted_maximum(name):
    case = ai.PLANTED_CASES[name]()
    got = case.run(ops)
    torch.cuda.synchronize()
    ai.assert_close(got.cpu(), case.expected(), what=name)


# ------------------------------------------------------------------------------------------------- negative controls
@pytest.mark.parametrize("d", [-1, 1])
@pytest.mark.parametrize("ragged", [False, True])
def test_decode_with_a_wrong_length_is_rejected(d, ragged):
    cap = 4096 + ai.GUARD
    lengths = [4095, 2000, 77] if ragged else [4095] * 3
    case = ai.DecodeExact(3, 2, 128, cap, lengths, shared=not ragged)
    got = case.run(ops, lengths=[n + d for n in lengths])
    torch.cuda.synchronize()
    with pytest.raises(AssertionError):
        ai.assert_exact(got.cpu(), case.expected(), case.zero_tol)
    for b in range(3):  # in every sequence
        with pytest.raises(AssertionError):
            ai.assert_exact(got[b].cpu(), case.expected()[b], case.zero_tol)


@pytest.mark.parametrize("d", [-1, 1])
def test_extend_with_a_wrong_offset_is_rejected(d):
    offs = [1, 129, 1500]
    case = ai.ExtendExact(3, 2, 64, 7, offs, 2048)
    got = case.run(ops, offsets=[o + d for o in offs])
    torch.cuda.synchronize()
    for b in range(3):
        with pytest.raises(AssertionError):
            ai.assert_exact(got[b].cpu(), case.expected()[b], case.zero_tol)


@pytest.mark.parametrize("hd", [64, 128])
def test_non_causal_launch_is_rejected_against_the_causal_expectation(hd):
    case = ai.AttnExact(2, 3, hd, 1024, 1024, causal=True)
    case.causal = False
    got = case.run(ops)
    case.causal = True
    torch.cuda.synchronize()
    with pytest.raises(AssertionError):
        ai.assert_exact(got.cpu(), case.expected(), case.zero_tol)
