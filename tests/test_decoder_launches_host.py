"""The library launches a decoder or encoder stack issues, pinned call for call (no GPU needed).

The value tests compare outputs, so a stack that lost a fused LayerNorm-statistics epilogue and ran one more kernel
would still pass them. This test replaces the `ops` entry points the modules call with recorders that launch nothing,
runs `Decoder.run` / `KVCache` construction / `Decoder.prefill` / `Decoder.step` and `Encoder.run` on CPU tensors, and
compares every call with ``tests/golden/decoder_launches.json``: entry point, positional and keyword arguments, and
for each tensor its storage (numbered in order of first appearance), storage offset, shape, stride and dtype, written
as ``s<storage>+<offset> (<shape>) (<stride>) <dtype>``.

``python tests/test_decoder_launches_host.py`` rewrites the data file.
"""
from __future__ import annotations

import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "golden", "decoder_launches.json")

# entry point -> index of the positional argument it returns
RECORDED = dict(linear=3, attention=3, attention_decode=3, row_stats=2, layernorm=4, decode_advance=0)
B, L, LM, CAPACITY = 2, 5, 7, 16


class Recorder:
    def __init__(self) -> None:
        self.calls: list = []
        self.labels: dict[int, int] = {}
        self.keep: list = []  # recorded storages stay alive, so no later allocation can reuse their address

    def _arg(self, v):
        if isinstance(v, torch.Tensor):
            s = v.untyped_storage()
            if s.data_ptr() not in self.labels:
                self.labels[s.data_ptr()] = len(self.labels)
                self.keep.append(s)
            shape, stride = ",".join(map(str, v.shape)), ",".join(map(str, v.stride()))
            return f"s{self.labels[s.data_ptr()]}+{v.storage_offset()} ({shape}) ({stride}) {str(v.dtype)[6:]}"
        return v

    def entry(self, name: str, ret: int):
        def record(*args, **kwargs):
            self.calls.append([name, [self._arg(a) for a in args], {k: self._arg(kwargs[k]) for k in sorted(kwargs)}])
            return args[ret]

        return record


def _decoder_cases() -> dict:
    cases = {}
    for norm in ("pre", "post"):
        for attn in ("self", "cross", "cross_nomem"):
            for d, hd in ((128, 64), (128, 80), (1600, 64)):
                cases[f"decoder_{norm}_{attn}_d{d}_hd{hd}"] = dict(
                    kind="decoder", pre_norm=norm == "pre", cross=attn != "self", memory=attn == "cross", d=d, hd=hd)
    for norm in ("pre", "post"):
        for d in (128, 1600):
            cases[f"encoder_{norm}_d{d}"] = dict(kind="encoder", pre_norm=norm == "pre", d=d, hd=64)
    return cases


CASES = _decoder_cases()


def record(case: dict, monkeypatch) -> dict:
    import pytorch_models_b200 as pm
    from pytorch_models_b200 import ops
    from pytorch_models_b200.transformer import KVCache

    rec = Recorder()
    for name, ret in RECORDED.items():
        monkeypatch.setattr(ops, name, rec.entry(name, ret))
    torch.manual_seed(0)
    d = case["d"]
    x3 = torch.zeros(B, L, d, dtype=torch.bfloat16)
    phases = {}

    def phase(name: str, fn) -> None:
        n = len(rec.calls)
        fn()
        phases[name] = rec.calls[n:]

    if case["kind"] == "encoder":
        enc = pm.Encoder(2, d, head_dim=case["hd"], pre_norm=case["pre_norm"]).eval()
        stats0 = torch.zeros(B * L, (d + 127) // 128, 2, dtype=torch.float32)
        phase("run", lambda: enc.run(x3))
        phase("run_stats0", lambda: enc.run(x3, stats0))
        return phases
    dec = pm.Decoder(2, d, head_dim=case["hd"], cross_attn=case["cross"], pre_norm=case["pre_norm"]).eval()
    m3 = torch.zeros(B, LM, d, dtype=torch.bfloat16) if case["memory"] else None
    phase("run_final_stats", lambda: dec.run(x3, m3, final_stats=True))
    phase("run", lambda: dec.run(x3, m3))
    if case["cross"] and not case["memory"]:
        return phases
    cache = []
    phase("kv_cache", lambda: cache.append(KVCache(dec, B, CAPACITY, m3)))
    phase("prefill", lambda: dec.prefill(x3, cache[0]))
    x1 = torch.zeros(B, 1, d, dtype=torch.bfloat16)
    phase("step", lambda: dec.step(x1, cache[0]))
    phase("step_2", lambda: dec.step(x1, cache[0]))
    return phases


@pytest.mark.parametrize("name", list(CASES))
def test_launch_sequence(name, monkeypatch):
    with open(DATA) as f:
        want = json.load(f)[name]
    got = json.loads(json.dumps(record(CASES[name], monkeypatch)))
    assert list(got) == list(want)
    for phase in want:
        g, w = got[phase], want[phase]
        for i, (gc, wc) in enumerate(zip(g, w)):
            assert gc == wc, f"{phase}: launch {i} differs:\n got  {gc}\n want {wc}"
        assert len(g) == len(w), f"{phase}: {len(g)} launches, want {len(w)}"


def _write() -> None:
    mp = pytest.MonkeyPatch()
    out = []
    try:
        for name, case in CASES.items():
            phases = record(case, mp)
            mp.undo()
            out.append(f"{json.dumps(name)}: {{\n" + ",\n".join(
                f"  {json.dumps(p)}: [" + ",".join("\n    " + json.dumps(c, separators=(",", ":")) for c in calls)
                + ("\n  ]" if calls else "]") for p, calls in phases.items()) + "\n}")
    finally:
        mp.undo()
    with open(DATA, "w") as f:
        f.write("{\n" + ",\n".join(out) + "\n}\n")


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _write()
