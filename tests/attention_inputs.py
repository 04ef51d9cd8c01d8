"""Attention inputs whose outputs are known exactly, planted-maximum inputs, their references, and the mistakes
("mutants") each check must be able to reject. Shared by test_attention_inputs_host.py (CPU: every mutant breaks the
bound of its case) and test_gpu_attention_exact.py (the kernels meet it). Not collected as a test module.

Exact-count inputs. q = 0, so every score is exactly 0, every softmax weight is equal and an output is the plain mean
of the value rows the query may see. Every v entry is 0 or 1, so output element c of a query that sees n keys is
count_c / n: known exactly, and each column answers a question about which keys were read:

  columns [0, G)   class columns: v[j, c] = 1 iff (j // u) mod G == c (unit classes; u = the kernel's smallest unit
                   of keys), or j mod G == c (position classes, for causal and extend masks, where a one-key leak must
                   move a column by several bf16 ulps at every row)
  KEY0             key 0
  UNIT_FLAGS       the first and the last key of each of the last two units of the sequence's n keys
  LAST             the last cached row (the last key before the new ones)
  NEW              the new row of a decode append (k_new / v_new)
  STALE            set only in rows the kernel must not attend: the stale row a speculative rollback leaves at cache
                   row `len`, and the finite rows past an extend's keys inside its last 128-key block
  B_BITS, H_BITS   the bits of the sequence b and the head h, in every key: a work item that reads another sequence's
                   or head's rows gives wrong bits, not a small drift
  ONES             1 in every key: the output is exactly 1 (the normalisation)

Rows the kernel must not read at all hold NaN (k and v).

Why the bound is 1 bf16 ulp of the exact value, and exactly 0 where that is 0 (`assert_exact`):
  - decode (csrc/attention_decode.cuh): exp2f(0) = 1 for every key, the lane-group, warp and chunk merges scale by
    exp2f(0) = 1, l and o are sums of 0/1 values (exact in fp32 below 2^24), and o / l is one correctly rounded fp32
    division: the only error is its rounding and the rounding to bf16, together at most 1 bf16 ulp. Keys out of range
    get P = exp2f(-inf) = 0 and are never loaded, so a zero count stays exactly 0.
  - tensor-core kernels (attention_short / _stream / _wide.cuh): P enters the P.V MMA as bf16, where 1 is exact, so
    O = count exactly. exp2_poly2 (every 4th pair of scores) returns 0.99992895 for 0, which rounds to 1 in bf16. The
    single-pass kernel sums l from the bf16 P (l = n exactly); the streaming and wide kernels sum l from the fp32 P,
    so l is n (1 - 1.8e-5) at worst and O / l can cross one bf16 rounding boundary: still within 1 ulp.
    Where the exact value is 0 the tensor-core kernels give at most TC_ZERO_TOL, not 0: exp2_poly2 clamps its
    argument at -126, so a masked score (-inf) in a polynomial column gets P = 2^-126 instead of 0, and a masked key
    whose v is 1 adds 2^-126 to O. At most 128 masked keys of a row share its last block: |out| <= 128 * 2^-126 / l.
    A key that is really read adds at least 1 / n >= 2^-16.

Planted maxima. Exact-count inputs make every merge scale exactly 1, so they cannot test the online-softmax rescale.
Random background inputs (gain 1.5, as the suite draws them) get one key per (b, h) whose score is the row maximum by
a margin of 3, built along q and rounded to bf16, with v = 4 in every column; it sits at the first or the last key of
a late decode chunk or 128-key block. Its share of the output is of order 1, so the usual bound against fp64 SDPA
(`assert_close`) catches a partial of that chunk scaled by 2^+-1.

Every input is drawn with a CPU torch.Generator, so the host and GPU tests see identical tensors."""
from __future__ import annotations

import math

import torch

DEC_MIN_CHUNK = 64     # csrc/attention_decode.cuh: every decode chunk is a multiple of it
DEC_MAX_CHUNK = 4096
ATT_BKV = 128          # csrc/attention_common.cuh: key block of the tensor-core kernels
GUARD = 8              # rows past the keys of an ops.attention input (NaN) or a decode cache

G = 40
KEY0 = 40
UNIT_FLAGS = (41, 42, 43, 44)
LAST = 45
NEW = 46
STALE = 47
B_BITS = 48            # 8 bits: B <= 256
H_BITS = 56            # 6 bits: H <= 64
ONES = 62
TC_ZERO_TOL = 128 * 2.0 ** -126
PLANT_MARGIN = 3.0
PLANT_V = 4.0


def decode_chunk(B, H, keys):
    """Keys per work item of the decode kernel (decode_chunk in csrc/api_decode.cu)."""
    bh = B * H
    nch = 1 if bh >= 4096 else -(-4096 // bh)
    kc = -(-keys // nch)
    kc = -(-kc // DEC_MIN_CHUNK) * DEC_MIN_CHUNK
    return min(max(kc, DEC_MIN_CHUNK), DEC_MAX_CHUNK)


# ------------------------------------------------------------------------------------------------- comparisons
def bf16_round(x):
    return x.to(torch.bfloat16).double()


def bf16_ulp(x):
    """Spacing of bf16 numbers at |x| (x != 0): 2^(floor(log2 |x|) - 7)."""
    e = torch.floor(torch.log2(x.abs().clamp(min=2.0 ** -126)))
    return torch.exp2(e - 7)


def assert_exact(got, want, zero_tol=0.0, what=""):
    """|got - want| <= 1 bf16 ulp of want where want != 0, |got| <= zero_tol where want == 0, NaN where want is NaN."""
    got, want = got.double().cpu(), want.double().cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    nan = want.isnan()
    zero = want == 0
    bad = nan & ~got.isnan()
    bad |= ~nan & zero & ~(got.abs() <= zero_tol)
    bad |= ~nan & ~zero & ~((got - want).abs() <= bf16_ulp(want))
    if bool(bad.any()):
        idx = tuple(int(i) for i in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements off the exact output, first at {idx}: "
                             f"got {got[idx].item():.9g}, want {want[idx].item():.9g}")


def assert_close(got, want, atol=0.02, rtol=0.02, what=""):
    """The suite's bound against a reference: |got - want| <= atol + rtol |want|."""
    err = (got.double().cpu() - want.double().cpu()).abs()
    bound = atol + rtol * want.double().cpu().abs()
    ok = err <= bound
    if not bool(ok.all()):
        raise AssertionError(f"{what}: max err {err.max().item():.4g}, worst excess {(err - bound).max().item():.4g}")


# ------------------------------------------------------------------------------------------------- value rows
def value_rows(j, b, H, hd, *, u, n, last, position=False):
    """float32 (len(j), H*hd) exact-count value rows of sequence b for key indices j (see the module docstring)."""
    j = torch.as_tensor(j, dtype=torch.long).view(-1, 1, 1)
    c = torch.arange(hd).view(1, 1, hd)
    h = torch.arange(H).view(1, H, 1)
    cls = j % G if position else (j // u) % G
    v = (c < G) & (cls == c)
    v = v | ((c == KEY0) & (j == 0))
    if n >= 1:
        U1 = (n - 1) // u
        for col, r in zip(UNIT_FLAGS, (U1 * u, n - 1, (U1 - 1) * u, U1 * u - 1)):
            if r >= 0:
                v = v | ((c == col) & (j == r))
    v = v | ((c == LAST) & (j == last))
    for i in range(8):
        if (b >> i) & 1:
            v = v | (c == B_BITS + i)
    hb = (c >= H_BITS) & (c < H_BITS + 6) & (((h >> (c - H_BITS).clamp(min=0)) & 1) == 1)
    v = v | hb | (c == ONES)
    return v.float().reshape(j.shape[0], H * hd)


class _Prefix:
    """Prefix sums of value rows (R, W): sums of any row range, NaN rows counted apart."""

    def __init__(self, rows):
        rows = rows.float()
        nan = rows.isnan().any(1)
        z = torch.where(nan[:, None], torch.zeros(()), rows)
        self.S = torch.cat([torch.zeros(1, rows.shape[1]), z.cumsum(0)])
        self.N = torch.cat([torch.zeros(1, dtype=torch.long), nan.long().cumsum(0)])
        self.R = rows.shape[0]

    def range(self, r0, r1):
        """r0, r1: (Q,) long -> (sum (Q, W) float64, count (Q,), any NaN (Q,)). Rows past R read as zero rows."""
        a, e = r0.clamp(0, self.R), r1.clamp(0, self.R)
        e = torch.maximum(a, e)
        return (self.S[e] - self.S[a]).double(), (r1 - r0).clamp(min=0), self.N[e] - self.N[a] > 0


def mean_of(terms, Q, W):
    """terms: [(prefix, r0, r1, weight)] with r0 / r1 ints or (Q,) tensors -> (Q, W) float64 weighted mean of the rows;
    NaN where a NaN row has non-zero weight or no key is left."""
    num = torch.zeros(Q, W, dtype=torch.float64)
    den = torch.zeros(Q, dtype=torch.float64)
    nan = torch.zeros(Q, dtype=torch.bool)
    for pf, r0, r1, w in terms:
        r0 = torch.as_tensor(r0, dtype=torch.long).expand(Q)
        r1 = torch.as_tensor(r1, dtype=torch.long).expand(Q)
        s, cnt, nn = pf.range(r0, r1)
        num += w * s
        den += w * cnt
        nan |= nn & (cnt > 0)
    out = num / den.clamp(min=1e-300)[:, None]
    out[nan | (den <= 0)] = float("nan")
    return out


def _units(n, u):
    """Named units of n keys: first, middle, last full unit, partial tail unit (those that exist)."""
    if n < 1:
        return {}
    count = -(-n // u)
    names = {"first": 0, "middle": count // 2}
    if n >= u:
        names["last_full"] = n // u - 1
    if n % u:
        names["tail"] = n // u
    return names


def unit_mutants(n, u):
    """Mutants that drop or duplicate one unit of keys [0, n): {name: (first key, end key, weight)}."""
    out = {}
    for name, U in _units(n, u).items():
        out[f"drop_{name}_unit"] = (U * u, min(U * u + u, n), -1)
    if n > u:  # duplicating every key leaves the softmax unchanged
        U = _units(n, u)["middle"]
        out["dup_middle_unit"] = (U * u, min(U * u + u, n), 1)
    return out


def _nan_rows(t, r0):
    t[r0:] = float("nan")


# ------------------------------------------------------------------------------------------------- ops.attention
class AttnExact:
    """ops.attention on exact-count inputs: q = 0, k / v views of (B, Lkv + GUARD, 2W) rows whose guard rows are NaN.
    causal: top-left aligned (SDPA's is_causal), position classes. bias: a fixed random 0 / -inf bias (30 % masked,
    every row keeps at least one key)."""

    u = ATT_BKV
    zero_tol = TC_ZERO_TOL

    def __init__(self, B, H, hd, Lq, Lkv, causal=False, bias=False, streaming=False, seed=0):
        self.B, self.H, self.hd, self.Lq, self.Lkv = B, H, hd, Lq, Lkv
        self.causal, self.use_bias, self.streaming = causal, bias, streaming
        self.W = W = H * hd
        R = Lkv + GUARD
        self.kv = torch.zeros(B, R, 2 * W)
        for b in range(B):
            self.kv[b, :Lkv, W:] = value_rows(torch.arange(Lkv), b, H, hd, u=self.u, n=Lkv, last=Lkv - 1,
                                              position=causal)
            _nan_rows(self.kv[b], Lkv)
        self.kv = self.kv.bfloat16()
        self.q = torch.zeros(B, Lq, W, dtype=torch.bfloat16)
        self.bias = None
        if bias:
            g = torch.Generator().manual_seed(seed)
            keep = torch.rand(B, H, Lq, Lkv, generator=g) >= 0.3
            first = torch.randint(0, Lkv, (B, H, Lq, 1), generator=g)
            keep.scatter_(3, first, True)
            self.keep = keep
            self.bias = torch.where(keep, 0.0, float("-inf"))
        self.pf = [_Prefix(self.kv[b, :, W:]) for b in range(B)]
        self.n_seen = int(self.hi().max())  # keys [0, n_seen) are seen by some query

    def hi(self, align="top_left", d=0):
        """Keys [0, hi_i) seen by query i; d shifts the causal diagonal."""
        if not self.causal:
            return torch.full((self.Lq,), self.Lkv)
        shift = 0 if align == "top_left" else self.Lkv - self.Lq
        return (torch.arange(self.Lq) + 1 + shift + d).clamp(0, self.Lkv)

    def mutants(self):
        ms = list(unit_mutants(self.n_seen, self.u)) + ["kv_minus_1", "kv_plus_1"]
        if self.causal:
            ms += ["diag_minus_1", "diag_plus_1"]
            if self.Lq != self.Lkv:
                ms.append("bottom_right")
        if self.use_bias:
            ms.append("mask_leak")
        return [m for m in ms if any(self.applies(m, b) for b in range(self.B))]

    def applies(self, mutant, b):
        if mutant == "mask_leak":
            return bool((~self.keep[b]).any())
        if mutant == "diag_plus_1":  # a query that does not see every key
            return bool((self.hi() < self.Lkv).any())
        if mutant.startswith("kv_"):  # a query that sees every key
            return self.n_seen == self.Lkv and not (mutant == "kv_minus_1" and self.Lkv == 1)
        return True

    def expected(self, mutant=None):
        if self.use_bias:
            return self._expected_bias(mutant)
        B, Q, W, Lkv = self.B, self.Lq, self.W, self.Lkv
        out = torch.empty(B, Q, W, dtype=torch.float64)
        units = unit_mutants(self.n_seen, self.u)
        for b in range(B):
            pf = self.pf[b]
            d = {"diag_minus_1": -1, "diag_plus_1": 1}.get(mutant, 0)
            hi = self.hi("bottom_right" if mutant == "bottom_right" else "top_left", d)
            extra = []
            if mutant == "kv_minus_1":
                hi = hi.clamp(max=Lkv - 1)
            elif mutant == "kv_plus_1":
                hi = torch.where(hi == Lkv, hi + 1, hi)
            elif mutant in units:
                a, e, w = units[mutant]
                extra = [(pf, torch.full((Q,), a), torch.minimum(hi, torch.tensor(e)), w)]
            out[b] = mean_of([(pf, 0, hi, 1)] + extra, Q, W)
        return out

    def _expected_bias(self, mutant):
        B, H, hd, Q, Lkv = self.B, self.H, self.hd, self.Lq, self.Lkv
        w = self.keep.double()
        units = unit_mutants(Lkv, self.u)
        R = Lkv
        if mutant == "kv_plus_1":
            w = torch.cat([w, torch.ones(B, H, Q, 1, dtype=torch.float64)], 3)
            R = Lkv + 1
        elif mutant == "kv_minus_1":
            w = w.clone()
            w[..., Lkv - 1] = 0
        elif mutant == "mask_leak":
            w = w.clone()
            masked = ~self.keep
            first = masked.double().argmax(3, keepdim=True)
            w.scatter_(3, first, torch.where(masked.any(3, keepdim=True), 1.0, w.gather(3, first)))
        elif mutant in units:
            a, e, s = units[mutant]
            w = w.clone()
            w[..., a:e] *= 1 + s
        v = self.kv[:, :R, self.W:].double().view(B, R, H, hd).transpose(1, 2)  # (B, H, R, hd)
        vz = torch.nan_to_num(v)
        num = w @ vz
        out = num / w.sum(3, keepdim=True)
        has_nan = (w * v.isnan().any(3).double()[:, :, None, :]).sum(3) > 0
        out[has_nan] = float("nan")
        out[w.sum(3) <= 0] = float("nan")
        return out.transpose(1, 2).reshape(B, Q, self.W)

    def run(self, ops, device="cuda"):
        W = self.W
        kv = self.kv.to(device)
        q = self.q.to(device)
        out = torch.full((self.B, self.Lq, W), float("nan"), device=device, dtype=torch.bfloat16)
        bias = None if self.bias is None else self.bias.to(device)
        ops.attention(q, kv[:, :self.Lkv, :W], kv[:, :self.Lkv, W:], out, self.H, self.hd ** -0.5,
                      causal=self.causal, bias=bias, streaming=self.streaming)
        return out


# ------------------------------------------------------------------------------------------------- extend
class ExtendExact:
    """kv_append + ops.attention_extend on exact-count inputs (position classes). Sequence b has `off` cached rows;
    the P new rows come from the q|k|v buffer. Before the append, rows [off, off + P) and the finite rows past the
    keys inside the last 128-key block hold STALE-flagged rows (a rolled-back speculative round); every row after that
    block is NaN. shared: one device length for the batch."""

    u = ATT_BKV
    zero_tol = TC_ZERO_TOL

    def __init__(self, B, H, hd, P, offsets, capacity, shared=False):
        self.B, self.H, self.hd, self.P, self.offsets, self.capacity = B, H, hd, P, list(offsets), capacity
        self.shared = shared
        assert not shared or len(set(offsets)) == 1
        self.W = W = H * hd
        kv = torch.zeros(B, capacity, 2 * W)
        qkv = torch.zeros(B, P, 3 * W)
        after = torch.zeros(B, capacity, W)
        for b, o in enumerate(self.offsets):
            n = o + P
            rows = value_rows(torch.arange(n), b, H, hd, u=self.u, n=n, last=o - 1, position=True)
            end = min(-(-n // ATT_BKV) * ATT_BKV, capacity)
            stale = value_rows(torch.arange(o, end), b, H, hd, u=self.u, n=n, last=o - 1, position=True)
            stale.view(-1, H, hd)[:, :, STALE] = 1
            kv[b, :o, W:] = rows[:o]
            kv[b, o:end, W:] = stale
            _nan_rows(kv[b], end)
            qkv[b, :, 2 * W:] = rows[o:]
            after[b] = kv[b, :, W:]
            after[b, o:n] = rows[o:]
        self.kv, self.qkv = kv.bfloat16(), qkv.bfloat16()
        self.pf = [_Prefix(after[b]) for b in range(B)]

    def mutants(self):
        ms = list(dict.fromkeys(m for o in self.offsets for m in unit_mutants(o + self.P, self.u)))
        ms += ["off_minus_1", "off_plus_1", "top_left"]
        if len(set(self.offsets)) > 1:
            ms += ["other_len_prev", "other_len_next"]
        return [m for m in ms if any(self.applies(m, b) for b in range(self.B))]

    def applies(self, mutant, b):
        o = self.offsets[b]
        if mutant.endswith("_unit"):
            return mutant in unit_mutants(o + self.P, self.u)
        if mutant == "off_minus_1" or mutant == "top_left":
            return o >= 1
        if mutant.startswith("other_len"):
            nb = b - 1 if mutant.endswith("prev") else b + 1
            return 0 <= nb < self.B and self.offsets[nb] != o
        return True

    def _hi(self, o):
        return o + torch.arange(self.P) + 1

    def expected(self, mutant=None):
        B, P, W, cap = self.B, self.P, self.W, self.capacity
        out = torch.empty(B, P, W, dtype=torch.float64)
        for b, o in enumerate(self.offsets):
            pf, extra = self.pf[b], []
            units = unit_mutants(o + P, self.u)
            hi = self._hi(o)
            if mutant in ("off_minus_1", "off_plus_1") or (mutant or "").startswith("other_len"):
                if mutant == "off_minus_1":
                    o2 = o - 1
                elif mutant == "off_plus_1":
                    o2 = o + 1
                else:
                    nb = b - 1 if mutant.endswith("prev") else b + 1
                    o2 = self.offsets[nb] if 0 <= nb < B else o
                if not 0 <= o2 <= cap - P:  # the kernel's range check: the whole sequence is NaN
                    out[b] = float("nan")
                    continue
                hi = self._hi(o2)
            elif mutant == "top_left":
                hi = torch.arange(P) + 1
            elif mutant in units:
                a, e, w = units[mutant]
                extra = [(pf, torch.full((P,), a), torch.minimum(hi, torch.tensor(e)), w)]
            out[b] = mean_of([(pf, 0, hi, 1)] + extra, P, W)
        return out

    def run(self, ops, device="cuda", offsets=None):
        W = self.W
        offsets = self.offsets if offsets is None else offsets
        self.kv_dev = kv = self.kv.to(device)
        qkv = self.qkv.to(device)
        length = torch.tensor(offsets[:1] if self.shared else offsets, device=device, dtype=torch.int32)
        out = torch.full((self.B, self.P, W), float("nan"), device=device, dtype=torch.bfloat16)
        ops.kv_append(qkv[:, :, W:], kv, length)
        ops.attention_extend(qkv[:, :, :W], kv[:, :, :W], kv[:, :, W:], out, self.H, self.hd ** -0.5, length)
        return out


# ------------------------------------------------------------------------------------------------- decode
class DecodeExact:
    """ops.attention_decode on exact-count inputs (unit classes, u = DEC_MIN_CHUNK).

    Append mode (lengths given): sequence b attends cache rows [0, len_b) plus the new row (k_new / v_new, flag NEW);
    cache row len_b holds a stale row (flag STALE, NEW cleared) that the kernel must replace, not read; rows past it
    are NaN. A length outside [0, capacity) must give a NaN output and leave its cache alone (its rows are all NaN).
    shared: one device length for the batch (every length equal). Cross mode (Lkv given): rows [0, Lkv), NaN past."""

    u = DEC_MIN_CHUNK
    zero_tol = 0.0

    def __init__(self, B, H, hd, capacity, lengths=None, Lkv=None, shared=False):
        self.B, self.H, self.hd, self.capacity = B, H, hd, capacity
        self.lengths, self.Lkv, self.shared = lengths, Lkv, shared
        self.append = lengths is not None
        assert self.append != (Lkv is not None)
        assert not shared or len(set(lengths)) == 1
        self.W = W = H * hd
        kv = torch.zeros(B, capacity, 2 * W, dtype=torch.bfloat16)
        new = torch.zeros(B, W)
        self.pf, self.pf_new = [], []
        for b in range(B):
            n = lengths[b] if self.append else Lkv
            if self.append and not 0 <= n < capacity:
                kv[b] = float("nan")
                new[b] = value_rows([0], b, H, hd, u=self.u, n=1, last=-1)[0]
            else:
                keys = n + 1 if self.append else n
                rows = value_rows(torch.arange(keys), b, H, hd, u=self.u, n=keys, last=n - 1)
                kv[b, :n, W:] = rows[:n].bfloat16()
                if self.append:
                    nr = rows[n].view(H, hd)
                    nr[:, NEW] = 1
                    new[b] = nr.reshape(W)
                    stale = rows[n].view(H, hd).clone()
                    stale[:, NEW], stale[:, STALE] = 0, 1
                    kv[b, n, W:] = stale.reshape(W).bfloat16()
                    kv[b, n + 1:] = float("nan")
                else:
                    kv[b, n:] = float("nan")
            self.pf.append(_Prefix(kv[b, :, W:]))
            self.pf_new.append(_Prefix(new[b:b + 1]))
        self.kv = kv
        self.qkv = torch.zeros(B, 3 * W, dtype=torch.bfloat16)
        self.qkv[:, 2 * W:] = new.bfloat16()

    def _n(self, b):
        return self.lengths[b] if self.append else self.Lkv

    def _valid(self, n):
        return 0 <= n < self.capacity if self.append else True

    def mutants(self):
        keys = [self._n(b) + self.append for b in range(self.B) if self._valid(self._n(b))]
        ms = list(dict.fromkeys(m for n in keys for m in unit_mutants(n, self.u)))
        ms += ["len_minus_1", "len_plus_1"]
        if self.append:
            ms.append("stale_for_new")
            if not self.shared and len(set(self.lengths)) > 1:
                ms += ["other_len_prev", "other_len_next"]
        return [m for m in ms if any(self.applies(m, b) for b in range(self.B))]

    def applies(self, mutant, b):
        n = self._n(b)
        if not self._valid(n):
            return False
        keys = n + 1 if self.append else n
        if mutant.endswith("_unit"):
            return mutant in unit_mutants(keys, self.u)
        if mutant == "len_minus_1":
            return n >= 1 if self.append else n >= 2
        if mutant == "len_plus_1":
            return self.append or n < self.capacity
        if mutant.startswith("other_len"):
            nb = b - 1 if mutant.endswith("prev") else b + 1
            return 0 <= nb < self.B and self.lengths[nb] != n
        return True

    def _terms(self, b, n, pf, pn):
        """Keys of a sequence of length n: cache rows [0, n) + the new row (append), or rows [0, n) (cross)."""
        if not self.append:
            return [(pf, 0, n, 1)]
        if not 0 <= n < self.capacity:
            return None
        return [(pf, 0, n, 1), (pn, 0, 1, 1)]

    def expected(self, mutant=None):
        B, W = self.B, self.W
        out = torch.empty(B, W, dtype=torch.float64)
        for b in range(B):
            n, pf, pn = self._n(b), self.pf[b], self.pf_new[b]
            if not self._valid(n):
                out[b] = float("nan")
                continue
            keys = n + 1 if self.append else n
            units = unit_mutants(keys, self.u)
            terms = self._terms(b, n, pf, pn)
            if mutant == "len_minus_1":
                terms = self._terms(b, n - 1, pf, pn)
            elif mutant == "len_plus_1":
                terms = self._terms(b, n + 1, pf, pn) or [(pf, 0, n + 1, 1), (pn, 0, 1, 1)]
            elif mutant == "stale_for_new":
                terms = [(pf, 0, n + 1, 1)]
            elif mutant is not None and mutant.startswith("other_len"):
                nb = b - 1 if mutant.endswith("prev") else b + 1
                if 0 <= nb < B:
                    terms = self._terms(b, self.lengths[nb], pf, pn)
            elif mutant in units:
                a, e, w = units[mutant]
                terms = terms + [(pf, a, min(e, n), w)]
                if self.append and a <= n < e:
                    terms.append((pn, 0, 1, w))
            out[b] = float("nan") if terms is None else mean_of(terms, 1, W)[0]
        return out

    def run(self, ops, device="cuda", lengths=None):
        W = self.W
        self.kv_dev = kv = self.kv.to(device)
        qkv = self.qkv.to(device)
        keys = self.capacity if self.append else self.Lkv
        work = torch.empty(ops.decode_workspace_bytes(self.B, self.H, self.hd, keys) // 4, device=device)
        out = torch.full((self.B, W), float("nan"), device=device, dtype=torch.bfloat16)
        if not self.append:
            ops.attention_decode(qkv[:, :W], kv[:, :, :W], kv[:, :, W:], out, self.H, self.hd ** -0.5, work,
                                 Lkv=self.Lkv)
            return out
        lengths = self.lengths if lengths is None else lengths
        length = torch.tensor(lengths[:1] if self.shared else lengths, device=device, dtype=torch.int32)
        ops.attention_decode(qkv[:, :W], kv[:, :, :W], kv[:, :, W:], out, self.H, self.hd ** -0.5, work,
                             k_new=qkv[:, W:2 * W], v_new=qkv[:, 2 * W:], length=length)
        return out

    def check_cache(self):
        """After an append: cache row len_b holds the new k|v row bit for bit, every other row is unchanged (NaN
        included), and a sequence with an out-of-range length is untouched."""
        kv = self.kv_dev.cpu().view(torch.int16)
        before = self.kv.view(torch.int16)
        new = self.qkv[:, self.W:].view(torch.int16)
        for b in range(self.B):
            n = self._n(b)
            keep = torch.ones(self.capacity, dtype=torch.bool)
            if self.append and 0 <= n < self.capacity:
                assert torch.equal(kv[b, n], new[b]), f"sequence {b}: the new k|v row was not written bit for bit"
                keep[n] = False
            assert torch.equal(kv[b, keep], before[b, keep]), f"sequence {b} (length {n}): another cache row changed"


# ------------------------------------------------------------------------------------------------- planted maxima
def _plant(q, k, scale, p, g):
    """q (Q, H, hd), k (R, H, hd) float64 of bf16 values; returns (q, k) with key p made every query's maximum by at
    least PLANT_MARGIN over the other keys of rows [0, R) (q shifted along one direction when Q > 1), rounded to bf16."""
    Q, H, hd = q.shape
    if Q == 1:
        u = q[0] / q[0].norm(dim=-1, keepdim=True)
    else:
        u = torch.randn(H, hd, generator=g, dtype=torch.float64)
        u = u / u.norm(dim=-1, keepdim=True)
        q = bf16_round(q + 8.0 * u)
    qu = (q * u).sum(-1)  # (Q, H)
    assert bool((qu > 0).all())
    s = torch.einsum("qhd,rhd->hqr", q, k) * scale
    s[:, :, p] = -math.inf
    top = s.max(-1).values.T  # (Q, H)
    beta = ((top + PLANT_MARGIN) / (scale * qu)).max(0).values  # (H,)
    k = k.clone()
    k[p] = bf16_round(beta[:, None] * u)
    return q, k


class Planted:
    """Random inputs (gain 1.5) with one planted maximum per (b, h) at the first or last key of a late unit: the
    second-to-last decode chunk (kind decode / ragged / cross) or 128-key block (stream / wide / extend) of the keys
    every query sees. Reference: fp64 SDPA; bound: `assert_close`."""

    def __init__(self, kind, B, H, hd, lengths, where, Lq=4, seed=0):
        self.kind, self.B, self.H, self.hd, self.lengths, self.where = kind, B, H, hd, list(lengths), where
        self.W = W = H * hd
        self.scale = hd ** -0.5
        g = torch.Generator().manual_seed(seed)
        r = lambda *s: bf16_round(torch.randn(*s, generator=g, dtype=torch.float64) * 1.5)  # noqa: E731
        decode = kind in ("decode", "ragged", "cross")
        self.Q = 1 if decode else Lq
        if kind in ("decode", "ragged"):
            self.capacity = max(lengths) + 1 + GUARD
            keys = [n + 1 for n in lengths]
        elif kind == "cross":
            self.capacity = max(lengths) + GUARD
            keys = list(lengths)
        elif kind == "extend":
            self.capacity = max(lengths) + GUARD
            keys = list(lengths)  # kv_len = offset + Q
        else:
            self.capacity = lengths[0] + GUARD
            keys = [lengths[0]] * B
        self.keys = keys
        self.unit = decode_chunk(B, H, self.capacity if kind != "cross" else max(lengths)) if decode else ATT_BKV
        R = self.capacity
        q = r(B, self.Q, H, hd)
        k = r(B, R, H, hd)
        v = r(B, R, H, hd)
        self.p = []
        for b in range(B):
            n_all = keys[b] - (self.Q - 1 if kind == "extend" else 0)  # keys every query of b sees
            U = max((n_all - 1) // self.unit - 1, 0)
            p = U * self.unit if where == "first" else min(U * self.unit + self.unit, n_all) - 1
            self.p.append(p)
            q[b], kb = _plant(q[b], k[b, :keys[b]], self.scale, p, g)
            k[b, :keys[b]] = kb
            v[b, p] = PLANT_V
            k[b, keys[b]:] = float("nan")
            v[b, keys[b]:] = float("nan")
        self.q, self.k, self.v = q, k, v

    def mutants(self):
        return ["planted_unit_x2", "planted_unit_x0.5"]

    def applies(self, mutant, b):
        return True

    def expected(self, mutant=None):
        """fp64 SDPA over each query's visible keys; a mutant scales the planted unit's partial by 2^+-1."""
        B, Q, H, hd = self.B, self.Q, self.H, self.hd
        out = torch.empty(B, Q, H, hd, dtype=torch.float64)
        for b in range(B):
            n = self.keys[b]
            k, v = self.k[b, :n], self.v[b, :n]
            s = torch.einsum("qhd,rhd->hqr", self.q[b], k) * self.scale
            if self.kind == "extend":
                o = n - Q
                vis = torch.arange(n)[None, :] <= o + torch.arange(Q)[:, None]
                s = s.masked_fill(~vis, -math.inf)
            w = torch.exp(s - s.max(-1, keepdim=True).values)
            if mutant is not None:
                U = self.p[b] // self.unit
                w[:, :, U * self.unit:U * self.unit + self.unit] *= 2.0 if mutant.endswith("x2") else 0.5
            out[b] = torch.einsum("hqr,rhd->qhd", w / w.sum(-1, keepdim=True), v)
        out = out.reshape(B, Q, self.W)
        return out[:, 0] if self.Q == 1 else out

    def run(self, ops, device="cuda"):
        B, H, hd, W, R = self.B, self.H, self.hd, self.W, self.capacity
        to = lambda t: t.reshape(*t.shape[:-2], W).bfloat16().to(device)  # noqa: E731
        q, k, v = to(self.q), to(self.k), to(self.v)
        kv = torch.cat([k, v], -1)
        if self.kind in ("decode", "ragged", "cross"):
            keys = max(self.lengths) if self.kind == "cross" else R
            work = torch.empty(ops.decode_workspace_bytes(B, H, hd, keys) // 4, device=device)
            out = torch.full((B, W), float("nan"), device=device, dtype=torch.bfloat16)
            if self.kind == "cross":
                ops.attention_decode(q[:, 0], kv[:, :, :W], kv[:, :, W:], out, H, self.scale, work, Lkv=self.lengths[0])
                return out
            # the planted inputs hold the new row at key len_b: it is passed as k_new / v_new, and the cache row it
            # replaces is made NaN (the kernel must not read it)
            lens = self.lengths
            new = torch.stack([kv[b, n] for b, n in enumerate(lens)])
            for b, n in enumerate(lens):
                kv[b, n] = float("nan")
            length = torch.tensor(lens[:1] if self.kind == "decode" else lens, device=device, dtype=torch.int32)
            ops.attention_decode(q[:, 0], kv[:, :, :W], kv[:, :, W:], out, H, self.scale, work, k_new=new[:, :W],
                                 v_new=new[:, W:], length=length)
            return out
        out = torch.full((B, self.Q, W), float("nan"), device=device, dtype=torch.bfloat16)
        if self.kind == "extend":
            offs = [n - self.Q for n in self.lengths]
            qkv = torch.cat([q, torch.stack([kv[b, o:o + self.Q] for b, o in enumerate(offs)])], -1)
            for b, o in enumerate(offs):
                kv[b, o:o + self.Q] = float("nan")  # kv_append must write them
            length = torch.tensor(offs, device=device, dtype=torch.int32)
            ops.kv_append(qkv[:, :, W:], kv, length)
            ops.attention_extend(qkv[:, :, :W], kv[:, :, :W], kv[:, :, W:], out, H, self.scale, length)
            return out
        n = self.lengths[0]
        ops.attention(q, kv[:, :n, :W], kv[:, :n, W:], out, H, self.scale)
        return out


# ------------------------------------------------------------------------------------------------- the cases
def _exact_cases():
    c = {}
    for L in (1, 16, 192, 193, 224, 225, 256):  # head_dim 64, single-pass kernel, and the streaming kernel forced
        c[f"attn_hd64_Lkv{L}"] = lambda L=L: AttnExact(2, 3, 64, 130, L)
        c[f"attn_hd64_Lkv{L}_streaming"] = lambda L=L: AttnExact(2, 3, 64, 130, L, streaming=True)
    for L in (257, 1500, 4096):
        c[f"attn_hd64_Lkv{L}"] = lambda L=L: AttnExact(2, 3, 64, 130, L)
    for hd in (80, 96, 112, 128):
        for L in (1, 193, 1500):
            c[f"attn_hd{hd}_Lkv{L}"] = lambda hd=hd, L=L: AttnExact(2, 3, hd, 130, L)
    c["attn_hd128_Lkv4096"] = lambda: AttnExact(2, 3, 128, 130, 4096)
    for hd in (64, 128):  # B*H = 192 > 148 SMs
        for L in (193, 1500):
            c[f"attn_hd{hd}_Lkv{L}_B16H12"] = lambda hd=hd, L=L: AttnExact(16, 12, hd, 3, L)
        for L in (1, 128, 129, 1024, 4096):
            c[f"causal_hd{hd}_L{L}"] = lambda hd=hd, L=L: AttnExact(2, 3, hd, L, L, causal=True)
        for Lq, Lkv in ((5, 300), (300, 5)):
            c[f"causal_hd{hd}_{Lq}x{Lkv}"] = lambda hd=hd, Lq=Lq, Lkv=Lkv: AttnExact(2, 3, hd, Lq, Lkv, causal=True)
        c[f"bias_hd{hd}_130x300"] = lambda hd=hd: AttnExact(2, 3, hd, 130, 300, bias=True, seed=hd)
        cap = 1024
        for P in (1, 7, 128, 129, 300):
            offs = [0, 1, 127, 128, 129, cap - P]
            c[f"extend_hd{hd}_P{P}"] = lambda hd=hd, P=P, offs=offs, cap=cap: ExtendExact(6, 2, hd, P, offs, cap)
        for P in (7, 129):
            for o in (1, 129, cap - P):
                c[f"extend_shared_hd{hd}_P{P}_off{o}"] = \
                    lambda hd=hd, P=P, o=o, cap=cap: ExtendExact(2, 3, hd, P, [o, o], cap, shared=True)
        cap = 32768 + GUARD
        kc = decode_chunk(2, 3, cap)
        for n in (0, 1, kc - 1, kc, kc + 1, cap - 1, 32767):
            c[f"decode_hd{hd}_len{n}"] = lambda hd=hd, n=n, cap=cap: DecodeExact(2, 3, hd, cap, [n, n], shared=True)
        kc = decode_chunk(10, 2, cap)
        ragged = [32766, 0, 1, -1, kc - 1, kc, cap, kc + 1, cap - 1, 32767]
        c[f"decode_ragged_hd{hd}"] = lambda hd=hd, ragged=ragged, cap=cap: DecodeExact(10, 2, hd, cap, ragged)
        for B, H in ((2, 3), (40, 4)):
            cap = 1500 + GUARD
            for L in (1, 64, 1500, cap):
                c[f"cross_hd{hd}_B{B}H{H}_Lkv{L}"] = lambda hd=hd, B=B, H=H, L=L, cap=cap: \
                    DecodeExact(B, H, hd, cap, Lkv=L)
    cap = 2048 + GUARD  # B*H = 160 > 148 SMs
    kc = decode_chunk(40, 4, cap)
    for n in (0, 1, kc - 1, kc, kc + 1, cap - 1):
        c[f"decode_hd64_B40H4_len{n}"] = lambda n=n, cap=cap: DecodeExact(40, 4, 64, cap, [n] * 40, shared=True)
    return c


def _planted_cases():
    c = {}
    for where in ("first", "last"):
        for hd in (64, 128):
            for n in (4096, 32767):
                c[f"planted_decode_hd{hd}_keys{n}_{where}"] = \
                    lambda hd=hd, n=n, where=where: Planted("decode", 2, 3, hd, [n - 1, n - 1], where, seed=n + hd)
                c[f"planted_cross_hd{hd}_Lkv{n}_{where}"] = \
                    lambda hd=hd, n=n, where=where: Planted("cross", 2, 3, hd, [n, n], where, seed=n + hd + 1)
            c[f"planted_ragged_hd{hd}_{where}"] = \
                lambda hd=hd, where=where: Planted("ragged", 3, 2, hd, [4095, 32766, 700], where, seed=hd + 2)
            for n in (1500, 4096):
                kind = "stream" if hd == 64 else "wide"
                c[f"planted_{kind}_hd{hd}_Lkv{n}_{where}"] = \
                    lambda hd=hd, n=n, where=where, kind=kind: Planted(kind, 2, 3, hd, [n], where, seed=n + hd + 3)
            c[f"planted_extend_hd{hd}_{where}"] = \
                lambda hd=hd, where=where: Planted("extend", 2, 3, hd, [1500, 4096], where, seed=hd + 4)
    return c


EXACT_CASES = _exact_cases()
PLANTED_CASES = _planted_cases()
