"""Bit-exact checks of the axial attention kernels against float64, on data whose softmax is exact.

Softmax cannot use the integer trick of test_exact_gpu.py in general, but it can where the logits are far apart:
when the winning logit of a row exceeds every other logit of the row by at least 128, ``exp`` of each other logit
(relative to the row maximum) is below 2^-184 and underflows to exactly 0 in fp32, for ``expf`` and for
``__expf`` alike, while the winners get ``exp(0) = 1``.  Attention is then exactly one-hot, or exactly 2^-m on 2^m
tied winners, in fp32 and after the tensor-core kernel's rounding of it to bf16.  ``out = attn . v`` and
``kv = skew(attn) . rv`` are then dyadic sums of small integers, exact in fp32 in any order, and each kernel must
store ``ref64.float().to(dtype)``.

The cases build q and k from 8-dimensional +-1 codes (two distinct codes have a dot product of at most 6, a code
with itself 8) and use sim scales that are multiples of 64, so every logit is a multiple of 128 and a unique
maximum is 128 clear of the rest.  One case per term of ``sim`` isolates it:

- dots: ``k[j]`` carries the code of its group (groups of 1, 2, 4, 8 or 16 tied keys), ``q[d]`` the code of the
  group row d selects;
- qr: ``rq[:, r]`` carries a distinct code per offset r, ``q[d]`` the code of ``r* = d - j* + L - 1``;
- kr: the same through ``k[d]`` (the KR term uses k at the row position d) and ``rk``;
- combined: all three scales non-zero and different per head (a permutation of 64, 128, 192), and in at least half
  of the rows the winners stop winning once two scale roles are swapped;
- uniform: ``q = k = 0`` with L a power of two, so attention is exactly 1/L;
- rounding: the dots pattern with wide v / rv / affine values, so at least a third of the outputs round to bf16.

In the dots, qr and kr cases row d of sequence s selects key ``j* = (d + c[s, head]) mod L``; with at least L
sequences of distinct offsets every key column wins in some row of every 16-row block, and every offset r in
[0, 2L-2] is used.  The combined case draws q until every row has such a winner set.

The fp32 CUDA-core kernel on the same data is the control: if it is not exact, the harness is wrong.  Each case
runs the bf16 kernel that ``eds_axial_attention`` picks, the bf16 CUDA-core kernel (through a ``qk`` view at a
2-byte offset, which the tensor-core kernel declines), with ReLU off and on.

The premise checks (exactness of the expected values, logit gaps, coverage, and that each fault model of the
reference changes an expected element) run on the CPU without a GPU; everything else is marked ``gpu``.
"""
import itertools
import math
from collections import namedtuple

import pytest
import torch
import torch.nn.functional as F

from eyediseasesegmentation_b200 import _lib, kernels as K
from test_exact_gpu import (_hist, big_memory, expected, guard_intact, guarded, nan_free, seed_of,  # noqa: F401
                            TWO31, DEV)

GAP = 128                   # every non-winning logit is at least this far below the row maximum
FP32_TINY = 2.0 ** -150     # exp() results at or below this round to 0 in fp32


# ------------------------------------------------------------------------------------------------ reference
def attention_ref64(q, k, v, rel, sim_scale, out_scale, out_shift, relu=False, parts=False, drop=None,
                    shift=None, kr_at_j=False):
    """The kernels' operation in float64.  q, k [S, heads, L, dqk], v [S, heads, L, dv]; rel [2 dqk + dv, 2L - 1];
    sim_scale [heads, 3] (qr, kr, dots); out_scale / out_shift [2, heads * dv] (kv, out).  Returns y [S, L, heads * dv]
    (channel head * dv + i), and with parts=True also attn [S, heads, L, L], sum_j attn |rv| and sum_j attn |v|
    ([S, L, heads * dv]).

    softmax: exp terms at or below 2^-150 are 0, as they are in fp32; on random data this changes nothing.
    The fault models: drop = (s, head, d, j) removes one key of one row; shift = {"qr" | "kr" | "rv": +-1} reads that
    table at r + shift (clamped); kr_at_j takes the KR term with k[j] instead of k[d]."""
    q, k, v, rel = q.double(), k.double(), v.double(), rel.double()
    S, heads, L, dqk = q.shape
    dv = v.shape[-1]
    ar = torch.arange(L, device=q.device)
    r = ar.view(L, 1) - ar.view(1, L) + L - 1                                  # [d, j]
    sh = shift or {}

    def table(lo, hi, name):
        return rel[lo:hi][:, (r + sh.get(name, 0)).clamp(0, 2 * L - 2)]       # [c, d, j]

    rq, rk, rv = table(0, dqk, "qr"), table(dqk, 2 * dqk, "kr"), table(2 * dqk, 2 * dqk + dv, "rv")
    qr = torch.einsum("shdi,idj->shdj", q, rq)
    kr = (torch.einsum("shji,idj->shdj", k, rk) if kr_at_j else torch.einsum("shdi,idj->shdj", k, rk))
    dots = torch.einsum("shdi,shji->shdj", q, k)
    sc = sim_scale.double().view(1, heads, 3, 1, 1)
    sim = sc[:, :, 0] * qr + sc[:, :, 1] * kr + sc[:, :, 2] * dots
    if drop is not None:
        sim[drop] = -math.inf
    e = torch.exp(sim - sim.amax(-1, keepdim=True))
    e = torch.where(e <= FP32_TINY, torch.zeros_like(e), e)
    attn = e / e.sum(-1, keepdim=True)
    out = torch.einsum("shdj,shji->sdhi", attn, v).reshape(S, L, heads * dv)
    kv = torch.einsum("shdj,idj->sdhi", attn, rv).reshape(S, L, heads * dv)
    osc, osh = out_scale.double().view(2, -1), out_shift.double().view(2, -1)
    y = (osc[0] * kv + osh[0]) + (osc[1] * out + osh[1])
    if relu:
        y = y.clamp_min(0)
    if not parts:
        return y
    arv = torch.einsum("shdj,idj->sdhi", attn, rv.abs()).reshape(S, L, heads * dv)
    av = torch.einsum("shdj,shji->sdhi", attn, v.abs()).reshape(S, L, heads * dv)
    return y, attn, arv, av, sim


def seq_to_map(t, axis, N, H, W):
    """[S, L, C] sequences -> [N, H, W, C]; axis 0: s = n W + w along h, axis 1: s = n H + h along w."""
    C = t.shape[-1]
    return t.reshape(N, W, H, C).permute(0, 2, 1, 3) if axis == 0 else t.reshape(N, H, W, C)


def map_to_seq(t, axis):
    N, H, W, C = t.shape
    return t.permute(0, 2, 1, 3).reshape(N * W, H, C) if axis == 0 else t.reshape(N * H, W, C)


# ------------------------------------------------------------------------------------------------ routing
def mma_accepts(heads, dqk, dv, L, aligned=True):
    """The shape rule of axial_attention_mma_try (bf16 only): heads % 4 == 0, dqk == 8, dv in {8, 16, 64},
    1 <= L <= 64, 16-byte aligned pointers."""
    return heads % 4 == 0 and dqk == 8 and dv in (8, 16, 64) and 1 <= L <= 64 and aligned


# ------------------------------------------------------------------------------------------------ cases
# N x H x W map, attention along `axis`, `heads` heads of dqk / dv channels, v separate when cross.
Cfg = namedtuple("Cfg", "N H W axis heads dv cross dqk", defaults=(8,))


def cfg_L(c):
    return c.H if c.axis == 0 else c.W


def cfg_seqs(c):
    return c.N * (c.W if c.axis == 0 else c.H)


def _other(L):
    """The map's other side: at least L sequences over N = 2 maps, and never equal to L."""
    o = max(3, (L + 1) // 2 + 1)
    return o + 1 if o == L else o


def _cfg(L, heads, dv, cross, axis, dqk=8):
    o = _other(L)
    return Cfg(2, L, o, 0, heads, dv, cross, dqk) if axis == 0 else Cfg(2, o, L, 1, heads, dv, cross, dqk)


# Every L class of the tensor-core kernel (LP = 16 / 32 / 48 / 64 and every ragged last row block), with dv, heads,
# self / cross attention and the axis cycling through their values.
TC_LS = [1, 8, 15, 16, 17, 19, 31, 32, 33, 38, 47, 48, 63, 64]
TC_CFGS = {f"L{L}_h{h}_dv{dv}_{'cross' if x else 'self'}_ax{a}": _cfg(L, h, dv, x, a)
           for i, L in enumerate(TC_LS)
           for h, dv, x, a in [((4, 8, 12)[i % 3], (8, 16, 64)[(i // 3) % 3], i % 2 == 1, (i // 2) % 2)]}
TC_CFGS.update({
    "L64_h12_dv64_cross_ax1": _cfg(64, 12, 64, True, 1),
    "L32_h8_dv8_self_ax0": _cfg(32, 8, 8, False, 0),
    "L19_h12_dv16_cross_ax0": _cfg(19, 12, 16, True, 0),
})
# shapes the tensor-core kernel declines: L > 64, heads % 4 != 0, dv outside {8, 16, 64}, dqk != 8
SIMT_CFGS = {
    "L65_h4_dv16_self_ax0": _cfg(65, 4, 16, False, 0),
    "L100_h8_dv8_cross_ax1": _cfg(100, 8, 8, True, 1),
    "L128_h4_dv64_self_ax1": _cfg(128, 4, 64, False, 1),
    "L19_h1_dv32_self_ax1": _cfg(19, 1, 32, False, 1),
    "L32_h2_dv4_cross_ax0": _cfg(32, 2, 4, True, 0),
    "L17_h3_dv1_self_ax0": _cfg(17, 3, 1, False, 0),
    "L8_h4_dv16_dqk4_cross_ax1": _cfg(8, 4, 16, True, 1, dqk=4),
    "L33_h4_dv8_dqk16_self_ax0": _cfg(33, 4, 8, False, 0, dqk=16),
    "L64_h8_dv64_dqk16_cross_ax1": _cfg(64, 8, 64, True, 1, dqk=16),
}
# the benchmark's two attention shapes at 48 maps (built on the device: too large for a CPU reference)
BENCH_CFGS = {
    "mhsa_48x64x64_h8_dv64": Cfg(48, 64, 64, 1, 8, 64, False),
    "mhca_48x64x64_h4_dv16": Cfg(48, 64, 64, 0, 4, 16, True),
}
SMALL_CFGS = {**TC_CFGS, **SIMT_CFGS}

KINDS = ("dots", "qr", "kr", "combined", "uniform", "rounding")


def kinds_for(c):
    L = cfg_L(c)
    # (4-dimensional codes leave too few logit values for the combined case)
    ks = ["dots", "combined", "rounding"] if L > 1 and c.dqk >= 8 else ["dots", "rounding"]
    if 2 * L - 1 <= 1 << c.dqk:                # a distinct code for every offset r
        ks[1:1] = ["qr", "kr"]
    if L & (L - 1) == 0:
        ks.append("uniform")
    return ks


Case = namedtuple("Case", "q k v rel sim_scale out_scale out_shift")


def _gen(seed, device):
    return torch.Generator(device=device).manual_seed(seed)


def _ints(shape, lo, hi, g, device):
    return torch.randint(lo, hi + 1, shape, generator=g, device=device).double()


def _codes(n, dqk, g, device, distinct=True):
    """n +-1 codes of dqk dimensions (distinct ones when asked)."""
    idx = torch.randperm(1 << dqk, generator=g, device=device)[:n] if distinct else \
        torch.randint(0, 1 << dqk, (n,), generator=g, device=device)
    bits = (idx.view(-1, 1) >> torch.arange(dqk, device=device)) & 1
    return (2 * bits - 1).double()


def _targets(S, heads, L, g, device):
    """The selected key of every row: j*(s, h, d) = (d + c[s, h]) mod L, c[s, h] = (s + off[h]) mod L."""
    off = torch.randperm(L, generator=g, device=device).repeat(-(-heads // L))[:heads]   # adjacent heads differ
    c = (torch.arange(S, device=device).view(S, 1) + off.view(1, heads)) % L
    return (torch.arange(L, device=device).view(1, 1, L) + c.view(S, heads, 1)) % L       # [S, heads, L]


def _pow2_partition(L, heads, g):
    """Per head: group sizes from {1, 2, 4, 8, 16}, at most L / 2 (one group of all keys would be uniform), summing
    to L, drawn at random."""
    out = []
    for _ in range(heads):
        sizes, left = [], L
        while left:
            opts = [p for p in (1, 2, 4, 8, 16) if p <= left and (p == 1 or 2 * p <= L)]
            sizes.append(opts[int(torch.randint(0, len(opts), (1,), generator=g, device=g.device))])
            left -= sizes[-1]
        out.append(sizes)
    return out


SWAPS = [(1, 0, 2), (2, 1, 0), (0, 2, 1)]          # (qr, kr, dots) with two scale roles exchanged
COMBINED_MOVED = 0.5                               # share of rows whose winners lose under each swap


def _combined_q(k, rq, rk, alpha, g, device, rounds=24, max_rounds=400):
    """q for the combined case (alpha [heads, 3] are the scales / 64): the q rows are redrawn until each row has a
    power-of-two winner set, and for `rounds` rounds also while a winner still wins with two scale roles swapped."""
    S, heads, L, dqk = k.shape
    k, rq, rk = k.float(), rq.float(), rk.float()
    q = (2 * torch.randint(0, 2, k.shape, generator=g, device=device) - 1).float()
    ar = torch.arange(L, device=device)
    r = ar.view(L, 1) - ar.view(1, L) + L - 1
    kr = torch.einsum("shdi,idj->shdj", k, rk[:, r])
    for it in range(max_rounds):
        qr = torch.einsum("shdi,idj->shdj", q, rq[:, r])
        dots = torch.einsum("shdi,shji->shdj", q, k)
        terms = torch.stack([qr, kr, dots], 2)                               # [S, h, 3, L, L]
        a = alpha.float().view(1, heads, 3, 1, 1)
        sim = (a * terms).sum(2)
        win = sim == sim.amax(-1, keepdim=True)
        n = win.sum(-1)
        ok = (n & (n - 1)) == 0
        if it < rounds:
            for p in SWAPS:
                sw = (a[:, :, list(p)] * terms).sum(2)
                ok &= ~(win & (sw == sw.amax(-1, keepdim=True))).any(-1)
        if bool(ok.all()):
            return q.double()
        bad = ~ok
        fresh = (2 * torch.randint(0, 2, q.shape, generator=g, device=device) - 1).float()
        q = torch.where(bad.unsqueeze(-1), fresh, q)
    raise AssertionError("combined case: some rows have no power-of-two winner set")


def make_case(c, kind, seed, device="cpu"):
    """The operands of one case, float64 on `device`: q, k [S, heads, L, dqk], v [S, heads, L, dv], rel, scales."""
    g = _gen(seed, device)
    S, L, heads, dqk, dv = cfg_seqs(c), cfg_L(c), c.heads, c.dqk, c.dv
    R = 2 * L - 1
    CO = heads * dv
    wide = kind == "rounding"
    vr = 100 if wide else 3
    v = _ints((S, heads, L, dv), -vr, vr, g, device)
    rel = torch.cat([_codes(R, dqk, g, device, distinct=False).t(), _codes(R, dqk, g, device, distinct=False).t(),
                     _ints((dv, R), -vr, vr, g, device)], 0)
    sr = (9, 300) if wide else (2, 4)
    out_scale = _ints((2, CO), 1, sr[0], g, device) * (2 * _ints((2, CO), 0, 1, g, device) - 1)
    out_shift = _ints((2, CO), -sr[1], sr[1], g, device)
    rand_codes = lambda: (2 * torch.randint(0, 2, (S, heads, L, dqk), generator=g, device=device) - 1).double()  # noqa
    q, k = rand_codes(), rand_codes()
    scale = torch.zeros(heads, 3, dtype=torch.float64, device=device)
    tgt = _targets(S, heads, L, g, device)
    d = torch.arange(L, device=device).view(1, 1, L)
    if kind in ("dots", "rounding"):
        # keys grouped (sizes 1 .. 16, a power of two each), key slots permuted per (sequence, head)
        parts = _pow2_partition(L, heads, g)
        ng = max(len(p) for p in parts)
        assert ng <= 1 << dqk
        slot_group = torch.tensor([sum(([gi] * s for gi, s in enumerate(p)), []) for p in parts],
                                  device=device)                                        # [heads, L]
        perm = torch.rand(S, heads, L, generator=g, device=device).argsort(-1)          # slot -> key
        group = torch.empty_like(perm)
        group.scatter_(-1, perm, slot_group.view(1, heads, L).expand(S, heads, L))      # key -> group
        codes = torch.stack([_codes(ng, dqk, g, device) for _ in range(heads)])         # [heads, ng, dqk]
        hidx = torch.arange(heads, device=device).view(1, heads, 1)
        k = codes[hidx, group]
        q = codes[hidx, group.gather(-1, tgt)]
        scale[:, 2] = 64
    elif kind in ("qr", "kr"):
        codes = _codes(R, dqk, g, device)                                               # distinct per offset
        lo = 0 if kind == "qr" else dqk
        rel[lo:lo + dqk] = codes.t()
        sel = codes[d - tgt + L - 1]                                                    # [S, heads, L, dqk]
        if kind == "qr":
            q = sel
        else:
            k = sel
        scale[:, 0 if kind == "qr" else 1] = 64
    elif kind == "combined":
        roles = list(itertools.permutations((1, 2, 3)))
        alpha = torch.tensor([roles[(h + seed) % 6] for h in range(heads)], dtype=torch.float64, device=device)
        q = _combined_q(k, rel[:dqk], rel[dqk:2 * dqk], alpha, g, device)
        scale = 64 * alpha
    elif kind == "uniform":
        q, k = torch.zeros_like(q), torch.zeros_like(k)
        scale = 64 * _ints((heads, 3), 1, 3, g, device)
    else:
        raise ValueError(kind)
    return Case(q, k, v, rel, scale, out_scale, out_shift)


def case_ref(case, relu=False, parts=False, **fault):
    return attention_ref64(case.q, case.k, case.v, case.rel, case.sim_scale, case.out_scale, case.out_shift,
                           relu=relu, parts=parts, **fault)


def case_maps(c, case, dtype, device=DEV, misalign=False):
    """qk (and v for cross attention) maps in `dtype` on `device`; misalign: qk is a view 2 bytes into its buffer."""
    S, heads, L, _ = case.q.shape
    parts = [case.q, case.k] if c.cross else [case.q, case.k, case.v]
    qk_seq = torch.cat(parts, -1).permute(0, 2, 1, 3).reshape(S, L, -1)               # [S, L, heads * G]
    qk = seq_to_map(qk_seq.to(device=device, dtype=dtype), c.axis, c.N, c.H, c.W).contiguous()
    if misalign:
        buf = torch.empty(qk.numel() + 1, dtype=dtype, device=device)
        buf[1:].copy_(qk.view(-1))
        qk = buf[1:].view(qk.shape)
        assert qk.data_ptr() % 16 != 0
    v = None
    if c.cross:
        v = seq_to_map(case.v.permute(0, 2, 1, 3).reshape(S, L, -1).to(device=device, dtype=dtype), c.axis,
                       c.N, c.H, c.W).contiguous()
    return qk, v


def f32(t, device=DEV):
    return t.to(device=device, dtype=torch.float32).contiguous()


def run_attention(c, case, qk, v, relu, out):
    return K.axial_attention(qk, v, c.axis, c.heads, c.dqk, c.dv, f32(case.rel), f32(case.sim_scale),
                             f32(case.out_scale), f32(case.out_shift), relu, out=out)


# ------------------------------------------------------------------------------------------------ reporting
def attention_mismatch_report(got, want, heads, dv, limit=8):
    """None when got == want bit for bit, else where the differing elements are.  got / want: [S, L, heads * dv]."""
    if tuple(got.shape) != tuple(want.shape):
        return f"shape {tuple(got.shape)} != {tuple(want.shape)}"
    if torch.equal(got, want):
        return None
    bad = (got != want).cpu()
    S, L, CO = bad.shape
    count = int(bad.sum())
    nan = int(torch.isnan(got.float()).sum())
    lines = [f"{count} of {bad.numel()} elements differ ({nan} NaN: never written)"]
    for s, d, ch in bad.nonzero()[:limit].tolist():
        lines.append(f"  (sequence {s}, head {ch // dv}, row d={d} in 16-row block {d // 16}, channel {ch % dv}): "
                     f"got {float(got[s, d, ch])}, want {float(want[s, d, ch])}")
    per_d = bad.sum((0, 2))
    per_block = torch.zeros((L + 15) // 16, dtype=torch.long).index_add_(0, torch.arange(L) // 16, per_d)
    per_head = bad.sum((0, 1)).view(heads, dv).sum(1)
    lines.append(f"by 16-row block: {_hist(per_block)}")
    lines.append(f"by head: {_hist(per_head)}")
    lines.append(f"by channel within the head: {_hist(bad.sum((0, 1)).view(heads, dv).sum(0), 16)}")
    lines.append(f"sequences: {_hist(bad.sum((1, 2)))}")
    return "\n".join(lines)


# ------------------------------------------------------------------------------------------------ premise (CPU)
def winners(sim):
    return sim == sim.amax(-1, keepdim=True)


def bf16_rounded_fraction(ref):
    return float((ref != ref.float().bfloat16().double()).double().mean())


# the fault models of the reference that each kind must be able to show
FAULTS = {
    "dots": ["drop", "rv-1", "rv+1", "shift_dropped"],
    "rounding": ["drop", "rv-1", "rv+1", "shift_dropped"],
    "qr": ["drop", "qr-1", "qr+1", "rv-1", "rv+1", "shift_dropped"],
    "kr": ["drop", "kr-1", "kr+1", "kr_at_j", "rv-1", "rv+1", "shift_dropped"],
    "combined": ["drop", "qr-1", "qr+1", "kr-1", "kr+1", "kr_at_j", "rv-1", "rv+1", "heads_swapped",
                 "shift_dropped"],
    "uniform": ["drop", "rv-1", "rv+1", "shift_dropped"],
}


def faulty_ref(case, fault, win):
    if fault == "drop":
        s, h, d, j = win.nonzero()[0].tolist()                       # a winner key of some row
        return case_ref(case, drop=(s, h, d, j))
    if fault[:2] in ("qr", "kr", "rv") and fault[2:] in ("-1", "+1"):
        return case_ref(case, shift={fault[:2]: int(fault[2:])})
    if fault == "kr_at_j":
        return case_ref(case, kr_at_j=True)
    if fault == "heads_swapped":
        sc = case.sim_scale.clone()
        sc[[0, 1]] = sc[[1, 0]]
        return case_ref(case._replace(sim_scale=sc))
    if fault == "shift_dropped":
        return case_ref(case._replace(out_shift=torch.zeros_like(case.out_shift)))
    raise ValueError(fault)


SMALL_MATRIX = [(name, kind) for name, c in SMALL_CFGS.items() for kind in kinds_for(c)]


@pytest.mark.parametrize("name,kind", SMALL_MATRIX, ids=[f"{n}-{k}" for n, k in SMALL_MATRIX])
def test_case_premises(name, kind):
    """Exact expected values, logit gaps >= 128, power-of-two winner sets, coverage of every key column in every
    16-row block and of every offset r, per-head patterns, and sensitivity to each fault model."""
    c = SMALL_CFGS[name]
    case = make_case(c, kind, seed_of(name + kind))
    S, heads, L, _ = case.q.shape
    ref, attn, _, _, sim = case_ref(case, parts=True)
    expected(ref, torch.float32)                                     # asserts exactness in fp32
    expected(ref.clamp_min(0), torch.float32)
    win = winners(sim)
    n = win.sum(-1)
    assert bool(((n & (n - 1)) == 0).all()), "a winner set is not a power of two"
    if kind == "uniform":
        assert bool((n == L).all())
    else:
        gap = (sim.amax(-1, keepdim=True) - sim.masked_fill(win, -math.inf)).amin(-1)
        assert L == 1 or float(gap.min()) >= GAP, f"logit gap {float(gap.min())} < {GAP}"
        if kind in ("dots", "qr", "kr", "rounding"):
            ar = torch.arange(L)
            r = ar.view(L, 1) - ar.view(1, L) + L - 1
            for h in range(heads):
                for b in range(0, L, 16):
                    cover = win[:, h, b:b + 16].any(0).any(0)        # over sequences and the block's rows
                    assert bool(cover.all()), f"head {h}, block {b // 16}: keys {(~cover).nonzero().view(-1)}"
                hit = torch.zeros(2 * L - 1, dtype=torch.bool)
                hit[r[win[:, h].any(0)]] = True
                assert bool(hit.all()), f"head {h}: offsets {(~hit).nonzero().view(-1)} never win"
        if heads > 1 and L > 1:
            for h in range(heads - 1):
                assert not torch.equal(win[:, h], win[:, h + 1]), f"heads {h} and {h + 1} share their pattern"
        if kind == "combined":
            sc = case.sim_scale
            assert bool((sc > 0).all()) and all(len(set(row.tolist())) == 3 for row in sc)
            for p in SWAPS:                      # most rows lose their winners with two scale roles swapped
                _, _, _, _, sim2 = case_ref(case._replace(sim_scale=sc[:, list(p)].contiguous()), parts=True)
                moved = ~(win & winners(sim2)).any(-1)
                assert float(moved.double().mean()) >= COMBINED_MOVED, f"scale roles {p}: {float(moved.double().mean())}"
    if kind == "rounding":
        assert bf16_rounded_fraction(ref) >= 1 / 3
    elif kind != "uniform":                  # (a mean over L keys needs log2(L) fraction bits)
        assert 1 - bf16_rounded_fraction(ref) >= 0.9, "too coarse to see one term"
    few = slice(0, 4)                        # the fault models on the first sequences
    case = Case(case.q[few], case.k[few], case.v[few], *case[3:])
    want = expected(ref[few], torch.bfloat16)
    win = win[few]
    for fault in FAULTS[kind]:
        if (fault == "heads_swapped" and heads < 2) or (L == 1 and fault != "shift_dropped"):
            continue                         # one key, one offset: nothing to drop or shift
        bad = faulty_ref(case, fault, win)
        if fault == "drop":
            bad = torch.nan_to_num(bad, nan=1e9)                     # a row with its only key dropped
        assert not torch.equal(bad.float().bfloat16(), want), f"fault {fault} leaves every expected value"


def test_mismatch_report_names_sequence_head_row_block_and_channel():
    want = torch.zeros(5, 40, 3 * 8)
    got = want.clone()
    got[:, 17, 8 + 2] = 1                                            # head 1, channel 2, row 17 (block 1)
    got[2, 33, 0] = float("nan")
    msg = attention_mismatch_report(got, want, 3, 8)
    assert msg.startswith("6 of 4800 elements differ (1 NaN")
    assert "(sequence 0, head 1, row d=17 in 16-row block 1, channel 2)" in msg
    assert "by 16-row block: {1: 5, 2: 1}" in msg and "by head: {0: 1, 1: 5}" in msg
    assert attention_mismatch_report(want, want.clone(), 3, 8) is None


def test_reference_matches_the_oracle_attend():
    """The float64 restatement agrees with oracle.nets._attend (pinned to AxialAttention / CrossAxialAttention) on
    random float64 data, with the BatchNorms built from scale and shift (running_mean 0, running_var 1 - 1e-5)."""
    from oracle import nets
    g = torch.Generator().manual_seed(3)
    for (S, heads, L, dqk, dv) in [(3, 4, 19, 8, 16), (2, 8, 32, 8, 8), (2, 2, 7, 4, 5)]:
        qkv = torch.randn(S, heads, L, 2 * dqk + dv, generator=g, dtype=torch.float64)
        v_cross = torch.randn(S, heads, L, dv, generator=g, dtype=torch.float64)
        q, k = qkv[..., :dqk], qkv[..., dqk:2 * dqk]
        for cross, v in ((False, qkv[..., 2 * dqk:]), (True, v_cross)):
            rel = torch.randn(2 * dqk + dv, 2 * L - 1, generator=g, dtype=torch.float64)
            sim_scale = torch.randn(heads, 3, generator=g, dtype=torch.float64)
            out_scale = torch.randn(2, heads * dv, generator=g, dtype=torch.float64)
            out_shift = torch.randn(2, heads * dv, generator=g, dtype=torch.float64)
            p = "att"
            sd = {p + ".RelativePosEncQKV.relative": rel}
            for name, w, b in (("attention_norm", sim_scale.reshape(-1), torch.randn(3 * heads, generator=g,
                                                                                       dtype=torch.float64)),
                               ("out_norm", out_scale.reshape(-1), out_shift.reshape(-1))):
                sd[f"{p}.{name}.weight"], sd[f"{p}.{name}.bias"] = w, b
                sd[f"{p}.{name}.running_mean"] = torch.zeros_like(w)
                sd[f"{p}.{name}.running_var"] = torch.full_like(w, 1 - 1e-5)
            oracle = nets._attend(sd, p, q.transpose(2, 3), k.transpose(2, 3), v.transpose(2, 3), L, heads, dqk, dv)
            ours = attention_ref64(q, k, v, rel, sim_scale, out_scale, out_shift)     # [S, L, heads * dv]
            assert (ours - oracle.transpose(1, 2)).abs().max().item() < 1e-12, (S, heads, L, cross)


# ------------------------------------------------------------------------------------------------ random data: bound
# The shapes of test_kernels_gpu.test_axial_attention: N, H, W, heads, dv (dqk = 8).
RANDOM_SHAPES = [(2, 16, 16, 4, 16), (1, 64, 64, 8, 64), (2, 32, 32, 4, 16), (1, 19, 19, 8, 64), (1, 38, 38, 4, 8),
                 (1, 24, 40, 4, 16), (1, 8, 8, 8, 64), (1, 16, 16, 2, 16)]
U_BF16 = 2.0 ** -8          # unit roundoff of bf16 (8 significant bits)
EPS32 = 2.0 ** -24          # unit roundoff of fp32


def random_case(shape, axis, cross, dtype):
    """The random operands of test_axial_attention on the CPU: (Cfg, Case, qk map, v map); q / k / v are the values
    the kernel reads (rounded to `dtype`), and rel is rounded to bf16 where the tensor-core kernel runs, which
    rounds it when staging it."""
    N, H, W, heads, dv = shape
    dqk = 8
    L = H if axis == 0 else W
    G = 2 * dqk + (0 if cross else dv)

    def rnd(*sh, seed, scale=1.0):
        return torch.randn(*sh, generator=torch.Generator().manual_seed(seed)) * scale

    qk = rnd(N, H, W, heads * G, seed=40, scale=0.5).to(dtype)
    vt = rnd(N, H, W, heads * dv, seed=41, scale=0.5).to(dtype) if cross else None
    rel = rnd(2 * dqk + dv, 2 * L - 1, seed=42, scale=0.5)
    c = Cfg(N, H, W, axis, heads, dv, cross, dqk)
    if dtype == torch.bfloat16 and mma_accepts(heads, dqk, dv, L):
        rel = rel.bfloat16().float()
    x = map_to_seq(qk, axis).double().reshape(-1, L, heads, G).permute(0, 2, 1, 3)
    v = (map_to_seq(vt, axis).double().reshape(-1, L, heads, dv).permute(0, 2, 1, 3) if cross else x[..., 2 * dqk:])
    case = Case(x[..., :dqk], x[..., dqk:2 * dqk], v, rel, rnd(heads, 3, seed=43, scale=0.3),
                rnd(2, heads * dv, seed=44), rnd(2, heads * dv, seed=45))
    return c, case, qk, vt


def error_bound(case, ref, arv, av, dtype, tensor_core):
    """Per-element bound on |y - ref| for a correct kernel (ref: float64 on the operands the kernel reads).

    Both kernels compute sim, the softmax, attn . v, attn . rv and the affine epilogue in fp32 (unit roundoff e), and
    round once more when they store a bf16 y (unit roundoff u = 2^-8).  The tensor-core kernel also rounds each
    attention probability to bf16 before the two products: p~ = p (1 + d), |d| <= u.  To first order:
      - sim: each of the three dqk-term dot products and their scaled sum lose at most (dqk + 2) e M, where M is the
        row's largest |a_qr| sum|q rq| + |a_kr| sum|k rk| + |a_dots| sum|q k|; a softmax moves each p_j by at most
        2 max|d sim| relative to p_j, and the exponent's argument (|sim - max| <= 2M) adds 2M e, __expf's error
        (2 + 1.2 |x|) ulp adds (2.4 M + 2) e;
      - the row sum (at most L / 32 + 5 additions per lane and shuffle), the reciprocal and the product add
        (L / 32 + 7) e relative to p_j;
      - attn . x over L terms in fp32 adds L e of sum_j p_j |x_j|.
    Together |kv~ - kv| <= d_p sum_j p_j |rv_j| with d_p = u [tensor core] + ((2 dqk + 11) M + 2 L + 14) e, and the
    same for out.  The epilogue adds a few e of |a kv| + |c_kv| + |a out| + |c_out| (below 1e-6 for these values),
    the store adds u |y| (u = e for an fp32 y), and ReLU is 1-Lipschitz.  Hence
      |y - ref| <= u_store |ref| + d_p (|a_kv| sum_j attn |rv| + |a_out| sum_j attn |v|) + 1e-6.
    For the bf16 tensor-core kernel d_p stays below 1.25 u on these shapes (asserted)."""
    S, heads, L, dqk = case.q.shape
    dv = case.v.shape[-1]
    absc = Case(case.q.abs(), case.k.abs(), case.v.abs(), case.rel.abs(), case.sim_scale.abs(),
                case.out_scale.abs(), case.out_shift.abs())
    M = case_ref(absc, parts=True)[4].amax(-1)                                          # [S, heads, L]
    d_p = ((2 * dqk + 11) * M + 2 * L + 14) * EPS32
    if tensor_core:
        assert float(d_p.max()) <= 0.25 * U_BF16
        d_p = d_p + U_BF16
    d_p = d_p.permute(0, 2, 1).unsqueeze(-1).expand(S, L, heads, dv).reshape(S, L, heads * dv)
    osc = case.out_scale.double().abs().view(2, -1)
    u_store = U_BF16 if dtype == torch.bfloat16 else EPS32
    return u_store * ref.abs() + d_p * (osc[0] * arv + osc[1] * av) + 1e-6


@pytest.mark.parametrize("shape", RANDOM_SHAPES)
def test_random_data_bound_sees_one_dropped_key_and_an_offset_shift(shape):
    """On the data of test_axial_attention, dropping one (row, key) term from the softmax moves some output of that
    row past the bf16 bound at >= 99 % of 200 sampled positions, and so does reading rv at r +- 1."""
    c, case, _, _ = random_case(shape, 0, False, torch.bfloat16)
    S, heads, L, _ = case.q.shape
    tc = mma_accepts(heads, 8, c.dv, L)
    g = torch.Generator().manual_seed(7)
    caught = 0
    for _ in range(200):
        s, h, d, j = (int(torch.randint(0, n, (1,), generator=g)) for n in (S, heads, L, L))
        one = Case(case.q[s:s + 1], case.k[s:s + 1], case.v[s:s + 1], *case[3:])
        ref, _, arv, av, _ = case_ref(one, parts=True)
        bound = error_bound(one, ref, arv, av, torch.bfloat16, tc)
        moved = (case_ref(one, drop=(0, h, d, j)) - ref).abs()[0, d, h * c.dv:(h + 1) * c.dv]
        caught += bool((moved > bound[0, d, h * c.dv:(h + 1) * c.dv]).any())
    assert caught >= 198, f"{caught} of 200 dropped keys stay inside the bound"
    ref, _, arv, av, _ = case_ref(case, parts=True)
    bound = error_bound(case, ref, arv, av, torch.bfloat16, tc)
    for sh in (-1, 1):
        assert bool(((case_ref(case, shift={"rv": sh}) - ref).abs() > bound).any()), sh


# ------------------------------------------------------------------------------------------------ exact (GPU)
def _run_case(c, kind, case, ref, tag):
    """Every kernel on one case, ReLU off and on; returns the failure messages."""
    errors = []
    S, heads, L, _ = case.q.shape
    CO = heads * c.dv
    shape = (c.N, c.H, c.W, CO)
    qk32, v32 = case_maps(c, case, torch.float32)
    qk16, v16 = case_maps(c, case, torch.bfloat16)
    qk16m, _ = case_maps(c, case, torch.bfloat16, misalign=True)
    tc = mma_accepts(heads, c.dqk, c.dv, L)
    runs = [("fp32 CUDA-core, the control (when it is not exact, the harness is wrong)", torch.float32, qk32, v32),
            (f"bf16 {'tensor-core' if tc else 'CUDA-core'}", torch.bfloat16, qk16, v16),
            ("bf16 CUDA-core (qk at a 2-byte offset)", torch.bfloat16, qk16m, v16)]
    for relu in (False, True):
        r = ref.clamp_min(0) if relu else ref
        for what, dtype, qk, v in runs:
            out, guard = guarded(shape, dtype)
            run_attention(c, case, qk, v, relu, out)
            torch.cuda.synchronize()
            if not guard_intact(guard):
                errors.append(f"{tag} {kind} relu={relu}: {what} wrote past its output")
            msg = attention_mismatch_report(map_to_seq(out, c.axis), expected(r, dtype).to(out.device), heads, c.dv)
            if msg:
                errors.append(f"{tag} {kind} relu={relu}: {what}\n{msg}")
    return errors


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SMALL_CFGS))
def test_attention_exact(name):
    c = SMALL_CFGS[name]
    errors = []
    for kind in kinds_for(c):
        case = make_case(c, kind, seed_of(name + kind))
        errors += _run_case(c, kind, case, case_ref(case).to(DEV), f"{name} {c}")
    if errors:
        pytest.fail("\n".join(errors))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BENCH_CFGS))
def test_attention_exact_benchmark_shapes(name):
    """The MHSA and MHCA shapes of the benchmark at 48 maps; operands and reference on the device."""
    c = BENCH_CFGS[name]
    assert mma_accepts(c.heads, c.dqk, c.dv, cfg_L(c))
    errors = []
    for kind in ("dots", "qr", "kr", "combined", "uniform"):
        case = make_case(c, kind, seed_of(name + kind), device=DEV)
        ref, _, _, _, sim = case_ref(case, parts=True)
        win = winners(sim)
        if kind != "uniform":
            gap = (sim.amax(-1, keepdim=True) - sim.masked_fill(win, -math.inf)).amin(-1)
            assert float(gap.min()) >= GAP, (kind, float(gap.min()))
        del sim, win
        errors += _run_case(c, kind, case, ref, name)
    if errors:
        pytest.fail("\n".join(errors))


# ------------------------------------------------------------------------------------------------ routing
ROUTING = [(n, c, False) for n, c in SMALL_CFGS.items()] + [("L64_h8_dv64_self_misaligned", _cfg(64, 8, 64, False, 1),
                                                            True)]


def _profiled_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if "axial_attention" in e.name]


@pytest.mark.gpu
def test_routing_picks_the_tensor_core_kernel_exactly_where_it_accepts_the_shape():
    seen = set()
    errors = []
    for name, c, misalign in ROUTING:
        case = make_case(c, "uniform" if "uniform" in kinds_for(c) else "dots", seed_of("route" + name))
        qk, v = case_maps(c, case, torch.bfloat16, misalign=misalign)
        run_attention(c, case, qk, v, False, None)                    # warm-up: module load, smem opt-in
        names = _profiled_kernels(lambda: run_attention(c, case, qk, v, False, None))
        want = "axial_attention_mma_kernel" if mma_accepts(c.heads, c.dqk, c.dv, cfg_L(c), not misalign) else \
            "axial_attention_kernel"
        seen.add(want)
        if len(names) != 1 or want + "<" not in names[0]:
            errors.append(f"{name}: launched {names}, expected {want}")
    assert seen == {"axial_attention_mma_kernel", "axial_attention_kernel"}
    assert not errors, "\n".join(errors)


# ------------------------------------------------------------------------------------------------ rejections
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_shape_over_the_shared_memory_limit_is_rejected(dtype):
    """L = 150, dv = 64 needs 234,280 B of shared memory in the CUDA-core kernel (> 227 KB): EdsError, no launch."""
    c = _cfg(150, 4, 64, True, 1)
    L, dqk, dv = 150, 8, 64
    smem = 4 * (2 * dqk * L + L * dv + 2 * dqk * (2 * L - 1) + dv * (2 * L - 1) + L * (L + 1))
    assert smem > 227 * 1024
    case = make_case(c, "dots", 1)
    qk, v = case_maps(c, case, dtype)
    out, guard = guarded((c.N, c.H, c.W, c.heads * dv), dtype)

    def call():
        with pytest.raises(_lib.EdsError, match="shared memory"):
            run_attention(c, case, qk, v, False, out)
    names = _profiled_kernels(call)
    assert names == []
    assert bool(torch.isnan(out).all()) and guard_intact(guard)


# ------------------------------------------------------------------------------------------------ mhca_gate
def mhca_gate_ref64(ori, att):
    """ori * up2x_bilinear(sigmoid(att)); att in {-200, 0, 200}, where the fp32 sigmoid is exactly 0, 1/2 or 1."""
    sig = torch.where(att > 0, 1.0, torch.where(att < 0, 0.0, 0.5)).double()
    up = F.interpolate(sig.permute(0, 3, 1, 2), scale_factor=2, mode="bilinear", align_corners=False)
    return ori.double() * up.permute(0, 2, 3, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_mhca_gate_exact(dtype):
    """Gates are multiples of 1/32 (bilinear weights 1/4, 3/4 on {0, 1/2, 1}); odd h / w and h = 1 or w = 1 run the
    border clamps."""
    for N, h, w, C in [(2, 5, 7, 16), (1, 1, 6, 8), (3, 4, 1, 24), (1, 1, 1, 8), (2, 32, 32, 64)]:
        seed = seed_of(f"mhca{N}{h}{w}{C}")
        g = torch.Generator(device=DEV).manual_seed(seed)
        att = (200 * torch.randint(-1, 2, (N, h, w, C), generator=g, device=DEV)).to(dtype)
        ori = torch.randint(-64, 65, (N, 2 * h, 2 * w, C), generator=g, device=DEV).to(dtype)
        ref = mhca_gate_ref64(ori, att)
        out, guard = guarded(tuple(ori.shape), dtype)
        K.mhca_gate(ori, att, out=out)
        assert guard_intact(guard)
        want = expected(ref, dtype)
        if not torch.equal(out, want):
            bad = (out != want).nonzero()[:8].tolist()
            pytest.fail(f"mhca_gate {N}x{h}x{w}x{C}: {int((out != want).sum())} differ, e.g. (n, y, x, c) {bad}")


# ------------------------------------------------------------------------------------------------ past 2^31 elements
# One launch per kernel with a tensor of more than 2^31 elements; the per-image sizes do not divide 2^31.  The images
# holding element 2^31 and the last image are compared with float64, the whole output is checked for NaN.
BIG_TC = Cfg(830, 64, 64, 1, 8, 64, False)        # qk 830 x 64 x 64 x 640 = 2.18 G elements, out 1.74 G
BIG_SIMT = Cfg(4240, 63, 63, 1, 2, 64, True)      # heads 2: CUDA-core kernel; v and out 2.15 G elements each


def _big_qr_case(c, seed):
    """The qr pattern built straight into the [N, H, W, C] map (axis 1: the map is the sequence layout)."""
    g = _gen(seed, DEV)
    S, L, heads, dqk, dv = cfg_seqs(c), cfg_L(c), c.heads, c.dqk, c.dv
    R = 2 * L - 1
    G = 2 * dqk + (0 if c.cross else dv)
    codes = _codes(R, dqk, g, DEV)
    rel = torch.cat([codes.t(), _codes(R, dqk, g, DEV, distinct=False).t(), _ints((dv, R), -3, 3, g, DEV)], 0)
    qk = torch.empty(S, L, heads, G, dtype=torch.bfloat16, device=DEV)
    tgt = _targets(S, heads, L, g, DEV)                                                  # [S, heads, L]
    d = torch.arange(L, device=DEV).view(1, 1, L)
    for h in range(heads):                                                               # keeps temporaries small
        qk[:, :, h, :dqk] = codes[(d - tgt + L - 1)[:, h]].to(torch.bfloat16)
    qk[..., dqk:2 * dqk].random_(0, 2, generator=g).mul_(2).sub_(1)
    v = None
    if c.cross:
        v = torch.empty(c.N, c.H, c.W, heads * dv, dtype=torch.bfloat16, device=DEV).random_(-3, 4, generator=g)
    else:
        qk[..., 2 * dqk:].random_(-3, 4, generator=g)
    CO = heads * dv
    out_scale = _ints((2, CO), 1, 2, g, DEV)
    out_shift = _ints((2, CO), -4, 4, g, DEV)
    scale = torch.zeros(heads, 3, dtype=torch.float64, device=DEV)
    scale[:, 0] = 64
    return qk.view(c.N, c.H, c.W, heads * G), v, rel, scale, out_scale, out_shift


def _big_attention(c, seed):
    qk, v, rel, scale, osc, osh = _big_qr_case(c, seed)
    S, L, heads, dqk, dv = cfg_seqs(c), cfg_L(c), c.heads, c.dqk, c.dv
    CO = heads * dv
    out, guard = guarded((c.N, c.H, c.W, CO), torch.bfloat16)
    K.axial_attention(qk, v, c.axis, heads, dqk, dv, f32(rel), f32(scale), f32(osc), f32(osh), False, out=out)
    torch.cuda.synchronize()
    errors = []
    if not guard_intact(guard):
        errors.append("wrote past the output")
    if not nan_free(out):
        errors.append("left output elements unwritten (NaN)")
    big = [t for t in (qk, v, out) if t is not None and t.numel() > TWO31]
    imgs = sorted({TWO31 // t[0].numel() for t in big} | {c.N - 1})
    if not big or any(TWO31 % t[0].numel() == 0 for t in big):
        errors.append(f"case does not reach past 2^31 elements at an image boundary-free offset: {imgs}")
    print(f"axial_attention {c}: images {imgs} against float64")
    G = 2 * dqk + (0 if c.cross else dv)
    for n in imgs:
        seqs = slice(n * c.H, (n + 1) * c.H)
        x = qk[n].reshape(c.H, L, heads, G).permute(0, 2, 1, 3)
        vv = (v[n].reshape(c.H, L, heads, dv).permute(0, 2, 1, 3) if c.cross else x[..., 2 * dqk:])
        ref = attention_ref64(x[..., :dqk], x[..., dqk:2 * dqk], vv, rel, scale, osc, osh)
        got = map_to_seq(out[n:n + 1], c.axis)
        msg = attention_mismatch_report(got, expected(ref, torch.bfloat16), heads, dv)
        if msg:
            errors.append(f"image {n} (sequences {seqs.start}..{seqs.stop - 1}):\n{msg}")
    return "\n".join(errors) or None


@pytest.mark.gpu
@pytest.mark.parametrize("c", [BIG_TC, BIG_SIMT], ids=["tensor-core-qk", "cuda-core-v-out"])
def test_attention_past_2_31_elements(c, big_memory):
    assert mma_accepts(c.heads, c.dqk, c.dv, cfg_L(c)) == (c is BIG_TC)
    msg = _big_attention(c, seed_of(f"bigattn{c}"))
    if msg is not None:
        pytest.fail(msg)
