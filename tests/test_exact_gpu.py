"""Bit-exact checks of every convolution and data-movement kernel against float64.

Every convolution multiplies bf16 operands and accumulates in fp32.  The operands here are small integers
(bias and residual too; gates are multiples of 1/8, bilinear weights 1/4 and 3/4), chosen so that every
product and every partial sum is a dyadic number well inside fp32's 24 significant bits: for a convolution
``K * max|x| * max|w| + max|bias| + max|residual| < 2^16`` with K = R * S * C / groups.  Such sums are exact in
fp32 whatever the summation order, the split into MMAs or the accumulator shuffle of a kernel, so the only
rounding left is the final fp32 -> bf16 cast (round to nearest even) and the expected output is
``ref64.float().to(dtype)``, where ``ref64`` is the same operation in float64.  The kernels must match it under
``torch.equal``: one missing product changes an element.

The fp32 CUDA-core convolution (``impl="simt"``, plain FFMA) is the control: it is exact by IEEE arithmetic on
the same data, so if it disagrees the harness is wrong, not the kernel.

A mismatch is reported with its position (image, row, column, channel), the kernel's tile and in-tile
coordinates, and how the wrong elements are distributed over images, tile rows / columns and channels.

The premise checks (bounds of every case, the rounding of the expected value, the operand generator) run
without a GPU; everything else is marked ``gpu``.
"""
import gc
import math
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from eyediseasesegmentation_b200 import _lib, kernels as K

DEV = "cuda"
BOUND = 1 << 16             # every partial sum stays below this in magnitude
GUARD = 4096                # guard elements allocated right behind every output
TWO31 = 1 << 31
BIG_BUDGET = 12 << 30       # bytes the past-2^31 tests may hold at once (the GPUs are shared)


# ------------------------------------------------------------------------------------------------ harness
def ints(shape, lo, hi, seed, dtype=torch.bfloat16, device=DEV):
    """Uniform integers in [lo, hi], drawn where they live (multi-GB operands are never built on the host)."""
    g = torch.Generator(device=device).manual_seed(seed)
    return torch.empty(shape, dtype=dtype, device=device).random_(lo, hi + 1, generator=g)


def eighths(shape, seed, device=DEV):
    """Gates: multiples of 1/8 in [0, 1] (fp32)."""
    return ints(shape, 0, 8, seed, torch.float32, device) / 8


def seed_of(name):
    return zlib.crc32(name.encode()) & 0x7FFFFFFF


def expected(ref64, dtype):
    """What an exact kernel stores: the float64 result, exact in fp32 (checked), rounded once to `dtype`."""
    assert torch.equal(ref64, ref64.float().double()), "premise broken: the float64 result is not exact in fp32"
    return ref64.float().to(dtype)


def bf16_exact_fraction(ref64):
    return float((ref64 == ref64.float().bfloat16().double()).double().mean())


def check_sensitivity(ref64, rounding):
    """A fine case must be able to show a one-product error (>= 90 % of its values exact in bf16); a rounding
    case must exercise round-to-nearest-even (>= 1/3 of its values rounded)."""
    frac = bf16_exact_fraction(ref64)
    if rounding:
        assert 1 - frac >= 1 / 3, f"only {1 - frac:.1%} of the outputs need rounding"
    else:
        assert frac >= 0.9, f"only {frac:.1%} of the outputs are exact in bf16: too coarse to see one product"


def nchw(t):
    return t.permute(0, 3, 1, 2)


def nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def conv_ref64(x, w, bias, stride=1, pad=1, relu=False, residual=None, groups=1, gate=None):
    """float64 convolution on the device: x [N,H,W,C], w [Cout,R,S,C/groups] -> [N,Ho,Wo,Cout]
    = relu((conv + bias) * gate[n, co] + residual)."""
    y = F.conv2d(nchw(x.double()), nchw(w.double()), None if bias is None else bias.double(), stride=stride,
                 padding=pad, groups=groups)
    if gate is not None:
        y.mul_(gate.double()[:, :, None, None])
    if residual is not None:
        y.add_(nchw(residual.double()))
    if relu:
        y.clamp_min_(0)
    return nhwc(y)


def guarded(shape, dtype):
    """An output pre-filled with NaN and a guard of 7.0 right behind it in the same allocation: every element
    must be written, and nothing past the end."""
    n = math.prod(shape)
    buf = torch.empty(n + GUARD, dtype=dtype, device=DEV)
    buf[:n].fill_(float("nan"))
    buf[n:].fill_(7.0)
    return buf[:n].view(shape), buf[n:]


def guard_intact(guard):
    return bool((guard == 7.0).all())


# kernel tiles, for the mismatch report: th x tw pixels of tn images (and cn output channels)
Tiling = namedtuple("Tiling", "name th tw tn cn", defaults=(1, None))
HALO_TILE = Tiling("conv3x3_halo", 32, 8)
WIDE_TILE = Tiling("conv3x3_wide", 8, 30)
SMALL_TILE = Tiling("conv3x3_small", 16, 32)
STEM_TILE = Tiling("stem", 16, 16)


def _pow2_ceil(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def igemm_tiling(N, Ho, Wo, Cout, groups=1):
    """The pixel tile TN x TH x TW = 128 and the cout tile that eds_conv2d_igemm_bf16 picks for this shape."""
    bn = 256
    while bn > 16 and Cout % bn:
        bn -= 16
    if groups > 1:
        bn = 64
    best, tw_best = None, 8
    for tw in (8, 16, 32, 64, 128):
        th = min(128 // tw, _pow2_ceil(Ho))
        tn = 128 // (tw * th)
        tiles = -(-Wo // tw) * -(-Ho // th) * -(-N // tn)
        if best is None or tiles <= best:
            best, tw_best = tiles, tw
    th = min(128 // tw_best, _pow2_ceil(Ho))
    return Tiling("conv_igemm", th, tw_best, 128 // (tw_best * th), bn)


def _hist(counts, limit=12):
    nz = [(i, int(c)) for i, c in enumerate(counts.tolist()) if c]
    s = ", ".join(f"{i}: {c}" for i, c in nz[:limit])
    return "{" + s + (", ..." if len(nz) > limit else "") + "}"


def mismatch_report(got, want, tiling=None, limit=8):
    """None when got == want bit for bit, else where the differing elements are.  got / want: [N,H,W,C]."""
    if tuple(got.shape) != tuple(want.shape):
        return f"shape {tuple(got.shape)} != {tuple(want.shape)}"
    if torch.equal(got, want):
        return None
    bad = got != want                                       # NaN (never written) compares unequal
    N, H, W, C = bad.shape
    per_n = bad.sum((1, 2, 3)).cpu()
    per_c = bad.sum((0, 1, 2)).cpu()
    hw = bad.sum((0, 3)).cpu()                              # [H, W]
    count = int(per_n.sum())
    nan = int(torch.isnan(got.float()).sum())
    lines = [f"{count} of {bad.numel()} elements differ ({nan} NaN: never written)"]
    n0 = int(per_n.nonzero()[0])
    for h, w, c in bad[n0].nonzero()[:limit].tolist():
        s = f"  (n={n0}, h={h}, w={w}, c={c}): got {float(got[n0, h, w, c])}, want {float(want[n0, h, w, c])}"
        if tiling is not None:
            t = tiling
            s += f"; {t.name} tile (n {n0 // t.tn}, h {h // t.th}, w {w // t.tw}"
            s += f", c {c // t.cn})" if t.cn else ")"
            s += f", in-tile row {h % t.th} col {w % t.tw}"
        lines.append(s)
    lines.append(f"images: {_hist(per_n)}")
    groups16 = per_c.view(-1, 16).sum(1) if C % 16 == 0 else per_c
    lines.append(f"channels: {_hist(per_c, 16)}; by 16-channel group: {_hist(groups16)}")
    rows, cols = hw.sum(1), hw.sum(0)
    ri, ci = torch.arange(H), torch.arange(W)
    border = ((ri == 0) | (ri == H - 1)).view(H, 1) | ((ci == 0) | (ci == W - 1)).view(1, W)
    lines.append(f"on the map border: {int(hw[border].sum())} of {count}")
    if tiling is not None:
        th, tw = tiling.th, tiling.tw
        rows_t = torch.zeros(th, dtype=torch.long).index_add_(0, ri % th, rows)
        cols_t = torch.zeros(tw, dtype=torch.long).index_add_(0, ci % tw, cols)
        edge = ((ri % th == 0) | (ri % th == th - 1)).view(H, 1) | ((ci % tw == 0) | (ci % tw == tw - 1)).view(1, W)
        lines.append(f"rows in tile (h % {th}): {_hist(rows_t)}")
        lines.append(f"columns in tile (w % {tw}): {_hist(cols_t)}")
        lines.append(f"on {tiling.name} tile edges: {int(hw[edge].sum())} of {count}")
    return "\n".join(lines)


def assert_exact(got, want, tiling=None, what=""):
    msg = mismatch_report(got, want, tiling)
    if msg is not None:
        pytest.fail(f"{what}\n{msg}")


# ------------------------------------------------------------------------------------------------ case tables
# C is the total reduction width, C1 the part of it that comes from the second input.  x in [-xr, xr],
# w in [-wr, wr], bias in [-br, br] (no bias when br is None), residual in [-rr, rr] (none when rr is None).
# rounding: the wide-operand case of a kernel (>= 1/3 of the outputs are rounded to bf16).
Conv = namedtuple("Conv", "N H W C Cout R stride relu rr br C1 groups xr wr rounding",
                  defaults=(3, 1, False, None, 8, 0, 1, 2, 1, False))

IGEMM_CASES = {
    "bk64": Conv(2, 20, 24, 64, 64, relu=True),
    "bk32_bn32_st32_res": Conv(1, 17, 19, 96, 32, rr=8),
    "bk16_bn48_st16": Conv(2, 13, 11, 48, 48, relu=True),
    "bn256x2_1x1_stbufs2_res": Conv(2, 16, 16, 256, 512, R=1, relu=True, rr=8),
    "bn256x4_1x1_stbufs2_nobias": Conv(1, 12, 20, 512, 1024, R=1, br=None),
    "bn256x8_1x1_stbufs1_res": Conv(3, 7, 7, 1024, 2048, R=1, relu=True, rr=8),
    "bn160_st32": Conv(1, 10, 14, 512, 640, R=1, relu=True),
    "bn80_st16": Conv(2, 15, 21, 64, 80, relu=True),
    "bn16x17": Conv(1, 9, 14, 32, 272),
    "s2_odd": Conv(2, 19, 23, 64, 128, stride=2, relu=True),
    "s2_odd_bk16_res": Conv(1, 21, 17, 48, 64, stride=2, rr=8),
    "1x1_s2": Conv(2, 17, 15, 128, 64, R=1, stride=2),
    "tn2_n5": Conv(5, 6, 5, 64, 64, relu=True),
    "w1": Conv(3, 5, 1, 64, 64),
    "w200_tw128": Conv(1, 3, 200, 64, 32, relu=True),
    "2src_bk32": Conv(1, 20, 18, 96, 64, C1=32, relu=True),
    "2src_bk16_res": Conv(2, 11, 13, 112, 32, C1=16, rr=8),
    "rounding": Conv(1, 10, 12, 64, 64, rr=16, br=16, xr=8, wr=8, rounding=True),
    "rounding_1x1_bn256": Conv(2, 9, 11, 256, 256, R=1, br=16, xr=16, wr=8, rounding=True),
}

GROUPED_CASES = {
    "cpg4": Conv(2, 13, 17, 64, 64, relu=True, groups=16),
    "cpg8_s2_res": Conv(1, 15, 21, 128, 128, stride=2, rr=8, groups=16),
    "cpg16_res": Conv(3, 9, 11, 128, 128, relu=True, rr=8, groups=8),
    "cpg32_s2": Conv(2, 14, 10, 256, 256, stride=2, groups=8),
    "cpg32_rounding": Conv(1, 12, 9, 64, 64, xr=12, wr=12, br=16, groups=2, rounding=True),
}

HALO_CASES = {
    "cout16_bk16": Conv(1, 45, 19, 16, 16, relu=True),
    "cout48_bk32_res": Conv(2, 33, 9, 32, 48, rr=8),
    "cout80_bk64": Conv(1, 40, 17, 64, 80, relu=True),
    "cout112_h31": Conv(1, 31, 23, 128, 112),
    "cout128_res": Conv(2, 70, 50, 192, 128, relu=True, rr=8),
    "smaller_than_tile": Conv(3, 7, 5, 64, 64, br=None),
    "many_tiles": Conv(8, 256, 256, 16, 32, relu=True),
    "2src_bk16_res": Conv(1, 37, 21, 112, 64, C1=48, rr=8),
    "rounding": Conv(1, 35, 17, 32, 64, xr=12, wr=12, br=16, rounding=True),
}

WIDE_CASES = {
    "cout16_w60_h15": Conv(1, 15, 60, 16, 16, relu=True),
    "cout32_w61_h17_res": Conv(2, 17, 61, 32, 32, rr=8),
    "cout48_w59_h23": Conv(1, 23, 59, 64, 48, relu=True),
    "staged_w29_res": Conv(3, 9, 29, 64, 64, relu=True, rr=8),
    "staged_w31_nobias": Conv(2, 8, 31, 64, 64, br=None),
    "streamed_w91_h25": Conv(1, 25, 91, 128, 64, relu=True),
    "streamed_448_w89_h31": Conv(1, 31, 89, 448, 64),
    "streamed_cout32_w30": Conv(2, 33, 30, 320, 32),
    "2src_streamed": Conv(1, 24, 61, 128, 64, C1=64, relu=True),
    "2src_bk32_res": Conv(2, 16, 31, 128, 32, C1=96, rr=8),
    "2src_resident_bk16": Conv(1, 7, 35, 32, 16, C1=16, relu=True),
    "many_tiles_staged": Conv(6, 256, 270, 64, 64, relu=True),
    "many_tiles_streamed": Conv(3, 200, 300, 128, 48, rr=8),
    "rounding_bk16": Conv(1, 17, 31, 16, 64, xr=16, wr=16, br=16, rounding=True),
    "rounding_staged": Conv(1, 16, 33, 64, 64, xr=8, wr=8, br=16, rr=16, rounding=True),
}

SMALL_CASES = {
    "cout16": Conv(3, 21, 19, 16, 16, relu=True),
    "cout32_nobias": Conv(2, 33, 65, 16, 32, br=None),
    "cout32_rounding": Conv(1, 17, 31, 16, 32, xr=16, wr=16, br=16, rounding=True),
}

SIMT_CASES = {
    "3x3_s2_res": Conv(2, 13, 11, 32, 48, stride=2, rr=8),
    "1x1": Conv(1, 9, 10, 64, 16, R=1, relu=True),
    "3x3_rounding": Conv(1, 11, 9, 16, 32, xr=16, wr=16, br=16, rounding=True),
    "grouped_cpg8_res": Conv(2, 9, 7, 64, 64, relu=True, rr=8, groups=8),
}

GATED_CASES = {                         # 1x1, ReLU, residual always
    "cout512": Conv(2, 10, 12, 256, 512, R=1, rr=8),
    "cout2048": Conv(1, 7, 9, 512, 2048, R=1, rr=8),
    "rounding": Conv(1, 8, 8, 64, 256, R=1, xr=32, wr=30, br=16, rr=16, rounding=True),
}

CONV_MATRIX = [(kind, name, c)
               for kind, table in (("igemm", IGEMM_CASES), ("grouped", GROUPED_CASES), ("halo", HALO_CASES),
                                   ("wide", WIDE_CASES), ("small", SMALL_CASES), ("simt", SIMT_CASES))
               for name, c in table.items()]

# stem: B, S (square: the rot90 views), x range, w range
STEM_CASES = {"s40": (2, 40, 4, 4), "s100_rounding": (1, 100, 16, 27)}
# head: N, H, W, C, classes, x range, w range
HEAD_CASES = {"c16_cls1": (2, 13, 17, 16, 1, 8, 8), "c64_cls2": (1, 9, 30, 64, 2, 8, 8)}


def conv_bound(c):
    k = c.R * c.R * (c.C // c.groups)
    return k * c.xr * c.wr + (c.br or 0) + (c.rr or 0)


# ------------------------------------------------------------------------------------------------ premise (CPU)
def test_every_case_stays_below_the_exactness_bound():
    for kind, name, c in CONV_MATRIX + [("gated", k, c) for k, c in GATED_CASES.items()]:
        assert conv_bound(c) < BOUND, (kind, name, conv_bound(c))
        assert c.xr <= 256 and c.wr <= 256, (kind, name)          # the operands themselves are exact in bf16
    for name, (B, S, xr, wr) in STEM_CASES.items():
        assert 147 * xr * wr + 8 < BOUND, name
    for name, (N, H, W, C, cls, xr, wr) in HEAD_CASES.items():
        assert 9 * C * xr * wr + 8 < BOUND, name
    for c in (BIG_IGEMM_IN, BIG_IGEMM_OUT, BIG_HALO, BIG_WIDE, BIG_WIDE_2SRC):
        assert conv_bound(c) < BOUND, c


def np_bf16_rne(f32):
    """float32 -> bfloat16 (as float32) by round to nearest, ties to even, on the bit pattern."""
    u = np.asarray(f32, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return r.astype(np.uint32).view(np.float32)


def test_expected_value_rounds_to_nearest_even():
    # integers from 256 up: bf16 keeps 8 significant bits, so every odd value in [256, 512) is a tie
    v = np.concatenate([np.arange(-70000, 70000, 1, dtype=np.float64), np.arange(-300, 300, 1 / 128),
                        np.random.default_rng(0).normal(0, 1000, 10000).astype(np.float32).astype(np.float64)])
    got = expected(torch.from_numpy(v), torch.bfloat16).float().numpy()
    assert np.array_equal(got, np_bf16_rne(v.astype(np.float32)))
    ties = expected(torch.tensor([257.0, 259.0, 261.0, -257.0, 513.0, 515.0, 258.0], dtype=torch.float64),
                    torch.bfloat16).float().tolist()
    assert ties == [256.0, 260.0, 260.0, -256.0, 512.0, 516.0, 258.0]
    with pytest.raises(AssertionError):
        expected(torch.tensor([1.0 + 2.0 ** -30], dtype=torch.float64), torch.bfloat16)


def test_operand_generator_is_deterministic():
    a = ints((3, 5, 7, 16), -2, 2, 11, device="cpu")
    assert torch.equal(a, ints((3, 5, 7, 16), -2, 2, 11, device="cpu"))
    assert not torch.equal(a, ints((3, 5, 7, 16), -2, 2, 12, device="cpu"))
    assert a.dtype == torch.bfloat16 and set(a.float().unique().tolist()) == {-2.0, -1.0, 0.0, 1.0, 2.0}
    g = eighths((4, 64), 3, device="cpu")
    assert torch.equal(g, eighths((4, 64), 3, device="cpu")) and torch.equal(g * 8, (g * 8).round())
    assert float(g.min()) >= 0 and float(g.max()) <= 1


def test_igemm_tiling_covers_the_configurations_the_cases_claim():
    t = igemm_tiling(5, 6, 5, 64)
    assert t.tn == 2 and 5 % t.tn                      # several images per tile, N not a multiple of TN
    assert igemm_tiling(1, 3, 200, 32).tw == 128
    assert igemm_tiling(3, 5, 1, 64).tw == 8
    assert igemm_tiling(1, 9, 14, 272).cn == 16 and igemm_tiling(1, 10, 14, 640).cn == 160
    assert igemm_tiling(1, 12, 20, 1024).cn == 256


def test_mismatch_report_localises_a_wrong_channel_at_a_tile_column():
    """The report of an injected fault (channel 7 of the last column of every wide tile) names that channel,
    that in-tile column and the images, and says the elements sit on tile edges."""
    want = ints((2, 17, 75, 32), -2, 2, 1, device="cpu")
    got = want.clone()
    got[:, :, 29::30, 7] += 1
    got[1, 3, 4, 5] = float("nan")
    msg = mismatch_report(got, want, WIDE_TILE)
    assert msg.startswith(f"{2 * 17 * 2 + 1} of {want.numel()} elements differ (1 NaN")
    assert "channels: {5: 1, 7: 68}" in msg and "columns in tile (w % 30): {4: 1, 29: 68}" in msg
    assert "images: {0: 34, 1: 35}" in msg and "tile edges: 68 of 69" in msg
    assert "(n=0, h=0, w=29, c=7): got" in msg and "in-tile row 0 col 29" in msg
    assert mismatch_report(want, want.clone(), WIDE_TILE) is None


# ------------------------------------------------------------------------------------------------ convolutions
def conv_operands(c, seed):
    C0 = c.C - c.C1
    Ho, Wo = K.conv_out_hw(c.H, c.W, c.R, c.stride, c.R // 2)
    x0 = ints((c.N, c.H, c.W, C0), -c.xr, c.xr, seed)
    x1 = ints((c.N, c.H, c.W, c.C1), -c.xr, c.xr, seed + 1) if c.C1 else None
    w = ints((c.Cout, c.R, c.R, c.C // c.groups), -c.wr, c.wr, seed + 2)
    b = ints((c.Cout,), -c.br, c.br, seed + 3, torch.float32) if c.br is not None else None
    res = ints((c.N, Ho, Wo, c.Cout), -c.rr, c.rr, seed + 4) if c.rr is not None else None
    return x0, x1, w, b, res, (Ho, Wo)


def run_conv(kind, c, x0, x1, w, b, res, out):
    pad = c.R // 2
    if kind == "small":
        return K.conv3x3_small(x0, w, b, c.relu, out=out)
    if kind == "grouped":
        return K.conv2d(x0, K.pack_grouped_weights(w), b, c.stride, pad, c.relu, res, out=out, impl="tc",
                        groups=c.groups)
    return K.conv2d(x0, w, b, c.stride, pad, c.relu, res, out=out, impl=kind, x1=x1)


def conv_tiling(kind, c, Ho, Wo):
    if kind in ("igemm", "grouped"):
        return igemm_tiling(c.N, Ho, Wo, c.Cout, c.groups)
    return {"halo": HALO_TILE, "wide": WIDE_TILE, "small": SMALL_TILE}.get(kind)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,name,c", CONV_MATRIX, ids=[f"{k}-{n}" for k, n, _ in CONV_MATRIX])
def test_conv_exact(kind, name, c):
    x0, x1, w, b, res, (Ho, Wo) = conv_operands(c, seed_of(kind + name))
    x = x0 if x1 is None else torch.cat([x0, x1], -1)
    ref = conv_ref64(x, w, b, c.stride, c.R // 2, c.relu, res, c.groups)
    check_sensitivity(ref, c.rounding)
    # the control: fp32 FFMA on the same values must already be exact
    ctrl = K.conv2d(x.float(), w.float(), b, c.stride, c.R // 2, c.relu, None if res is None else res.float(),
                    impl="simt", groups=c.groups)
    assert_exact(ctrl, expected(ref, torch.float32), what="control (fp32 CUDA-core kernel): the harness is wrong")
    if kind == "simt":
        out, guard = guarded((c.N, Ho, Wo, c.Cout), torch.bfloat16)
        K.conv2d(x, w, b, c.stride, c.R // 2, c.relu, res, out=out, impl="simt", groups=c.groups)
        assert guard_intact(guard), "simt bf16 wrote past its output"
        assert_exact(out, expected(ref, torch.bfloat16), what="simt bf16")
        return
    out, guard = guarded((c.N, Ho, Wo, c.Cout), torch.bfloat16)
    run_conv(kind, c, x0, x1, w, b, res, out)
    assert guard_intact(guard), f"{kind} wrote past the end of its output"
    assert_exact(out, expected(ref, torch.bfloat16), conv_tiling(kind, c, Ho, Wo), f"{kind} {name} {c}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GATED_CASES))
def test_conv1x1_se_gated_epilogue_exact(name):
    """relu((conv1x1(x) + bias) * gate[n, co] + residual) with dyadic gates."""
    c = GATED_CASES[name]
    x, _, w, b, res, _ = conv_operands(c, seed_of("gated" + name))
    gate = eighths((c.N, c.Cout), seed_of("gate" + name))
    ref = conv_ref64(x, w, b, 1, 0, True, res, gate=gate)
    check_sensitivity(ref, c.rounding)
    out, guard = guarded((c.N, c.H, c.W, c.Cout), torch.bfloat16)
    K.conv1x1_se(x, w, b, gate, res, out=out)
    assert guard_intact(guard)
    assert_exact(out, expected(ref, torch.bfloat16), igemm_tiling(c.N, c.H, c.W, c.Cout), f"gated {name}")


ROUTING = [
    # N, H, W, C, Cout, R, kernel conv2d(impl="tc") must pick, forced impl
    (1, 20, 20, 16, 16, 3, "conv3x3_small (mma.sync)", "small"),
    (1, 64, 70, 32, 64, 3, "conv3x3_wide (tcgen05)", "wide"),
    (1, 63, 80, 32, 64, 3, "conv_igemm 3x3 (tcgen05)", "igemm"),          # one side below WIDE_MIN_HW
    (1, 64, 66, 64, 128, 3, "conv3x3_halo (tcgen05)", "halo"),             # Cout > 64: not wide
    (1, 80, 63, 64, 128, 3, "conv_igemm 3x3 (tcgen05)", "igemm"),          # one side below HALO_MIN_HW
    (1, 64, 64, 32, 160, 3, "conv_igemm 3x3 (tcgen05)", "igemm"),          # Cout > 128
    (2, 30, 30, 64, 256, 1, "conv_igemm 1x1 (tcgen05)", "igemm"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ROUTING, ids=[f"{r[6].split()[0]}-{r[1]}x{r[2]}-{r[4]}" for r in ROUTING])
def test_tc_routing_picks_the_expected_kernel(case):
    """impl="tc" picks the kernel its size rules (HALO_MIN_HW, WIDE_MIN_HW, the small-kernel rule) say, and the
    result is bit-identical to that kernel forced."""
    N, H, W, C, Cout, R, tag, forced = case
    assert K.HALO_MIN_HW == 64 and K.WIDE_MIN_HW == 64 and K.WIDE_MIN_CIN == 16
    x = ints((N, H, W, C), -2, 2, 5)
    w = ints((Cout, R, R, C), -1, 1, 6)
    b = ints((Cout,), -8, 8, 7, torch.float32)
    K.KERNEL_TRACE = []
    try:
        y = K.conv2d(x, w, b, 1, R // 2, True, None, impl="tc")
        tags = [t for t, _ in K.KERNEL_TRACE]
    finally:
        K.KERNEL_TRACE = None
    assert tags == [tag]
    y2 = K.conv3x3_small(x, w, b, True) if forced == "small" else K.conv2d(x, w, b, 1, R // 2, True, None, impl=forced)
    assert torch.equal(y, y2)
    assert_exact(y, expected(conv_ref64(x, w, b, 1, R // 2, True), torch.bfloat16))


# ------------------------------------------------------------------------------------------------ stem and head
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(STEM_CASES))
def test_stem_exact_all_d4_views(name):
    from eyediseasesegmentation_b200 import ttach_compat as tta
    B, S, xr, wr = STEM_CASES[name]
    seed = seed_of("stem" + name)
    tfm = tta.aliases.d4_transform()
    aug, _ = tta.view_maps(tfm, S, S)
    assert len(aug) == 8
    x = ints((B, 3, S, S), -xr, xr, seed, torch.float32)
    w = ints((64, 3, 7, 7), -wr, wr, seed + 1, torch.float32)
    b = ints((64,), -8, 8, seed + 2, torch.float32)
    ref = torch.cat([nhwc(F.conv2d(t.augment_image(x.double()), w.double(), b.double(), stride=2, padding=3))
                     for t in tfm], 0).clamp_min(0)
    check_sensitivity(ref, rounding=name.endswith("rounding"))
    w_hwio = w.permute(2, 3, 1, 0).contiguous()
    shape = (8 * B, S // 2, S // 2, 64)
    for dtype in (torch.float32, torch.bfloat16):
        out, guard = guarded(shape, dtype)
        K.stem_conv(x, aug, w_hwio, b, dtype, out=out)
        assert guard_intact(guard)
        assert_exact(out, expected(ref, dtype), STEM_TILE, f"stem_conv {dtype}")
    out, guard = guarded(shape, torch.bfloat16)
    K.stem_conv_mma(x, aug, K.stem_pack_weights(w_hwio), b, out=out)
    assert guard_intact(guard)
    assert_exact(out, expected(ref, torch.bfloat16), STEM_TILE, "stem_conv_mma")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("name", list(HEAD_CASES))
def test_head_conv3x3_logits_exact(name, dtype):
    N, H, W, C, classes, xr, wr = HEAD_CASES[name]
    seed = seed_of("head" + name)
    x = ints((N, H, W, C), -xr, xr, seed, dtype)
    w = ints((classes, 3, 3, C), -wr, wr, seed + 1, torch.float32)
    b = ints((classes,), -8, 8, seed + 2, torch.float32)
    ref = nchw(conv_ref64(x, w, b))
    out, guard = guarded((N, classes, H, W), torch.float32)
    K.head_conv3x3(x, w, b, out=out)
    assert guard_intact(guard)
    assert_exact(out.permute(0, 2, 3, 1), expected(ref, torch.float32).permute(0, 2, 3, 1), what="head_conv3x3")


# ------------------------------------------------------------------------------------------------ data movement
def up2x_ref64(x, mode):
    """x [N,h,w,C] -> float64 [N,2h,2w,C] (nearest, or bilinear with align_corners=False), or x itself."""
    if mode == _lib.UP_NONE:
        return x.double()
    if mode == _lib.UP_NEAREST:
        return x.double().repeat_interleave(2, 1).repeat_interleave(2, 2)
    return nhwc(F.interpolate(nchw(x.double()), scale_factor=2, mode="bilinear", align_corners=False))


DTYPES = [torch.float32, torch.bfloat16]
UP_MODES = {"nearest": _lib.UP_NEAREST, "bilinear": _lib.UP_BILINEAR, "none": _lib.UP_NONE}
MAP_SIZES = [(2, 5, 7), (1, 3, 1), (3, 1, 4)]              # odd h and w, and w = 1 / h = 1: the edge clamps run


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode", list(UP_MODES))
@pytest.mark.parametrize("n_skips", [0, 1, 5])
def test_upsample2x_concat_exact(mode, n_skips, dtype):
    m = UP_MODES[mode]
    up = 1 if m == _lib.UP_NONE else 2
    for N, h, w in MAP_SIZES:
        seed = seed_of(f"up{mode}{n_skips}{h}{w}")
        # integers up to 255: the bilinear mix needs 12 significant bits, so bf16 outputs are rounded
        x0 = ints((N, h, w, 24), -255, 255, seed, dtype)
        skips = [ints((N, up * h, up * w, 8 * (k + 1)), -255, 255, seed + 1 + k, dtype) for k in range(n_skips)]
        ref = torch.cat([up2x_ref64(x0, m)] + [s.double() for s in skips], -1)
        out, guard = guarded(tuple(ref.shape), dtype)
        K.upsample2x_concat(x0, skips, m, out=out)
        assert guard_intact(guard)
        assert_exact(out, expected(ref, dtype), what=f"upsample2x_concat {mode} {N}x{h}x{w}")


def gated_srcs(N, h, w, chans, gated, seed, dtype, xr=16):
    srcs = []
    for k, (c, g) in enumerate(zip(chans, gated)):
        hh, ww = (h, w) if k == 0 else (2 * h, 2 * w)
        x = ints((N, hh, ww, c), -xr, xr, seed + 3 * k, dtype)
        srcs.append((x, eighths((N, c), seed + 3 * k + 1), eighths((N, hh, ww), seed + 3 * k + 2)) if g else
                    (x, None, None))
    return srcs


def gated_part_ref64(x, cg, sg, up_mode, cgate, sgate):
    """One source of concat_gated in float64: (up2x of) x * (cg + sg), times the concat-level gate slice."""
    v = x.double()
    if cg is not None:
        v = v * (cg.double()[:, None, None, :] + sg.double()[..., None])
    if up_mode is not None:
        v = up2x_ref64(v, up_mode)
    if cgate is not None:
        v = v * (cgate.double()[:, None, None, :] + sgate.double()[..., None])
    return v


def concat_gated_ref64(srcs, mode, cgate, sgate):
    parts, off = [], 0
    for k, (x, cg, sg) in enumerate(srcs):
        C = x.shape[3]
        parts.append(gated_part_ref64(x, cg, sg, mode if k == 0 else None,
                                      None if cgate is None else cgate[:, off:off + C], sgate))
        off += C
    return torch.cat(parts, -1)


CONCAT_CASES = {
    # chans, per-source gates, concat-level gate
    "plain": ([64, 32, 48], [False, False, False], False),
    "gated_sources": ([32, 16, 64], [True, False, True], False),
    "all_gates": ([64, 32, 48], [True, True, False], True),
    "five_sources": ([16, 8, 24, 16, 32], [True, False, True, False, True], True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode", ["nearest", "bilinear"])
@pytest.mark.parametrize("name", list(CONCAT_CASES))
def test_concat_gated_and_split_exact(name, mode, dtype):
    chans, gated, top = CONCAT_CASES[name]
    m = UP_MODES[mode]
    for N, h, w in MAP_SIZES:
        seed = seed_of(f"cat{name}{mode}{h}{w}")
        srcs = gated_srcs(N, h, w, chans, gated, seed, dtype)
        cg = eighths((N, sum(chans)), seed + 100) if top else None
        sg = eighths((N, 2 * h, 2 * w), seed + 101) if top else None
        want = expected(concat_gated_ref64(srcs, m, cg, sg), dtype)
        out, guard = guarded(tuple(want.shape), dtype)
        K.concat_gated(srcs, m, cg, sg, out=out)
        assert guard_intact(guard)
        assert_exact(out, want, what=f"concat_gated {N}x{h}x{w}")
        y_up, y_skip = K.concat_gated_split(srcs, m, cg, sg)
        assert_exact(y_up, want[..., :chans[0]].contiguous(), what=f"concat_gated_split (upsampled part) {N}x{h}x{w}")
        assert_exact(y_skip, want[..., chans[0]:].contiguous(), what=f"concat_gated_split (skip part) {N}x{h}x{w}")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_gate_scale_pool_exact(dtype):
    """apply_gate, se_scale_add_relu and avgpool2_affine with dyadic gates / scales on integer maps."""
    N, H, W, C = 3, 6, 10, 40
    seed = seed_of(f"pointwise{dtype}")
    x = ints((N, H, W, C), -100, 100, seed, dtype)
    cg, sg = eighths((N, C), seed + 1), eighths((N, H, W), seed + 2)
    out, guard = guarded((N, H, W, C), dtype)
    K.apply_gate(x, cg, sg, out=out)
    assert guard_intact(guard)
    assert_exact(out, expected(x.double() * (cg.double()[:, None, None, :] + sg.double()[..., None]), dtype),
                 what="apply_gate")
    r = ints((N, H, W, C), -100, 100, seed + 3, dtype)
    out, guard = guarded((N, H, W, C), dtype)
    K.se_scale_add_relu(x, cg, r, out=out)
    assert guard_intact(guard)
    assert_exact(out, expected((x.double() * cg.double()[:, None, None, :] + r.double()).clamp_min(0), dtype),
                 what="se_scale_add_relu")
    scale, shift = eighths((C,), seed + 4) * 2 - 1, ints((C,), -8, 8, seed + 5, torch.float32)
    for relu in (False, True):
        out, guard = guarded((N, H // 2, W // 2, C), dtype)
        K.avgpool2_affine(x, scale, shift, relu, out=out)
        assert guard_intact(guard)
        ref = nhwc(F.avg_pool2d(nchw(x.double()), 2)) * scale.double() + shift.double()
        assert_exact(out, expected(ref.clamp_min(0) if relu else ref, dtype), what=f"avgpool2_affine relu={relu}")


# ------------------------------------------------------------------------------------------------ past 2^31 elements
# One launch each with an input or output of more than 2^31 elements (> 2^32 bytes).  The per-image sizes do not
# divide 2^31, so a 32-bit offset that wrapped would land on another pixel.  Compared against float64: every image
# holding element 2^31 of an input or the output, and the last image; the whole output is checked for NaN.
BIG_IGEMM_IN = Conv(50, 300, 300, 512, 64, relu=True)                    # input 2.30 G elements
BIG_IGEMM_OUT = Conv(54, 200, 200, 64, 1024, R=1, relu=True, rr=8)       # output and residual 2.21 G elements
BIG_HALO = Conv(110, 126, 126, 1280, 128, relu=True)                     # input 2.24 G elements
BIG_WIDE = Conv(20, 510, 510, 448, 64, relu=True)                        # input 2.33 G elements
BIG_WIDE_2SRC = Conv(24, 510, 510, 448, 64, C1=384, rr=8)                # second input 2.40 G elements


@pytest.fixture
def big_memory():
    """Start from an empty cache, report the peak, hold the test to BIG_BUDGET and give everything back."""
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    yield
    peak = torch.cuda.max_memory_allocated() - base
    gc.collect()
    torch.cuda.empty_cache()
    print(f"peak memory {peak / 2 ** 30:.2f} GiB")
    assert peak <= BIG_BUDGET, f"peak {peak / 2 ** 30:.2f} GiB over the {BIG_BUDGET / 2 ** 30:.0f} GiB budget"


def images_past_2_31(*tensors):
    """Indices of the images that hold element 2^31 of any of these [N,...] tensors, plus the last image."""
    imgs = set()
    for t in tensors:
        if t is not None and t.numel() > TWO31:
            per = t[0].numel()
            assert TWO31 % per, "the per-image size divides 2^31"
            imgs.add(TWO31 // per)
    return sorted(imgs | {tensors[0].shape[0] - 1})


def nan_free(t, chunk=1 << 28):
    flat = t.view(-1)
    return not any(bool(torch.isnan(part).any()) for part in flat.split(chunk))


def _big_conv(kind, c, seed):
    """Returns None or the failure message (the tensors are gone once this returns, even when it fails)."""
    x0, x1, w, b, res, (Ho, Wo) = conv_operands(c, seed)
    out, guard = guarded((c.N, Ho, Wo, c.Cout), torch.bfloat16)
    run_conv(kind, c, x0, x1, w, b, res, out)
    torch.cuda.synchronize()
    errors = []
    if not guard_intact(guard):
        errors.append(f"{kind} wrote past its output")
    if not nan_free(out):
        errors.append(f"{kind} left output elements unwritten (NaN)")
    imgs = images_past_2_31(x0, x1, res, out)
    if not (len(imgs) >= 2 and max(x.numel() for x in (x0, x1, out, res) if x is not None) > TWO31):
        errors.append(f"case does not reach past 2^31 elements: images {imgs}")
    tiling = conv_tiling(kind, c, Ho, Wo)
    print(f"{kind} {c.N}x{c.H}x{c.W}x{c.C}->{c.Cout}: images {imgs} against float64")
    for n in imgs:
        sl = slice(n, n + 1)
        x = x0[sl] if x1 is None else torch.cat([x0[sl], x1[sl]], -1)
        ref = conv_ref64(x, w, b, c.stride, c.R // 2, c.relu, None if res is None else res[sl])
        msg = mismatch_report(out[sl], expected(ref, torch.bfloat16), tiling)
        if msg:
            errors.append(f"image {n}:\n{msg}")
        del x, ref
    return "\n".join(errors) or None


@pytest.mark.gpu
@pytest.mark.parametrize("kind,c", [("igemm", BIG_IGEMM_IN), ("igemm", BIG_IGEMM_OUT), ("halo", BIG_HALO),
                                    ("wide", BIG_WIDE), ("wide", BIG_WIDE_2SRC)],
                         ids=["igemm-input", "igemm-output-residual", "halo-input", "wide-input", "wide-2src"])
def test_conv_past_2_31_elements(kind, c, big_memory):
    msg = _big_conv(kind, c, seed_of(f"big{kind}{c}"))
    if msg is not None:
        pytest.fail(msg)


def _big_concat(seed):
    N, h, w = 34, 127, 127                                  # skip part: 34 x 254 x 254 x 1024 = 2.25 G elements
    chans = [64, 512, 512]
    srcs = gated_srcs(N, h, w, chans, [True, True, False], seed, torch.bfloat16, xr=8)
    cg, sg = eighths((N, sum(chans)), seed + 100), eighths((N, 2 * h, 2 * w), seed + 101)
    y_up, y_skip = K.concat_gated_split(srcs, _lib.UP_BILINEAR, cg, sg)
    torch.cuda.synchronize()
    errors = []
    if y_skip.numel() <= TWO31:
        errors.append("the skip map does not reach past 2^31 elements")
    imgs = images_past_2_31(y_skip, y_up)
    print(f"concat_gated_split {N}x{2 * h}x{2 * w}x{sum(chans)}: images {imgs} against float64")
    for n in imgs:
        off = 0
        for k, (x, g, s) in enumerate(srcs):           # one source at a time: a whole image in float64 is 0.6 GB
            C = chans[k]
            one = lambda t: None if t is None else t[n:n + 1]  # noqa: E731
            ref = gated_part_ref64(one(x), one(g), one(s), _lib.UP_BILINEAR if k == 0 else None,
                                   cg[n:n + 1, off:off + C], sg[n:n + 1])
            got = y_up[n:n + 1] if k == 0 else y_skip[n:n + 1, ..., off - chans[0]:off - chans[0] + C]
            msg = mismatch_report(got, expected(ref, torch.bfloat16))
            if msg:
                errors.append(f"source {k}, image {n}:\n{msg}")
            off += C
    if not (nan_free(y_up) and nan_free(y_skip)):
        errors.append("NaN in the output")
    return "\n".join(errors) or None


@pytest.mark.gpu
def test_concat_gated_split_skip_map_past_2_31_elements(big_memory):
    msg = _big_concat(seed_of("bigconcat"))
    if msg is not None:
        pytest.fail(msg)
