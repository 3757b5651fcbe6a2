"""Bit-exact checks of the implicit-GEMM residual epilogue over many tiles per CTA.

The residual tile of each 64/32/16-channel output group is loaded by TMA into the staging buffer the group's result
leaves from, through a ring of st_bufs buffers per epilogue half (4 for short reductions, 2 for long ones).  The
cases of tests/test_exact_gpu.py mostly run one tile per CTA, so the ring never wraps there.  Every case here has
more than 148 x 4 tiles, so each buffer of each CTA is refilled many times, and together the cases cover the three
SE bottleneck tails, a residual without a gate (with and without ReLU), the 128 B / 64 B / 32 B swizzles of the
residual box (st_ch 64 / 32 / 16), several images per tile with ragged maps, and the two-input and grouped kernels.

Operands are the small integers of test_exact_gpu (gates multiples of 1/8), so the expected output is the float64
result rounded once to bf16.
"""
import pytest
import torch

from eyediseasesegmentation_b200 import kernels as K
from test_exact_gpu import (Conv, assert_exact, check_sensitivity, conv_bound, conv_operands, conv_ref64, eighths,
                            expected, guard_intact, guarded, igemm_tiling, seed_of, BOUND)

SMS = 148
RING = 4                    # the deepest staging ring (k_iters <= 8)

# SE bottleneck tails at the encoder's shapes (gate + residual + ReLU through K.conv1x1_se)
SE_CASES = {
    "layer1_256sq_64_256": Conv(4, 256, 256, 64, 256, R=1, rr=8),
    "layer2_128sq_128_512": Conv(4, 128, 128, 128, 512, R=1, rr=8),
    "layer3_64sq_256_1024": Conv(8, 64, 64, 256, 1024, R=1, rr=8),
}

# residual without a gate, through K.conv2d; kind "igemm" (dense), "grouped" or a C1 > 0 second input
RES_CASES = {
    "1x1_st64_relu": ("igemm", Conv(3, 130, 200, 64, 256, R=1, relu=True, rr=8)),
    "1x1_st64_norelu": ("igemm", Conv(3, 130, 200, 64, 256, R=1, relu=False, rr=8)),
    "1x1_st32_cout96": ("igemm", Conv(2, 190, 230, 64, 96, R=1, relu=True, rr=8)),
    "1x1_st16_cout48": ("igemm", Conv(2, 187, 229, 32, 48, R=1, rr=8)),
    "3x3_st16_cout48_ring2": ("igemm", Conv(7, 101, 99, 48, 48, relu=True, rr=8)),
    "tn2_7x6": ("igemm", Conv(1300, 7, 6, 64, 256, R=1, relu=True, rr=8)),
    "tn4_3x5": ("igemm", Conv(2500, 3, 5, 64, 96, R=1, rr=8)),
    "16x16_ragged_15x13": ("igemm", Conv(700, 13, 15, 64, 256, R=1, relu=True, rr=8)),
    "2src_1x1": ("2src", Conv(5, 128, 128, 96, 256, R=1, relu=True, rr=8, C1=32)),
    "grouped_3x3_cpg8": ("grouped", Conv(10, 64, 64, 128, 128, relu=True, rr=8, groups=16)),
}


def total_tiles(c, Ho, Wo):
    t = igemm_tiling(c.N, Ho, Wo, c.Cout, c.groups)
    return -(-Wo // t.tw) * -(-Ho // t.th) * -(-c.N // t.tn) * (c.Cout // t.cn)


def test_cases_wrap_the_staging_ring_and_stay_exact():
    for c in list(SE_CASES.values()) + [c for _, c in RES_CASES.values()]:
        assert conv_bound(c) < BOUND, c
        Ho, Wo = K.conv_out_hw(c.H, c.W, c.R, c.stride, c.R // 2)
        assert total_tiles(c, Ho, Wo) > SMS * RING, c
    assert igemm_tiling(1300, 7, 6, 256).tn == 2 and igemm_tiling(2500, 3, 5, 96).tn == 4
    assert {igemm_tiling(2, 190, 230, 96).cn, igemm_tiling(2, 187, 229, 48).cn} == {96, 48}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SE_CASES))
def test_se_tail_exact_many_tiles(name):
    c = SE_CASES[name]
    x, _, w, b, res, _ = conv_operands(c, seed_of("se" + name))
    gate = eighths((c.N, c.Cout), seed_of("segate" + name))
    ref = conv_ref64(x, w, b, 1, 0, True, res, gate=gate)
    check_sensitivity(ref, False)
    out, guard = guarded((c.N, c.H, c.W, c.Cout), torch.bfloat16)
    K.conv1x1_se(x, w, b, gate, res, out=out)
    assert guard_intact(guard)
    assert_exact(out, expected(ref, torch.bfloat16), igemm_tiling(c.N, c.H, c.W, c.Cout), f"se {name}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RES_CASES))
def test_residual_exact_many_tiles(name):
    kind, c = RES_CASES[name]
    x0, x1, w, b, res, (Ho, Wo) = conv_operands(c, seed_of("res" + name))
    x = x0 if x1 is None else torch.cat([x0, x1], -1)
    pad = c.R // 2
    ref = conv_ref64(x, w, b, c.stride, pad, c.relu, res, c.groups)
    check_sensitivity(ref, False)
    out, guard = guarded((c.N, Ho, Wo, c.Cout), torch.bfloat16)
    if kind == "grouped":
        K.conv2d(x0, K.pack_grouped_weights(w), b, c.stride, pad, c.relu, res, out=out, impl="tc", groups=c.groups)
    else:
        K.conv2d(x0, w, b, c.stride, pad, c.relu, res, out=out, impl="igemm", x1=x1)
    assert guard_intact(guard)
    assert_exact(out, expected(ref, torch.bfloat16), igemm_tiling(c.N, Ho, Wo, c.Cout, c.groups), f"{kind} {name}")
