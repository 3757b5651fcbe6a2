"""Per-kernel numerics: every C-ABI entry point against a plain PyTorch fp32 statement of
the same op (integer outputs bit-exact, floating point within the tolerance written in
each test).  Network-level parity against the oracle lives in test_parity_gpu.py."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from eyediseasesegmentation_b200 import _lib, kernels as K  # noqa: E402
from test_attention_exact_gpu import RANDOM_SHAPES, case_ref, error_bound, map_to_seq, mma_accepts, random_case  # noqa: E402,E501

DEV = "cuda"


def setup_module(module):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def nhwc(x):  # NCHW -> NHWC contiguous
    return x.permute(0, 2, 3, 1).contiguous()


def nchw(x):
    return x.permute(0, 3, 1, 2).contiguous()


def rel_err(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


# ------------------------------------------------------------------ convolutions
CONV_CASES = [
    # N, H, W, C, Cout, R, stride, pad, relu, residual
    (2, 32, 32, 64, 64, 3, 1, 1, True, False),
    (1, 64, 64, 128, 256, 3, 1, 1, True, False),
    (2, 16, 16, 256, 512, 1, 1, 0, False, True),
    (1, 32, 32, 64, 128, 3, 2, 1, False, False),
    (2, 32, 32, 128, 64, 1, 2, 0, True, False),
    (1, 19, 19, 64, 64, 3, 1, 1, True, False),
    (3, 8, 8, 64, 32, 3, 1, 1, True, False),
    (1, 64, 64, 32, 16, 3, 1, 1, True, False),
    (1, 64, 64, 16, 16, 3, 1, 1, True, False),
    (1, 16, 16, 512, 640, 1, 1, 0, False, False),
    (1, 38, 38, 64, 64, 3, 2, 1, True, False),
    (1, 128, 128, 320, 32, 3, 1, 1, True, False),
]


def conv_ref(x, w, bias, stride, pad, relu, residual):
    y = F.conv2d(nchw(x.float()), w.float().permute(0, 3, 1, 2), bias, stride=stride, padding=pad)
    if residual is not None:
        y = y + nchw(residual.float())
    if relu:
        y = F.relu(y)
    return nhwc(y)


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_simt_fp32(case):
    N, H, W, C, Cout, R, stride, pad, relu, use_res = case
    x = rnd(N, H, W, C, seed=1)
    w = rnd(Cout, R, R, C, seed=2, scale=1.0 / math.sqrt(R * R * C))
    b = rnd(Cout, seed=3)
    Ho, Wo = K.conv_out_hw(H, W, R, stride, pad)
    res = rnd(N, Ho, Wo, Cout, seed=4) if use_res else None
    y = K.conv2d(x, w, b, stride, pad, relu, res, impl="simt")
    ref = conv_ref(x, w, b, stride, pad, relu, res)
    assert y.shape == ref.shape
    err = (y - ref).abs().max().item()
    assert err < 2e-4, f"simt fp32 conv max abs err {err}"


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_tcgen05_bf16(case):
    N, H, W, C, Cout, R, stride, pad, relu, use_res = case
    x = rnd(N, H, W, C, seed=1).bfloat16()
    w = rnd(Cout, R, R, C, seed=2, scale=1.0 / math.sqrt(R * R * C)).bfloat16()
    b = rnd(Cout, seed=3)
    Ho, Wo = K.conv_out_hw(H, W, R, stride, pad)
    res = rnd(N, Ho, Wo, Cout, seed=4).bfloat16() if use_res else None
    y = K.conv2d(x, w, b, stride, pad, relu, res, impl="tc")
    torch.cuda.synchronize()
    ref = conv_ref(x, w, b, stride, pad, relu, res)
    # inputs are identical bf16 values; only the output rounding (2^-9 relative) and the fp32
    # accumulation order differ
    err = (y.float() - ref).abs().max().item()
    tol = 1e-2 * max(1.0, ref.abs().max().item())
    assert err < tol, f"tcgen05 conv max abs err {err} (tol {tol}), rel {rel_err(y, ref)}"
    assert rel_err(y, ref) < 4e-3
    # and against the CUDA-core kernel on the same bf16 data
    y2 = K.conv2d(x, w, b, stride, pad, relu, res, impl="simt")
    assert (y.float() - y2.float()).abs().max().item() < tol


def test_conv_tcgen05_large_k():
    # decoder-sized reduction: K = 9 * 1024
    x = rnd(1, 32, 32, 1024, seed=5).bfloat16()
    w = rnd(256, 3, 3, 1024, seed=6, scale=1.0 / 96).bfloat16()
    y = K.conv2d(x, w, None, 1, 1, True, None, impl="tc")
    ref = conv_ref(x, w, None, 1, 1, True, None)
    assert rel_err(y, ref) < 4e-3


HALO_CASES = [
    # N, H, W, C, Cout, relu, use_res
    (2, 64, 64, 64, 64, True, False),      # exact tiles
    (1, 96, 72, 128, 64, True, False),     # several tiles per SM slot, two channel chunks
    (3, 40, 20, 64, 32, False, True),      # ragged in H and W, residual, three images
    (1, 70, 13, 448, 64, True, False),     # long reduction (7 chunks), ragged
    (2, 64, 64, 32, 16, True, False),      # 64-byte swizzle (block_k 32), narrowest N
    (1, 66, 30, 16, 16, True, False),      # 32-byte swizzle (block_k 16)
    (1, 64, 64, 320, 128, True, True),     # widest supported N (two accumulator sets = all of TMEM)
    (1, 16, 16, 64, 48, True, False),      # map smaller than the 32x8 tile / 34-row slab
    (5, 32, 8, 96, 64, False, False),      # block_k 32 with 3 chunks, one tile per image
]


@pytest.mark.parametrize("case", HALO_CASES)
def test_conv3x3_halo_bf16(case):
    """Persistent halo-reuse 3x3 kernel == fp32 convolution of the same bf16 data, and == the generic
    tcgen05 kernel (every tap / half / accumulator set / tile-edge combination)."""
    N, H, W, C, Cout, relu, use_res = case
    x = rnd(N, H, W, C, seed=11).bfloat16()
    w = rnd(Cout, 3, 3, C, seed=12, scale=1.0 / math.sqrt(9 * C)).bfloat16()
    b = rnd(Cout, seed=13)
    res = rnd(N, H, W, Cout, seed=14).bfloat16() if use_res else None
    y = K.conv2d(x, w, b, 1, 1, relu, res, impl="halo")
    torch.cuda.synchronize()
    ref = conv_ref(x, w, b, 1, 1, relu, res)
    err = (y.float() - ref).abs().max().item()
    tol = 1e-2 * max(1.0, ref.abs().max().item())
    assert err < tol, f"halo conv max abs err {err} (tol {tol}), rel {rel_err(y, ref)}"
    assert rel_err(y, ref) < 4e-3
    y2 = K.conv2d(x, w, b, 1, 1, relu, res, impl="igemm")
    assert (y.float() - y2.float()).abs().max().item() < tol


def test_conv3x3_halo_many_tiles():
    """More tiles than SMs: every CTA walks several tiles through both accumulator sets."""
    x = rnd(2, 256, 256, 64, seed=15).bfloat16()
    w = rnd(64, 3, 3, 64, seed=16, scale=1.0 / 24).bfloat16()
    y = K.conv2d(x, w, None, 1, 1, True, None, impl="halo")
    ref = conv_ref(x, w, None, 1, 1, True, None)
    assert rel_err(y, ref) < 4e-3
    assert (y.float() - ref).abs().max().item() < 1e-2 * max(1.0, ref.abs().max().item())


# --------------------------------------------------------------------------- stem
def d4_maps(S):
    from eyediseasesegmentation_b200 import ttach_compat as tta
    return tta.view_maps(tta.aliases.d4_transform(), S, S)


def test_stem_conv_views():
    from eyediseasesegmentation_b200 import ttach_compat as tta
    B, S = 2, 64
    x = rnd(B, 3, S, S, seed=7)
    w = rnd(64, 3, 7, 7, seed=8, scale=0.1)
    b = rnd(64, seed=9)
    tfm = tta.aliases.d4_transform()
    aug, _ = tta.view_maps(tfm, S, S)
    y = K.stem_conv(x, aug, w.permute(2, 3, 1, 0).contiguous(), b, torch.float32)
    refs = []
    for t in tfm:
        refs.append(nhwc(F.relu(F.conv2d(t.augment_image(x), w, b, stride=2, padding=3))))
    ref = torch.cat(refs, 0)
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() < 1e-4
    yb = K.stem_conv(x, aug, w.permute(2, 3, 1, 0).contiguous(), b, torch.bfloat16)
    assert rel_err(yb, ref) < 5e-3
    # tensor-core stem (bf16 operands): against the fp32 reference and, tightly, against the same
    # convolution of the bf16-rounded operands
    ym = K.stem_conv_mma(x, aug, K.stem_pack_weights(w.permute(2, 3, 1, 0).contiguous()), b)
    assert ym.shape == ref.shape and rel_err(ym, ref) < 8e-3
    xr, wr = x.bfloat16().float(), w.bfloat16().float()
    ref_r = torch.cat([nhwc(F.relu(F.conv2d(t.augment_image(xr), wr, b, stride=2, padding=3))) for t in tfm], 0)
    assert rel_err(ym, ref_r) < 4e-3


@pytest.mark.parametrize("B,S", [(1, 32), (3, 96), (2, 608)])
def test_stem_conv_mma_ragged_tiles(B, S):
    """Sizes that are not multiples of the 8 x 16 output tile, one view."""
    x = rnd(B, 3, S, S, seed=17)
    w = rnd(64, 3, 7, 7, seed=18, scale=0.1)
    b = rnd(64, seed=19)
    ident = [(1, 0, 0, 0, 1, 0)]
    ym = K.stem_conv_mma(x, ident, K.stem_pack_weights(w.permute(2, 3, 1, 0).contiguous()), b)
    ref = nhwc(F.relu(F.conv2d(x.bfloat16().float(), w.bfloat16().float(), b, stride=2, padding=3)))
    assert ym.shape == ref.shape and rel_err(ym, ref) < 4e-3


# -------------------------------------------------------------------- pointwise
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_maxpool_variants(dtype):
    x = rnd(2, 33, 33, 64, seed=10).to(dtype)
    for k, s, p, ceil in [(3, 2, 0, True), (3, 2, 1, False), (2, 2, 0, False)]:
        y = K.maxpool2d(x, k, s, p, ceil)
        ref = nhwc(F.max_pool2d(nchw(x.float()), k, s, p, ceil_mode=ceil))
        assert y.shape == ref.shape, (k, s, p, ceil)
        assert torch.equal(y.float(), ref)
    x = rnd(1, 32, 32, 16, seed=11).to(dtype)
    y = K.maxpool2d(x, 3, 2, 0, True)
    assert y.shape == (1, 16, 16, 16)
    assert torch.equal(y.float(), nhwc(F.max_pool2d(nchw(x.float()), 3, 2, 0, ceil_mode=True)))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_avgpool2_affine(dtype):
    x = rnd(2, 16, 16, 64, seed=12).to(dtype)
    sc, sh = rnd(64, seed=13), rnd(64, seed=14)
    y = K.avgpool2_affine(x, sc, sh, True)
    ref = nhwc(F.relu(F.avg_pool2d(nchw(x.float()), 2) * sc.view(1, -1, 1, 1) + sh.view(1, -1, 1, 1)))
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    assert (y.float() - ref).abs().max().item() < tol


@pytest.mark.parametrize("C", [16, 64, 320, 1024, 3072])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_channel_mean(C, dtype):
    x = rnd(3, 20, 12, C, seed=15).to(dtype)
    m = K.channel_mean(x)
    ref = x.float().mean(dim=(1, 2))
    assert (m - ref).abs().max().item() < 1e-5


def test_se_gate():
    N, C, Cr = 3, 256, 16
    mean = rnd(N, C, seed=16)
    w1, b1, w2, b2 = rnd(Cr, C, seed=17, scale=0.1), rnd(Cr, seed=18), rnd(C, Cr, seed=19, scale=0.2), rnd(C, seed=20)
    g = K.se_gate(mean, w1, b1, w2, b2)
    ref = torch.sigmoid(F.relu(mean @ w1.t() + b1) @ w2.t() + b2)
    assert (g - ref).abs().max().item() < 1e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_se_scale_add_relu(dtype):
    x, r = rnd(2, 8, 8, 64, seed=21).to(dtype), rnd(2, 8, 8, 64, seed=22).to(dtype)
    g = torch.rand(2, 64, device=DEV)
    y = K.se_scale_add_relu(x, g, r)
    ref = F.relu(x.float() * g.view(2, 1, 1, 64) + r.float())
    assert (y.float() - ref).abs().max().item() < (1e-6 if dtype == torch.float32 else 3e-2)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_upsample2x_concat(mode, dtype):
    x0 = rnd(2, 5, 7, 32, seed=25).to(dtype)
    skips = [rnd(2, 10, 14, 16, seed=26).to(dtype), rnd(2, 10, 14, 64, seed=27).to(dtype)]
    y = K.upsample2x_concat(x0, skips, mode)
    up = F.interpolate(nchw(x0.float()), scale_factor=2, mode="bilinear" if mode else "nearest",
                       **({"align_corners": False} if mode else {}))
    ref = torch.cat([nhwc(up)] + [s.float() for s in skips], dim=-1)
    assert y.shape == ref.shape
    assert (y.float() - ref).abs().max().item() < (1e-6 if dtype == torch.float32 else 2e-2)
    y1 = K.upsample2x_concat(x0, [], mode)
    assert (y1.float() - nhwc(up)).abs().max().item() < (1e-6 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_mhca_gate(dtype):
    att = rnd(2, 6, 6, 16, seed=28).to(dtype)
    ori = rnd(2, 12, 12, 16, seed=29).to(dtype)
    y = K.mhca_gate(ori, att)
    g = F.interpolate(torch.sigmoid(nchw(att.float())), scale_factor=2, mode="bilinear", align_corners=False)
    ref = ori.float() * nhwc(g)
    assert (y.float() - ref).abs().max().item() < (1e-6 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_head_conv(dtype):
    x = rnd(2, 20, 24, 16, seed=30).to(dtype)
    w = rnd(1, 16, 3, 3, seed=31, scale=0.1)
    b = rnd(1, seed=32)
    y = K.head_conv3x3(x, w.permute(0, 2, 3, 1).contiguous(), b)
    ref = F.conv2d(nchw(x.float()), w, b, padding=1)
    assert (y - ref).abs().max().item() < 1e-5


# -------------------------------------------------------------------- attention
@pytest.mark.parametrize("axis", [0, 1])
@pytest.mark.parametrize("cross", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", RANDOM_SHAPES)
def test_axial_attention(axis, cross, dtype, shape):
    """bf16 runs the tensor-core kernel (attention_mma.cu) where the shape allows (heads % 4 == 0, L <= 64,
    incl. lengths that are not multiples of 16 -- base_dim 19 of the vessel configs), fp32 and the
    2-head case the CUDA-core kernel.  With ReLU off and on, checked per element against the float64 reference
    within the bound derived in test_attention_exact_gpu.error_bound (the roundings of the probabilities and of
    the store)."""
    c, case, qk, vt = random_case(shape, axis, cross, dtype)
    S, heads, L, dqk = case.q.shape
    tensor_core = dtype == torch.bfloat16 and mma_accepts(heads, dqk, c.dv, L)
    for relu in (False, True):
        y = K.axial_attention(qk.to(DEV), None if vt is None else vt.to(DEV), axis, heads, dqk, c.dv,
                              case.rel.to(DEV), case.sim_scale.to(DEV), case.out_scale.to(DEV),
                              case.out_shift.to(DEV), relu)
        ref, _, arv, av, _ = case_ref(case, relu=relu, parts=True)
        bound = error_bound(case, ref, arv, av, dtype, tensor_core)
        err = (map_to_seq(y, axis).double().cpu() - ref).abs()
        worst = float((err / bound).max())
        assert worst <= 1, f"relu={relu}: error {worst:.2f} x the bound; max |y - ref| = {float(err.max()):.3g}"


# ----------------------------------------------------------- TTA / paste / tile
@pytest.mark.parametrize("S", [96, 128, 192])       # 96: 32x32 scalar kernel; multiples of 64: the 64x64 vector kernel
@pytest.mark.parametrize("alias", ["d4_transform", "flip_transform", "hflip_transform"])
def test_tta_merge_matches_ttach_semantics(alias, S):
    from eyediseasesegmentation_b200 import ttach_compat as tta
    tfm = getattr(tta.aliases, alias)()
    B = 2
    V = len(tfm)
    logits = rnd(V, B, 1, S, S, seed=50)
    _, deaug = tta.view_maps(tfm, S, S)
    prob = K.tta_merge(logits.view(V, B, S, S).contiguous(), deaug, True)
    merger = tta.Merger("mean", V)
    for v, t in enumerate(tfm):
        merger.append(t.deaugment_mask(logits[v]))
    ref = torch.sigmoid(merger.result)[:, 0]
    assert (prob - ref).abs().max().item() < 2e-6
    mean = K.tta_merge(logits.view(V, B, S, S).contiguous(), deaug, False)
    assert torch.equal(mean, merger.result[:, 0])  # same fp32 summation order -> bit exact


def test_resize_paste_x2_and_general():
    src = torch.rand(64, 64, device=DEV)
    dst = torch.zeros(200, 210, device=DEV)
    K.resize_paste(src, dst, (0, 0, 64, 64), (10, 20), (128, 128))
    ref = F.interpolate(src[None, None], scale_factor=2, mode="bilinear", align_corners=False)[0, 0]
    assert (dst[10:138, 20:148] - ref).abs().max().item() < 1e-6
    assert dst[:10].abs().max().item() == 0 and dst[138:].abs().max().item() == 0
    # clipped paste + crop + non-integer scale
    dst2 = torch.zeros(100, 100, device=DEV)
    K.resize_paste(src, dst2, (4, 8, 40, 48), (50, 60), (90, 75))
    ref2 = F.interpolate(src[None, None, 4:44, 8:56], size=(90, 75), mode="bilinear", align_corners=False)[0, 0]
    assert (dst2[50:, 60:] - ref2[:50, :40]).abs().max().item() < 1e-5


def test_preprocess_tile_matches_numpy_float64():
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, size=(300, 260, 3), dtype=np.uint8)
    mean, std = [0.44976714, 0.2186806, 0.06459363], [0.33224553, 0.17116262, 0.086509705]
    S, y0, x0 = 64, 100, 50
    out = K.preprocess_tile(torch.from_numpy(img).to(DEV), y0, x0, S, mean, std).cpu().numpy()
    win = img[y0:y0 + 2 * S, x0:x0 + 2 * S].astype(np.int32)
    small = (win[0::2, 0::2] + win[0::2, 1::2] + win[1::2, 0::2] + win[1::2, 1::2] + 2) // 4
    ref = ((small / 255.0 - np.array(mean)) / np.array(std)).astype(np.float32).transpose(2, 0, 1)
    assert np.array_equal(out, ref)


# ---------------------------------------------------------------------- scoring
def _np_counts(prob, gt):
    tp, pp = [], []
    for t in np.array(_lib.PR_THRESHOLDS):
        m = prob > t
        tp.append(int((m & (gt > 0)).sum()))
        pp.append(int(m.sum()))
    return np.array(tp), np.array(pp)


def _quantise(prob):
    """include/eds_b200.h 'PR/ROC histogram geometry', from the exported constants."""
    hi = prob >= np.float32(0.5)
    q = np.where(hi, np.float32(1.0) - prob, prob).astype(np.float32)
    k = np.clip((q.view(np.int32).astype(np.int64) >> _lib.PR_KEY_SHIFT) - _lib.PR_KEY_BIAS, 0, _lib.PR_HALF - 1)
    return np.where(hi, _lib.PR_BINS - 1 - k, k)


@pytest.mark.parametrize("n_px", [4096 * 3, 10007, 1 << 20])
def test_pr_hist_and_scan(n_px):
    from sklearn.metrics import average_precision_score, roc_auc_score
    rng = np.random.default_rng(n_px)
    n_img = 3
    logit = rng.normal(-3, 2.5, size=(n_img, n_px)).astype(np.float32)
    prob = (1 / (1 + np.exp(-logit))).astype(np.float32)
    gt = (rng.random((n_img, n_px)) < 1 / (1 + np.exp(-(logit + rng.normal(0, 1.5, logit.shape))))).astype(np.uint8)
    # plant values exactly on and next to thresholds, zeros and ones
    th32 = np.array(_lib.PR_THRESHOLDS, dtype=np.float32)
    prob[0, :19] = th32
    prob[0, 19:38] = np.nextafter(th32, np.float32(2))
    prob[0, 38:57] = np.nextafter(th32, np.float32(-1))
    prob[1, :100] = 0.0
    prob[1, 100:200] = 1.0
    gt[2] = 0  # image without positives
    hist, strad = K.pr_hist(torch.from_numpy(prob).to(DEV), torch.from_numpy(gt).to(DEV))
    ap, roc, counts, totals = [t.cpu().numpy() for t in K.pr_scan(hist, strad)]
    hist = hist.cpu().numpy()
    for i in range(n_img):
        keys = _quantise(prob[i])
        for cls in (0, 1):
            ref = np.bincount(keys[(gt[i] > 0) == bool(cls)], minlength=_lib.PR_BINS)
            assert np.array_equal(hist[i, cls], ref)
        tp, pp = _np_counts(prob[i], gt[i])
        assert np.array_equal(counts[i, :, 0], tp) and np.array_equal(counts[i, :, 1], pp)
        assert totals[i, 0] == gt[i].sum() and totals[i, 1] == n_px - gt[i].sum()
        if gt[i].sum() == 0:
            assert np.isnan(ap[i])
            continue
        # exact on key-quantised scores, within the 1e-3 budget on raw fp32 scores
        assert abs(ap[i] - average_precision_score(gt[i], keys)) < 1e-12
        assert abs(roc[i] - roc_auc_score(gt[i], keys)) < 1e-12
        assert abs(ap[i] - average_precision_score(gt[i], prob[i])) < 1e-3
        assert abs(roc[i] - roc_auc_score(gt[i], prob[i])) < 1e-3


def test_pr_scan_resolves_confident_scores():
    """A trained network's sigmoid saturates: most positives sit within 1e-3 of 1, where fp32 still has 2^-24
    steps.  The key is symmetric about 1/2, so AP / ROC stay within the budget there too (a key built from the
    bits of p alone loses 9e-2 of AP on this case)."""
    from sklearn.metrics import average_precision_score, roc_auc_score
    rng = np.random.default_rng(77)
    n_px = 600_000
    for prevalence, sharp, sep in [(0.01, 6.0, 6.0), (0.05, 8.0, 3.0), (0.02, 4.0, 1.5)]:
        gt = (rng.random(n_px) < prevalence).astype(np.uint8)
        logit = rng.normal(size=n_px) * sharp + (gt.astype(np.float64) * 2 - 1) * sep
        prob = (1.0 / (1.0 + np.exp(-logit))).astype(np.float32)
        hist, strad = K.pr_hist(torch.from_numpy(prob[None]).to(DEV), torch.from_numpy(gt[None]).to(DEV))
        ap, roc, counts, _ = [t.cpu().numpy() for t in K.pr_scan(hist, strad)]
        assert abs(ap[0] - average_precision_score(gt, prob)) < 1e-4
        assert abs(roc[0] - roc_auc_score(gt, prob)) < 1e-4
        tp, pp = _np_counts(prob, gt)
        assert np.array_equal(counts[0, :, 0], tp) and np.array_equal(counts[0, :, 1], pp)


def test_pr_hist_flat_regions_and_accumulate():
    # large constant areas exercise the warp-aggregated path; two launches accumulate
    n_px = 1 << 18
    prob = np.full((1, n_px), 0.25, dtype=np.float32)
    prob[0, 1000:2000] = 0.75
    gt = np.zeros((1, n_px), dtype=np.uint8)
    gt[0, 1500:2500] = 1
    p, g = torch.from_numpy(prob).to(DEV), torch.from_numpy(gt).to(DEV)
    hist, strad = K.pr_hist(p, g)
    hist, strad = K.pr_hist(p, g, hist, strad)
    _, _, counts, totals = [t.cpu().numpy() for t in K.pr_scan(hist, strad)]
    tp, pp = _np_counts(prob[0], gt[0])
    assert np.array_equal(counts[0, :, 0], 2 * tp) and np.array_equal(counts[0, :, 1], 2 * pp)
    assert totals[0, 0] == 2000


@pytest.mark.parametrize("C0,skip_ch,mode,gated", [
    (32, [16, 64], 1, (True, False, True)), (128, [256, 512], 1, (True, True, False)), (64, [64], 0, (True, True)),
    (256, [256, 256, 256], 1, (False, True, True, False)), (512, [512], 1, (True, False)), (64, [64, 64, 64, 64], 1, (True,) * 5),
    (512, [256], 1, (False, False)), (32, [], 1, (True,)), (16, [], 0, (True,))])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_deferred_gate_scse(C0, skip_ch, mode, gated, dtype):
    """gated_stats + sse_finalize + concat_gated == SCSEModule(cat([up2x(g(x0)), g(skips)...])) where
    g(x) = x * (cgate[n,c] + sgate[n,p]) is the pending attention2 gate of a source."""
    N, h, w = 2, 6, 5
    H, W = 2 * h, 2 * w
    chans = [C0] + list(skip_ch)
    srcs, ref_parts = [], []
    for k, c in enumerate(chans):
        hh, ww = (h, w) if k == 0 else (H, W)
        x = rnd(N, hh, ww, c, seed=80 + k).to(dtype)
        if gated[k]:
            cg = torch.rand(N, c, device=DEV, generator=torch.Generator(DEV).manual_seed(90 + k))
            sg = torch.rand(N, hh, ww, device=DEV, generator=torch.Generator(DEV).manual_seed(95 + k))
            val = x.float() * (cg.view(N, 1, 1, c) + sg.unsqueeze(-1))
        else:
            cg = sg = None
            val = x.float()
        srcs.append((x, cg, sg))
        ref_parts.append(val)
    up = nchw(ref_parts[0])
    up = F.interpolate(up, scale_factor=2, mode="bilinear", align_corners=False) if mode == 1 else \
        F.interpolate(up, scale_factor=2, mode="nearest")
    ref_cat = torch.cat([nhwc(up)] + ref_parts[1:], dim=-1)
    Ct = sum(chans)
    tol = 2e-5 if dtype == torch.float32 else 4e-2
    # plain gated concat (no attention1): decoder blocks without a skip
    plain = K.concat_gated(srcs, mode)
    assert plain.shape == ref_cat.shape and (plain.float() - ref_cat).abs().max().item() < tol
    if not skip_ch:
        return
    w_sse, b_sse = rnd(Ct, seed=70, scale=0.1), -0.2
    mean = torch.full((N, Ct), 7.0, device=DEV)                       # zero_mean must clear it
    dot0 = torch.full((N, h, w), 3.0, device=DEV)
    dot1 = torch.full((N, H, W), 5.0, device=DEV)
    off = 0
    for k, (x, cg, sg) in enumerate(srcs):
        c = x.shape[3]
        K.gated_stats(x, cg, sg, w_sse[off:off + c], mean, off, k == 0, dot0 if k == 0 else dot1, k > 1)
        off += c
    assert (mean - ref_cat.mean(dim=(1, 2))).abs().max().item() < 1e-4
    ref_logit = (ref_cat * w_sse).sum(-1) + b_sse
    sgate = K.sse_finalize(dot0, dot1, mode, b_sse)
    assert (sgate - torch.sigmoid(ref_logit)).abs().max().item() < 1e-4
    cgate = torch.rand(N, Ct, device=DEV)
    y = K.concat_gated(srcs, mode, cgate, sgate)
    ref = ref_cat * cgate.view(N, 1, 1, Ct) + ref_cat * torch.sigmoid(ref_logit).unsqueeze(-1)
    assert (y.float() - ref).abs().max().item() < tol
    # attention2 form: statistics of a plain map, gate kept pending, materialised on demand
    x = srcs[-1][0]
    c = x.shape[3]
    m2 = torch.empty((N, c), device=DEV)
    d2 = torch.empty((N, H, W), device=DEV)
    K.gated_stats(x, None, None, w_sse[:c], m2, 0, True, d2, False)
    assert (m2 - x.float().mean(dim=(1, 2))).abs().max().item() < 1e-4
    s2 = K.sse_finalize(None, d2, 2, 0.3)
    assert (s2 - torch.sigmoid((x.float() * w_sse[:c]).sum(-1) + 0.3)).abs().max().item() < 1e-4
    cg2 = torch.rand(N, c, device=DEV)
    z = K.apply_gate(x, cg2, s2)
    refz = x.float() * (cg2.view(N, 1, 1, c) + s2.unsqueeze(-1))
    assert (z.float() - refz).abs().max().item() < tol


@pytest.mark.parametrize("case", [
    # N, H, W, C0, C1, Cout, R, impl
    (2, 64, 64, 64, 192, 64, 3, "halo"), (1, 40, 24, 128, 64, 32, 3, "halo"), (1, 64, 64, 32, 32, 16, 3, "halo"),
    (1, 32, 32, 512, 512, 256, 3, "tc"), (2, 16, 16, 256, 64, 512, 3, "tc"), (1, 24, 40, 64, 192, 128, 1, "tc"),
    (1, 64, 64, 64, 16, 64, 3, "halo"),      # block_k falls to 16 (must divide both inputs)
    (2, 64, 64, 64, 192, 64, 3, "wide"), (1, 40, 24, 128, 64, 32, 3, "wide"),
    (1, 64, 64, 32, 32, 16, 3, "wide"),      # two inputs with resident weights (block_k 32, two chunks)
])
def test_conv_two_inputs_equals_conv_of_concat(case):
    """conv2d(x0, ..., x1=x1) walks the channel chunks of x0 then x1 through two tensor maps: same result as
    the single-input kernel on torch.cat([x0, x1]) and as the fp32 reference."""
    N, H, W, C0, C1, Cout, R, impl = case
    x0 = rnd(N, H, W, C0, seed=21).bfloat16()
    x1 = rnd(N, H, W, C1, seed=22).bfloat16()
    w = rnd(Cout, R, R, C0 + C1, seed=23, scale=1.0 / math.sqrt(R * R * (C0 + C1))).bfloat16()
    b = rnd(Cout, seed=24)
    y2 = K.conv2d(x0, w, b, 1, R // 2, True, None, impl=impl, x1=x1)
    cat = torch.cat([x0, x1], dim=-1).contiguous()
    y1 = K.conv2d(cat, w, b, 1, R // 2, True, None, impl=impl)
    ref = conv_ref(cat, w, b, 1, R // 2, True, None)
    tol = 1e-2 * max(1.0, ref.abs().max().item())
    assert (y2.float() - ref).abs().max().item() < tol and rel_err(y2, ref) < 4e-3
    assert (y2.float() - y1.float()).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item()) / 4


@pytest.mark.parametrize("mode", [0, 1])
def test_concat_gated_split_equals_single_map(mode):
    """Two dense destinations hold exactly the channel slices of the single concatenated map."""
    N, h, w = 2, 7, 5
    srcs = []
    for k, c in enumerate([64, 32, 48]):
        hh, ww = (h, w) if k == 0 else (2 * h, 2 * w)
        x = rnd(N, hh, ww, c, seed=30 + k).bfloat16()
        g = torch.Generator(DEV).manual_seed(40 + k)
        srcs.append((x, torch.rand(N, c, device=DEV, generator=g), torch.rand(N, hh, ww, device=DEV, generator=g))
                    if k != 1 else (x, None, None))
    cg = torch.rand(N, 144, device=DEV)
    sg = torch.rand(N, 2 * h, 2 * w, device=DEV)
    one = K.concat_gated(srcs, mode, cg, sg)
    up, skip = K.concat_gated_split(srcs, mode, cg, sg)
    assert torch.equal(up, one[..., :64].contiguous()) and torch.equal(skip, one[..., 64:].contiguous())
    up2, skip2 = K.concat_gated_split(srcs, mode)
    one2 = K.concat_gated(srcs, mode)
    assert torch.equal(up2, one2[..., :64].contiguous()) and torch.equal(skip2, one2[..., 64:].contiguous())


@pytest.mark.parametrize("cout", [16, 32])
def test_conv3x3_small(cout):
    """Decoder-tail kernel == conv3x3(x) in fp32 on the same bf16 data; ragged tiles (sizes that are not
    multiples of the 16 x 32 output tile) and several images."""
    N, h, w, cin = 3, 21, 19, 16
    x = rnd(N, h, w, cin, seed=50).bfloat16()
    wt = rnd(cout, 3, 3, cin, seed=51, scale=1.0 / math.sqrt(9 * cin)).bfloat16()
    b = rnd(cout, seed=52)
    inp = nchw(x.float())
    ref = nhwc(F.relu(F.conv2d(inp, wt.float().permute(0, 3, 1, 2), b, padding=1)))
    y = K.conv3x3_small(x, wt, b, True)
    assert y.shape == ref.shape
    # the kernel rounds the input tile to bf16 before the MMA: compare against that too
    ref_r = nhwc(F.relu(F.conv2d(inp.bfloat16().float(), wt.float().permute(0, 3, 1, 2), b, padding=1)))
    assert rel_err(y, ref) < 8e-3 and rel_err(y, ref_r) < 4e-3
    assert (y.float() - ref_r).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())


def test_conv3x3_small_matches_implicit_gemm_at_tail_size():
    x = rnd(2, 256, 256, 16, seed=55).bfloat16()
    wt = rnd(16, 3, 3, 16, seed=56, scale=1.0 / 12).bfloat16()
    b = rnd(16, seed=57)
    y = K.conv3x3_small(x, wt, b, True)
    y2 = K.conv2d(x, wt, b, 1, 1, True, None, impl="wide")
    assert (y.float() - y2.float()).abs().max().item() < 2e-2


@pytest.mark.parametrize("case", [
    # N, H, W, C, Cout, R, stride, impl
    (2, 37, 29, 64, 256, 3, 1, "tc"), (3, 19, 19, 128, 80, 1, 1, "tc"), (2, 38, 38, 64, 128, 3, 2, "tc"),
    (2, 70, 45, 64, 64, 3, 1, "halo"), (1, 67, 33, 32, 16, 3, 1, "halo"), (2, 131, 77, 16, 16, 3, 1, "tc"),
    (2, 70, 45, 64, 64, 3, 1, "wide"), (1, 67, 33, 448, 64, 3, 1, "wide"), (2, 131, 77, 32, 16, 3, 1, "wide"),
])
def test_conv_outputs_fully_written_and_repeatable(case):
    """Every output element is written exactly by the kernel (the buffer is pre-filled with NaN: the bulk
    tensor stores clip at ragged map edges and the staging buffers are reused across tiles) and two runs
    give bit-identical results (no race between the epilogue of tile t and the main loop of tile t+1)."""
    N, H, W, C, Cout, R, stride, impl = case
    x = rnd(N, H, W, C, seed=61).bfloat16()
    w = rnd(Cout, R, R, C, seed=62, scale=1.0 / math.sqrt(R * R * C)).bfloat16()
    b = rnd(Cout, seed=63)
    Ho, Wo = K.conv_out_hw(H, W, R, stride, R // 2)
    outs = []
    for _ in range(3):
        out = torch.full((N, Ho, Wo, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
        guard = torch.full((4096,), 7.0, device=DEV, dtype=torch.bfloat16)       # allocated right behind `out`
        K.conv2d(x, w, b, stride, R // 2, False, None, out=out, impl=impl)
        torch.cuda.synchronize()
        assert not torch.isnan(out.float()).any()
        assert bool((guard == 7.0).all())
        outs.append(out.clone())
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])
    ref = conv_ref(x, w, b, stride, R // 2, False, None)
    assert rel_err(outs[0], ref) < 4e-3


def test_paste_tiles_x2_equals_sequential_pastes():
    """One launch for a batch of overlapping tiles == the tiles pasted one after the other (last writer wins,
    make_grid order), bit for bit; tiles hanging over the image edge are clipped."""
    from eyediseasesegmentation_b200.util import make_grid
    S = 64
    H, W = 300, 420
    slices = make_grid((H, W), window=2 * S, min_overlap=32)
    origins = [(int(x1), int(y1)) for (x1, _, y1, _) in slices] + [(250, 380), (-20, -30)]
    B = len(origins)
    src = torch.rand(B, S, S, device=DEV)
    want = torch.full((H, W), -1.0, device=DEV)
    for b, (y, x) in enumerate(origins):
        K.resize_paste(src[b], want, (0, 0, S, S), (y, x), (2 * S, 2 * S))
    got = torch.full((H, W), -1.0, device=DEV)
    K.paste_tiles_x2(src, got, origins)
    assert torch.equal(got, want)


@pytest.mark.parametrize("M,S", [(2, 128), (3, 96), (3, 128), (5, 64), (8, 64)])
def test_ensemble_mean_is_the_running_sum_over_models(M, S):
    """ensemble.py:94-96: mean_pred = p0; mean_pred += p1; ...; mean_pred / M -- bit exact in fp32."""
    from eyediseasesegmentation_b200 import ensemble
    probs = torch.rand(M, 2, S, S, device=DEV)
    host = probs.cpu().numpy()
    want = host[0].copy()
    for m in range(1, M):
        want += host[m]
    want = want / M              # numpy true division, as in the reference (torch's CUDA `/ scalar` multiplies by 1/M)
    assert np.array_equal(ensemble.ensemble_mean(probs).cpu().numpy(), want)
    with pytest.raises(ValueError):
        ensemble.ensemble_mean(torch.rand(9, 1, 64, 64, device=DEV))


WIDE_CASES = [
    # N, H, W, C, Cout, relu, use_res
    (2, 64, 60, 64, 64, True, False),      # exact tiles (8 rows x 30 output columns)
    (1, 96, 72, 128, 64, True, False),     # two channel chunks, ragged in W (72 = 2 * 30 + 12)
    (3, 40, 20, 64, 32, False, True),      # a single (clipped) tile column, residual, three images
    (1, 70, 13, 448, 64, True, False),     # long reduction (7 chunks), map narrower than a slab
    (2, 64, 64, 32, 16, True, False),      # 64-byte swizzle (block_k 32), narrowest N = 48
    (1, 66, 31, 16, 16, True, False),      # 32-byte swizzle (block_k 16), one column past a tile
    (1, 16, 16, 64, 48, True, False),      # N = 144
    (5, 8, 30, 96, 64, False, False),      # block_k 32 with 3 chunks, one tile per image
    (1, 128, 128, 320, 32, True, False),   # x_0_3 shape class
    (2, 24, 45, 64, 64, True, True),       # resident weights + staged TMA-store epilogue + residual, ragged W and H
    (1, 64, 90, 128, 32, False, False),    # resident weights over two channel chunks
]


@pytest.mark.parametrize("case", WIDE_CASES)
def test_conv3x3_wide_bf16(case):
    """dw-grouped 3x3 kernel (one N = 3 * Cout MMA per kernel row, shuffle-combined accumulators) == fp32
    convolution of the same bf16 data, and == the generic tcgen05 kernel."""
    N, H, W, C, Cout, relu, use_res = case
    x = rnd(N, H, W, C, seed=11).bfloat16()
    w = rnd(Cout, 3, 3, C, seed=12, scale=1.0 / math.sqrt(9 * C)).bfloat16()
    b = rnd(Cout, seed=13)
    res = rnd(N, H, W, Cout, seed=14).bfloat16() if use_res else None
    y = torch.full((N, H, W, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    K.conv2d(x, w, b, 1, 1, relu, res, out=y, impl="wide")
    torch.cuda.synchronize()
    assert not torch.isnan(y.float()).any()
    ref = conv_ref(x, w, b, 1, 1, relu, res)
    err = (y.float() - ref).abs().max().item()
    tol = 1e-2 * max(1.0, ref.abs().max().item())
    assert err < tol, f"wide conv max abs err {err} (tol {tol}), rel {rel_err(y, ref)}"
    assert rel_err(y, ref) < 4e-3
    y2 = K.conv2d(x, w, b, 1, 1, relu, res, impl="halo")
    assert (y.float() - y2.float()).abs().max().item() < tol
    y3 = K.conv2d(x, w, b, 1, 1, relu, res, impl="wide")
    assert torch.equal(y, y3)              # repeatable: no race between the halves' barriers


def test_conv3x3_wide_many_tiles_and_two_inputs():
    """More tiles than SMs (every CTA walks several tiles, the per-half TMEM barriers wrap), and the two-input
    form against the convolution of the concatenation."""
    x = rnd(2, 256, 256, 64, seed=15).bfloat16()
    w = rnd(64, 3, 3, 64, seed=16, scale=1.0 / 24).bfloat16()
    y = K.conv2d(x, w, None, 1, 1, True, None, impl="wide")
    ref = conv_ref(x, w, None, 1, 1, True, None)
    assert rel_err(y, ref) < 4e-3
    assert (y.float() - ref).abs().max().item() < 1e-2 * max(1.0, ref.abs().max().item())
    x0 = rnd(2, 64, 64, 64, seed=21).bfloat16()
    x1 = rnd(2, 64, 64, 192, seed=22).bfloat16()
    w2 = rnd(64, 3, 3, 256, seed=23, scale=1.0 / 48).bfloat16()
    b = rnd(64, seed=24)
    y2 = K.conv2d(x0, w2, b, 1, 1, True, None, impl="wide", x1=x1)
    cat = torch.cat([x0, x1], dim=-1).contiguous()
    ref2 = conv_ref(cat, w2, b, 1, 1, True, None)
    assert rel_err(y2, ref2) < 4e-3
    assert torch.equal(y2, K.conv2d(cat, w2, b, 1, 1, True, None, impl="wide"))


# ------------------------------------------------------------------ (image, tile) partition kernels (SURVEY.md 8e)
def test_pr_hist_rects_sum_to_the_full_histogram():
    """Every tile's owned rectangles binned separately (as the ranks do) and summed == the one-launch histogram of
    the whole image, bin for bin and straddle counter for straddle counter; origins are not 16-byte aligned."""
    from eyediseasesegmentation_b200 import partition
    from eyediseasesegmentation_b200.util import make_grid
    H, W = 301, 424
    rng = np.random.default_rng(9)
    prob = rng.random((H, W), dtype=np.float32)
    th32 = np.array(_lib.PR_THRESHOLDS, dtype=np.float32)
    prob.reshape(-1)[:19] = th32
    prob.reshape(-1)[500:519] = np.nextafter(th32, np.float32(2))
    prob[200:, :] = 0.0                                   # a crowded tagged bin
    gt = (rng.random((H, W)) < 0.1).astype(np.uint8)
    p, g = torch.from_numpy(prob).to(DEV), torch.from_numpy(gt).to(DEV)
    want_h, want_s = K.pr_hist(p.reshape(1, -1), g.reshape(1, -1))
    slices = [tuple(int(v) for v in s) for s in make_grid((H, W), window=128, min_overlap=32)]
    cells = partition.owned_cells(slices, (H, W))
    hist = torch.zeros((2, _lib.PR_BINS), dtype=torch.int32, device=DEV)
    strad = torch.zeros((_lib.PR_NTHRESH, 2), dtype=torch.int32, device=DEV)
    for t in range(len(slices)):
        K.pr_hist_rects(p, g, cells[t], hist, strad)
    assert torch.equal(hist, want_h[0]) and torch.equal(strad, want_s[0])
    K.pr_hist_rects(p, g, [(0, 0, 0, 5), (3, 3, 4, 0)], hist, strad)           # empty rectangles add nothing
    assert torch.equal(hist, want_h[0])
    with pytest.raises(_lib.EdsError):
        K.pr_hist_rects(p, g, [(H - 2, 0, 5, 5)], hist, strad)


def test_paste_tiles_owned_per_rank_canvases_sum_to_single_process_paste():
    """Three emulated ranks paste only what their (round-robin) tiles own into zeroed canvases: the sum is the
    one-launch paste of all tiles, bit for bit, and the canvases are disjoint."""
    from eyediseasesegmentation_b200.util import make_grid
    S = 64
    H, W = 300, 420
    slices = make_grid((H, W), window=2 * S, min_overlap=32)
    origins = [(int(x1), int(y1)) for (x1, _, y1, _) in slices]
    B = len(origins)
    src = torch.rand(B, S, S, device=DEV) + 0.5            # strictly positive: written pixels are non-zero
    want = torch.zeros((H, W), device=DEV)
    K.paste_tiles_x2(src, want, origins)
    canvases = [torch.zeros((H, W), device=DEV) for _ in range(3)]
    for t in range(B):
        K.paste_tiles_owned_x2(src[t:t + 1], t, canvases[t % 3], origins)
    written = sum((c != 0).to(torch.int32) for c in canvases)
    assert int(written.max()) == 1 and int(written.min()) == 1
    assert torch.equal(canvases[0] + canvases[1] + canvases[2], want)
    two = torch.zeros((H, W), device=DEV)                   # several consecutive tiles in one call
    K.paste_tiles_owned_x2(src[2:5], 2, two, origins)
    ref = torch.zeros((H, W), device=DEV)
    for t in (2, 3, 4):
        K.paste_tiles_owned_x2(src[t:t + 1], t, ref, origins)
    assert torch.equal(two, ref)


def test_partitioned_group_with_emulated_ranks_equals_single_process():
    """_driver.partitioned_group run once per emulated rank (world size 3, two images of different sizes, tiles of
    both mixed in one batch): canvases and integer histograms summed over the ranks == the single-process tile
    loop + whole-image histogram, exactly.  The 'network' is an elementwise map, so results cannot depend on how
    tiles are batched (the real networks' SE / SCSE means are accumulated with fp32 atomics)."""
    from eyediseasesegmentation_b200 import _driver as drv, ttach_compat as tta

    class Pointwise(torch.nn.Module):
        def forward(self, x):
            return x[:, 0:1] * 0.7 - x[:, 1:2] * 0.3 + x[:, 2:3] * 0.1

    model, tfm = Pointwise(), tta.aliases.d4_transform()
    S = 64
    mean, std = [0.45, 0.22, 0.06], [0.33, 0.17, 0.09]
    rng = np.random.default_rng(3)
    images = [torch.from_numpy(rng.integers(0, 256, size=s + (3,), dtype=np.uint8)).to(DEV) for s in [(300, 420), (200, 262)]]
    gts = [drv.pad_width4((torch.rand(im.shape[:2], device=DEV) < 0.1).to(torch.uint8)) for im in images]
    n, world = len(images), 3
    hist = torch.zeros((n, 2, _lib.PR_BINS), dtype=torch.int32, device=DEV)
    strad = torch.zeros((n, _lib.PR_NTHRESH, 2), dtype=torch.int32, device=DEV)
    total = [None] * n
    for rank in range(world):
        canvases, nxt = drv.partitioned_group(model, tfm, images, gts, S, mean, std, hist, strad, 0, rank, world,
                                              tiles_per_batch=4)
        for k in range(n):
            total[k] = canvases[k] if total[k] is None else total[k] + canvases[k]
    assert nxt == sum(drv.tile_plan(int(im.shape[0]), int(im.shape[1]), S).n for im in images)
    for k, im in enumerate(images):
        H, W = int(im.shape[0]), int(im.shape[1])
        want = drv.tiled_probability_map(model, tfm, im, S, mean, std, tiles_per_batch=4)
        assert torch.equal(total[k][:, :W], want), k
        wh, ws = K.pr_hist(want.reshape(1, -1), gts[k][:, :W].contiguous().reshape(1, -1))
        assert torch.equal(hist[k], wh[0]) and torch.equal(strad[k], ws[0]), k


def test_gaussian_blend_mode_matches_numpy_restatement():
    """Opt-in Gaussian overlap-tile blending (no reference counterpart; the overwrite paste stays the default): tiles
    accumulated in order with w = g[oy] * g[ox], then acc / wsum -- against the numpy restatement built on cv2's x2
    resize, 1e-6 (the x2 bilinear itself agrees with cv2 to 2e-7); pixels no tile covers stay 0."""
    import cv2
    from eyediseasesegmentation_b200.util import make_grid
    from oracle import pipeline
    S = 48
    H, W = 230, 301                                          # width not a multiple of 4
    slices = [tuple(int(v) for v in s) for s in make_grid((H, W), window=2 * S, min_overlap=32)][:-1]   # last tile dropped
    src = torch.rand(len(slices), S, S, generator=torch.Generator().manual_seed(17)).to(DEV)
    acc = torch.zeros((H, W), device=DEV)
    wsum = torch.zeros((H, W), device=DEV)
    window = K.gaussian_window(2 * S, device=DEV)
    for t, (y1, _, x1, _) in enumerate(slices):
        K.blend_tile_gaussian_x2(src[t], (y1, x1), window, acc, wsum)
    got = K.blend_finalize(acc, wsum).cpu().numpy()
    g = pipeline.gaussian_window(2 * S)
    assert np.array_equal(g, window.cpu().numpy())
    w2d = (g[:, None] * g[None, :]).astype(np.float32)
    pa, pw = np.zeros((H, W), np.float32), np.zeros((H, W), np.float32)
    for t, (y1, y2, x1, x2) in enumerate(slices):
        up = cv2.resize(src[t].cpu().numpy(), (2 * S, 2 * S), interpolation=cv2.INTER_LINEAR)
        pa[y1:y2, x1:x2] += w2d * up
        pw[y1:y2, x1:x2] += w2d
    want = np.where(pw > 0, pa / np.where(pw > 0, pw, 1), 0)
    assert (pw == 0).any() and np.array_equal(got == 0, want == 0)
    assert np.abs(got - want).max() < 1e-6
    # seams: with constant tiles of different levels the overwrite paste jumps by the whole level difference at a
    # tile edge; the blended map moves by the entering tile's share of the weight there (the window still has
    # exp(-2) = 14 % of its peak at the edge, so about a quarter of the difference)
    flat = torch.stack([torch.full((S, S), 0.2 * (t + 1), device=DEV) for t in range(len(slices))])
    over = torch.zeros((H, W), device=DEV)
    acc.zero_()
    wsum.zero_()
    for t, (y1, _, x1, _) in enumerate(slices):
        K.resize_paste(flat[t], over, (0, 0, S, S), (y1, x1), (2 * S, 2 * S))
        K.blend_tile_gaussian_x2(flat[t], (y1, x1), window, acc, wsum)
    smooth = K.blend_finalize(acc, wsum)
    seam = slices[1][2]                                      # first column of the second tile
    jump_over = (over[:40, seam] - over[:40, seam - 1]).abs().mean().item()
    jump_blend = (smooth[:40, seam] - smooth[:40, seam - 1]).abs().mean().item()
    assert jump_over > 0.19 and jump_blend < 0.5 * jump_over


@pytest.mark.parametrize("alias,S,shape", [("d4_transform", 64, (300, 420)), ("flip_transform", 128, (400, 612)),
                                           ("d4_transform", 128, (256, 256)), ("hflip_transform", 64, (130, 200))])
def test_tta_blend_x2_equals_merge_then_paste(alias, S, shape):
    """eds_tta_blend_x2_f32 (views -> preds in one kernel, blocks under later tiles never read) against
    eds_tta_merge + eds_paste_tiles_x2_f32, bit for bit: whole batch in one launch, and tile by tile into per-rank
    canvases (the partition's use) whose sum is the same image."""
    from eyediseasesegmentation_b200 import ttach_compat as tta
    from eyediseasesegmentation_b200.util import make_grid
    H, W = shape
    tfm = getattr(tta.aliases, alias)()
    _, deaug = tta.view_maps(tfm, S, S)
    V = len(deaug)
    slices = make_grid((H, W), window=2 * S, min_overlap=32)
    origins = [(int(x1), int(y1)) for (x1, _, y1, _) in slices]
    B = len(origins)
    assert K.tta_blend_supported(V, S, deaug, W) and not K.tta_blend_supported(V, S, deaug, W + 1)
    logits = torch.randn(V, B, S, S, device=DEV) * 3
    want = torch.full((H, W), -1.0, device=DEV)
    K.paste_tiles_x2(K.tta_merge(logits, deaug, True), want, origins)
    got = torch.full((H, W), -1.0, device=DEV)
    K.tta_blend_x2(logits, deaug, got, origins)
    assert torch.equal(got, want)
    canvases = [torch.zeros((H, W), device=DEV) for _ in range(3)]
    for t in range(B):
        K.tta_blend_x2(logits, deaug, canvases[t % 3], origins, first_tile=t, b0=t, n_src=1)
    ref = torch.zeros((H, W), device=DEV)
    K.paste_tiles_x2(K.tta_merge(logits, deaug, True), ref, origins)
    assert torch.equal(canvases[0] + canvases[1] + canvases[2], ref)
    # a sub-batch: tiles 1..2 of the list live at positions 0..1 of their own logits tensor
    if B >= 3:
        sub = logits[:, 1:3].contiguous()
        a, b = torch.zeros((H, W), device=DEV), torch.zeros((H, W), device=DEV)
        K.tta_blend_x2(sub, deaug, a, origins, first_tile=1)
        K.paste_tiles_owned_x2(K.tta_merge(sub, deaug, True), 1, b, origins)
        assert torch.equal(a, b)


@pytest.mark.parametrize("C,gated,n_cons,dtype", [(64, True, 4, torch.bfloat16), (64, False, 3, torch.bfloat16),
                                                  (256, True, 2, torch.bfloat16), (24, True, 3, torch.float32),
                                                  (512, False, 1, torch.bfloat16)])
def test_gated_stats_multi_equals_one_pass_per_consumer(C, gated, n_cons, dtype):
    """eds_gated_stats_multi (one read of a skip source for all its consumers) against eds_gated_stats run once per
    consumer: same channel means in every consumer's row, same dot maps (fp32 sums in a different order: 1e-5
    relative), accumulation on top of what the buffers already hold."""
    torch.manual_seed(C + n_cons)
    N, h, w = 3, 19, 23
    x = (torch.randn(N, h, w, C, device=DEV)).to(dtype)
    cg = torch.rand(N, C, device=DEV) if gated else None
    sg = torch.rand(N, h, w, device=DEV) if gated else None
    cons, want = [], []
    for k in range(n_cons):
        stride = C + 16 * (k + 1)
        off = 8 * k
        ws = torch.randn(C, device=DEV)
        mean0 = torch.rand(N, stride, device=DEV)
        dot0 = torch.randn(N, h, w, device=DEV)
        m_ref, d_ref = mean0.clone(), dot0.clone()
        K.gated_stats(x, cg, sg, ws, m_ref, off, False, d_ref, True)
        want.append((m_ref, d_ref))
        cons.append((ws, mean0, off, dot0))
    K.gated_stats_multi(x, cg, sg, cons)
    for (ws, m, off, d), (m_ref, d_ref) in zip(cons, want):
        assert (m - m_ref).abs().max().item() < 1e-5 * max(1.0, m_ref.abs().max().item())
        assert (d - d_ref).abs().max().item() < 2e-5 * max(1.0, d_ref.abs().max().item())


@pytest.mark.parametrize("N,H,Cin,Cout", [(3, 40, 64, 256), (2, 19, 128, 512), (5, 8, 256, 1024)])
def test_se_tail_in_conv3_epilogue(N, H, Cin, Cout):
    """SE bottleneck tail fused into conv3 (Cadene SENet bottleneck, SURVEY A.1: conv3 + BN, no activation, then
    x * se(x) + residual -> ReLU): (1) the squeeze -- channel means of conv3's OUTPUT -- equals the affine map of the
    channel means of its INPUT (eds_affine_rows), because conv3 is linear; (2) eds_conv2d_igemm_bf16_gated =
    relu((conv + bias) * gate + residual) against fp32 PyTorch and against the unfused kernel sequence."""
    x = rnd(N, H, H, Cin, seed=31).bfloat16()
    w = (rnd(Cout, 1, 1, Cin, seed=32) / math.sqrt(Cin)).bfloat16()
    b = rnd(Cout, seed=33) * 0.1
    res = rnd(N, H, H, Cout, seed=34).bfloat16()
    y3 = K.conv2d(x, w, b, 1, 0, False, None, impl="tc")                         # what round 1 wrote to HBM
    squeeze = K.affine_rows(K.channel_mean(x), w.float().reshape(Cout, Cin).contiguous(), b)
    ref_sq = torch.einsum("nhwc,oc->no", x.float(), w.float().reshape(Cout, Cin)) / (H * H) + b
    assert (squeeze - ref_sq).abs().max().item() < 1e-4
    assert (squeeze - K.channel_mean(y3)).abs().max().item() < 5e-3             # y3 is bf16-rounded per element
    gate = torch.rand(N, Cout, device=DEV)
    got = K.conv1x1_se(x, w, b, gate, res).float()
    ref = F.relu((torch.einsum("nhwc,oc->nhwo", x.float(), w.float().reshape(Cout, Cin)) + b) * gate.view(N, 1, 1, Cout)
                 + res.float())
    assert rel_err(got, ref) < 4e-3
    unfused = K.se_scale_add_relu(y3, gate, res).float()
    assert rel_err(got, unfused) < 6e-3
