"""ResNet-50 family encoders on the GPU: the grouped tcgen05 / CUDA-core convolutions against F.conv2d(groups), their
rejected shapes, network parity of Unet / UNet++ with resnet50, resnext50_32x4d and se_resnext50_32x4d against the
fp32 restatement (tests/encoder_oracle.py), fused D4 TTA with CUDA-graph replay, and tta_patches from files on disk
against the oracle pipeline."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from PIL import Image

pytestmark = pytest.mark.gpu

from eyediseasesegmentation_b200 import _lib, kernels as K, tta as eds_tta, ttach_compat as tta  # noqa: E402
from oracle import pipeline, scoring  # noqa: E402

import encoder_oracle as eo  # noqa: E402
from helpers import build_product_model, rel_l2  # noqa: E402


def setup_module(module):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _rnd(*shape, seed, scale=1.0):
    return (torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale).cuda()


def _ref(x, w, bias, groups, stride, relu, res):
    """fp32 F.conv2d(groups) on the (possibly bf16-rounded) operands; NHWC in and out."""
    y = F.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(0, 3, 1, 2), bias, stride=stride, padding=1,
                 groups=groups)
    if res is not None:
        y = y + res.float().permute(0, 3, 1, 2)
    return (F.relu(y) if relu else y).permute(0, 2, 3, 1)


GROUPED_CASES = [
    # N, H, W, C (== Cout), channels per group, stride, relu, residual
    (2, 17, 23, 128, 4, 1, True, False),        # maps that are not tile multiples
    (2, 17, 23, 256, 8, 2, False, True),
    (1, 5, 3, 512, 16, 1, True, True),          # map smaller than one 128-pixel tile
    (3, 9, 11, 1024, 32, 2, True, False),
    (2, 2, 2, 1024, 32, 1, False, False),
    (4, 64, 64, 128, 4, 1, True, False),        # 256 tiles: more than the SMs
    (2, 64, 48, 256, 8, 2, True, True),
    (1, 32, 32, 1024, 32, 2, False, True),
]


@pytest.mark.parametrize("case", GROUPED_CASES)
def test_grouped_conv_tcgen05_bf16(case):
    N, H, W, C, cpg, stride, relu, use_res = case
    groups = C // cpg
    x = _rnd(N, H, W, C, seed=1).bfloat16()
    w = _rnd(C, 3, 3, cpg, seed=2, scale=1.0 / math.sqrt(9 * cpg)).bfloat16()
    b = _rnd(C, seed=3)
    Ho, Wo = K.conv_out_hw(H, W, 3, stride, 1)
    res = _rnd(N, Ho, Wo, C, seed=4).bfloat16() if use_res else None
    y = K.conv2d(x, K.pack_grouped_weights(w), b, stride, 1, relu, res, impl="tc", groups=groups)
    torch.cuda.synchronize()
    ref = _ref(x, w, b, groups, stride, relu, res)
    assert y.shape == ref.shape
    err = (y.float() - ref).abs().max().item()
    tol = 1e-2 * max(1.0, ref.abs().max().item())           # the tolerance of the dense tcgen05 kernel tests
    assert err < tol, f"grouped tcgen05 conv max abs err {err} (tol {tol})"
    assert rel_l2(y, ref) < 4e-3
    y2 = K.conv2d(x, w, b, stride, 1, relu, res, impl="simt", groups=groups)
    assert (y.float() - y2.float()).abs().max().item() < tol


@pytest.mark.parametrize("case", GROUPED_CASES)
def test_grouped_conv_simt_fp32(case):
    N, H, W, C, cpg, stride, relu, use_res = case
    groups = C // cpg
    x = _rnd(N, H, W, C, seed=1)
    w = _rnd(C, 3, 3, cpg, seed=2, scale=1.0 / math.sqrt(9 * cpg))
    b = _rnd(C, seed=3)
    Ho, Wo = K.conv_out_hw(H, W, 3, stride, 1)
    res = _rnd(N, Ho, Wo, C, seed=4) if use_res else None
    y = K.conv2d(x, w, b, stride, 1, relu, res, impl="simt", groups=groups)
    ref = _ref(x, w, b, groups, stride, relu, res)
    assert (y - ref).abs().max().item() < 1e-5 * max(1.0, ref.abs().max().item())


def test_grouped_conv_rejects_unsupported_shapes():
    lib = _lib.lib()
    x = torch.zeros(1, 8, 8, 256, dtype=torch.bfloat16, device="cuda")
    w = torch.zeros(256, 3, 3, 64, dtype=torch.bfloat16, device="cuda")
    y = torch.empty_like(x)

    def call(xp, C, groups, Cout, wp=w.data_ptr(), yp=y.data_ptr()):
        rc = lib.eds_conv2d_igemm_bf16_grouped(xp, 1, 8, 8, C, wp, None, groups, Cout, 3, 3, 1, 1, 1, None, yp,
                                               torch.cuda.current_stream().cuda_stream)
        return rc, lib.eds_last_error().decode()

    for C, groups, Cout, what in [(96, 32, 96, "divide 64"), (192, 2, 192, "divide 64"), (256, 32, 128, "Cout"),
                                  (96, 3, 96, "multiples of 64")]:
        rc, msg = call(x.data_ptr(), C, groups, Cout)
        assert rc != 0 and what in msg, (C, groups, Cout, msg)
        assert not lib.eds_conv2d_igemm_grouped_supported(C, Cout, groups, 3, 3, 1)
    rc, msg = call(x.data_ptr() + 2, 256, 32, 256)                  # misaligned input
    assert rc != 0 and "aligned" in msg
    assert lib.eds_conv2d_igemm_grouped_supported(256, 256, 32, 3, 3, 2)
    with pytest.raises(ValueError, match="not supported"):
        K.conv2d(torch.zeros(1, 8, 8, 96, dtype=torch.bfloat16, device="cuda"),
                 torch.zeros(96, 3, 3, 64, dtype=torch.bfloat16, device="cuda"), None, 1, 1, groups=32)
    torch.cuda.synchronize()                                        # nothing was launched, nothing faulted


# ------------------------------------------------------------------ network parity
NET_CASES = [(name, enc, att) for enc in eo.NEW_ENCODERS
             for name, att in (("Unet", None), ("unetplusplus_deepsup", "scse"))]
_ORACLE = {}


def _case(name, enc, att, size=256, batch=2):
    cfg = dict(encoder_name=enc, encoder_weights=None, classes=1)
    if att:
        cfg.update(decoder_attention_type=att, deep_supervision=True)
    model = build_product_model(name, cfg)
    key = (name, enc, att)
    if key not in _ORACLE:
        x = torch.randn(batch, 3, size, size, generator=torch.Generator().manual_seed(7))
        _ORACLE[key] = (x,) + eo.forward(name, model.state_dict(), x, return_features=True)
    return model, _ORACLE[key]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name,enc,att", NET_CASES)
def test_network_matches_oracle(name, enc, att, precision):
    model, (x, ref, ref_feats) = _case(name, enc, att)
    model = model.to("cuda")
    model.precision = precision
    eng = model.engine()
    eng.keep_features = True
    out = model(x.cuda()).cpu()
    assert out.shape == ref.shape
    feat_tol = 1e-4 if precision == "fp32" else 3e-2
    for i in range(1, 6):
        f = eng.features[f"f{i}"].float().permute(0, 3, 1, 2).cpu()
        assert rel_l2(f, ref_feats[i]) < feat_tol, f"encoder feature f{i}: {rel_l2(f, ref_feats[i])}"
    dprob = (torch.sigmoid(out) - torch.sigmoid(ref)).abs().max().item()
    if precision == "fp32":
        assert rel_l2(out, ref) < 1e-4
        assert dprob < 1e-4
    else:
        assert rel_l2(out - out.mean(), ref - ref.mean()) < 8e-2
        assert dprob < 2e-2


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_fused_d4_and_graph_replay_equal_eager(precision, monkeypatch):
    """se_resnext50_32x4d UNet++: fused D4 views against the oracle's D4 mean, and CUDA-graph replays (new inputs
    copied into the static buffer) against the eager launches."""
    name, cfg = "unetplusplus_deepsup", dict(encoder_name="se_resnext50_32x4d", encoder_weights=None, classes=1,
                                             decoder_attention_type="scse")
    model = build_product_model(name, cfg)
    sd = model.state_dict()
    xs = [torch.randn(2, 3, 128, 128, generator=torch.Generator().manual_seed(s)) for s in (7, 8)]
    with torch.no_grad():
        want = torch.sigmoid(pipeline.tta_mean_logits(lambda t: eo.forward(name, sd, t), xs[0], "d4"))
    model = model.to("cuda")
    model.precision = precision
    tfm = tta.aliases.d4_transform()
    monkeypatch.setenv("EDS_CUDA_GRAPHS", "0")
    eager = [model.forward_tta(x.cuda(), tfm, True).clone() for x in xs]
    assert (eager[0].cpu() - want).abs().max().item() < (2e-2 if precision == "bf16" else 1e-4)
    monkeypatch.setenv("EDS_CUDA_GRAPHS", "1")
    for rep in range(3):                      # call 1 eager, call 2 captures + replays, then pure replays
        for xi, x in enumerate(xs):
            got = model.forward_tta(x.cuda(), tfm, True)
            err = (got - eager[xi]).abs().max().item()
            assert err < (5e-3 if precision == "bf16" else 1e-5), f"input {xi} pass {rep}: {err}"
            assert (got - eager[1 - xi]).abs().max().item() > 10 * err + 1e-3
    assert any(isinstance(v, tuple) for v in model._graphs.values()), "no graph was captured"


def _fundus(h, w, seed):
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    yy, xx = np.mgrid[:h, :w]
    img[(yy - h / 2) ** 2 + (xx - w / 2) ** 2 > (0.48 * min(h, w)) ** 2] = 0
    return img


def test_tta_patches_from_disk_matches_oracle_pipeline(tmp_path, monkeypatch):
    """tta_patches (fp32 mode) with a resnext50_32x4d UNet++ checkpoint: the masks it writes equal the oracle
    pipeline's probability maps thresholded where tta.py thresholds them."""
    monkeypatch.setenv("EDS_PRECISION", "fp32")
    S = 64
    name, cfg = "unetplusplus_deepsup", dict(encoder_name="resnext50_32x4d", encoder_weights=None, classes=1)
    sd = build_product_model(name, cfg).state_dict()
    logdir = tmp_path / "models" / "IDRiD" / "EX" / "exp1"
    (logdir / "checkpoints").mkdir(parents=True)
    torch.save({"model_state_dict": sd}, logdir / "checkpoints" / "best.pth")
    img_dir, mask_root = tmp_path / "data" / "images", tmp_path / "data" / "masks"
    mask_dir = mask_root / "3. Hard Exudates"
    img_dir.mkdir(parents=True)
    mask_dir.mkdir(parents=True)
    rng = np.random.default_rng(11)
    for i, (h, w) in enumerate([(150, 200), (140, 131)]):
        Image.fromarray(_fundus(h, w, 20 + i)).save(img_dir / f"IDRiD_{i:02d}.jpg", quality=95)
        gt = (np.kron(rng.random((h // 10 + 1, w // 10 + 1)) < 0.1, np.ones((10, 10)))[:h, :w] * 255).astype(np.uint8)
        Image.fromarray(gt, "L").save(mask_dir / f"IDRiD_{i:02d}_EX.tif")
    out_dir = tmp_path / "outputs"
    config = {"dataset_name": "IDRiD", "lesion_type": "EX", "gray": False, "scale_size": S, "val_batch_size": 2,
              "model_name": name, "model_params": dict(cfg), "test_img_path": img_dir, "test_mask_path": mask_root,
              "out_dir": str(out_dir), "data_type": "tile"}
    eds_tta.tta_patches(str(logdir), config, {"best": "true", "tta": "d4", "createprob": "false", "optim_thres": 0})

    mean, std = pipeline.DATASET_STATS["IDRiD"]
    items = []
    for mp in sorted(mask_dir.glob("*.*")):
        image = np.asarray(Image.open(img_dir / mp.name.replace("_EX.tif", ".jpg")).convert("RGB")).astype("uint8")
        gt = (np.asarray(Image.open(mp).convert("L")) > 0).astype(np.uint8)
        pred = pipeline.tiled_probability_map(image, lambda t: eo.forward(name, sd, t), S, mean, std, "d4")
        items.append((pred, gt, mp.name))
    t3 = scoring.pr_curve(items)["thresholds"][2]
    written = out_dir / "IDRiD" / "tta" / "EX" / "exp1"
    for pred, _, mname in items:
        got = np.asarray(Image.open(written / mname.replace("_EX.tif", ".jpg")).convert("L")) > 127
        want = pred > t3
        if want.all():
            want = np.zeros_like(want)
        assert got.shape == want.shape
        assert np.mean(got != want) < 5e-3, mname
