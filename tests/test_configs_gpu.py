"""BASELINE.json configurations at their STATED sizes, and the third north-star tolerance.

  cfg-2   ``unetplusplus_deepsup`` (se_resnet50 + scse), batch 16 of 1024 x 1024, 4-view ``flip`` TTA, bf16
          (src/main/config.py:110-117, tta.py:92-99) -- and the same network in fp32 mode at batch 2
  cfg-5   vessel pipeline: ``pad_img.pad`` (data/augment_vessel/pad_img.py:8-38) on DRIVE-shaped 584 x 565 and
          CHASEDB1-shaped 960 x 999 files, then ``tta_vessel.test_tta`` (tta_vessel.py:55-136) at 608^2
          (base_dim 19) and 1024^2 (base_dim 32), ROC scoring
  AUC     ``tta_patches`` in the DEFAULT (bf16) precision, files to scores: |AUC-PR - reference path| < 1e-3,
          |AUC-ROC - reference path| < 1e-3 (aucpr.py:17-43 on the output of tta.py:189-215)

The checker is the oracle (oracle/nets.py + oracle/pipeline.py + oracle/scoring.py = sklearn) evaluated in fp32
on the GPU with TF32 off (the same torch ops as on the CPU, only faster: a 1024^2 proposed-net forward is 1.9
TFLOP).  The oracle is never on the product path.
"""
import numpy as np
import pytest
import torch
from PIL import Image

pytestmark = pytest.mark.gpu

from eyediseasesegmentation_b200 import aucpr as eds_aucpr, pad_img, tta as eds_tta, tta_vessel as eds_tta_vessel  # noqa: E402
from eyediseasesegmentation_b200 import ttach_compat as tta  # noqa: E402
from oracle import nets, pipeline, scoring  # noqa: E402
import helpers  # noqa: E402
from helpers import rel_l2, star_cfg  # noqa: E402


def setup_module(module):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _cuda_sd(sd):
    return {k: v.detach().cuda() for k, v in sd.items()}


def _oracle_tta_prob(name, cfg, sd_cuda, x, kind):
    """sigmoid of the TTA-mean logits of the oracle network, one sample at a time (bounded memory)."""
    out = []
    with torch.no_grad():
        for i in range(x.shape[0]):
            logit = nets.tta_mean_logits(lambda t: nets.forward(name, sd_cuda, t, cfg), x[i:i + 1].cuda(), kind)
            out.append(torch.sigmoid(logit)[0, 0].cpu())
    return torch.stack(out)


def _calibrate_head(name, cfg, sd, x, mean=0.0, std=2.0):
    """Rescale the segmentation head of a random-init network so that its logits on ``x`` have the given mean
    and spread: probabilities then cover the 19 thresholds and masks / ROC / PR are informative."""
    with torch.no_grad():
        logit = nets.forward(name, _cuda_sd(sd), x.cuda(), cfg)
    m, sdev = float(logit.mean()), float(logit.std())
    k = std / max(sdev, 1e-6)
    sd["segmentation_head.0.weight"] = sd["segmentation_head.0.weight"] * k
    sd["segmentation_head.0.bias"] = (sd["segmentation_head.0.bias"] - m) * k + mean
    return sd


# ------------------------------------------------------------------------------------------------ cfg-2
SE50 = dict(encoder_name="se_resnet50", encoder_weights=None, classes=1, decoder_attention_type="scse",
            deep_supervision=True)


def test_cfg2_batch16_1024_flip_bf16_matches_oracle():
    """64 maps of 1024^2 in one pass (16 images x 4 flip views): nearest-neighbour upsampling loader, SCSE on every
    decoder block, SE bottlenecks in all four encoder stages, every layer at the shape the benchmark runs."""
    name = "unetplusplus_deepsup"
    model = helpers.build_product_model(name, SE50)
    sd = model.state_dict()
    x = helpers.golden_input(16, 1024, seed=31)
    want = _oracle_tta_prob(name, SE50, _cuda_sd(sd), x, "flip")
    model = model.to("cuda")
    model.precision = "bf16"
    got = model.forward_tta(x.cuda(), tta.aliases.flip_transform(), apply_sigmoid=True)[:, 0].cpu()
    assert got.shape == want.shape == (16, 1024, 1024)
    err = (got - want).abs().max().item()
    assert err < 2e-2, f"max |dprob| {err}"                                   # north_star bf16 tolerance
    assert rel_l2(got - got.mean(), want - want.mean()) < 8e-2
    # per-sample: a batch-index mix-up would pass a pooled bound
    for i in range(16):
        assert rel_l2(got[i] - got[i].mean(), want[i] - want[i].mean()) < 0.1, i


def test_cfg2_1024_flip_fp32_matches_oracle():
    name = "unetplusplus_deepsup"
    model = helpers.build_product_model(name, SE50)
    sd = model.state_dict()
    x = helpers.golden_input(2, 1024, seed=32)
    want = _oracle_tta_prob(name, SE50, _cuda_sd(sd), x, "flip")
    model = model.to("cuda")
    model.precision = "fp32"
    got = model.forward_tta(x.cuda(), tta.aliases.flip_transform(), apply_sigmoid=True)[:, 0].cpu()
    assert (got - want).abs().max().item() < 1e-4                             # north_star fp32 tolerance
    assert rel_l2(got - got.mean(), want - want.mean()) < 1e-4


# ------------------------------------------------------------------------------------------------ cfg-5
def _vessel_like(h, w, seed):
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    yy, xx = np.mgrid[:h, :w]
    img[(yy - h / 2) ** 2 + (xx - w / 2) ** 2 > (0.49 * min(h, w)) ** 2] = 0
    return img


@pytest.mark.parametrize("raw_hw,size,base_dim,dataset", [((584, 565), 608, 19, "DRIVE"), ((960, 999), 1024, 32, "CHASEDB1")])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_cfg5_vessel_pad_then_test_tta(tmp_path, monkeypatch, raw_hw, size, base_dim, dataset, precision):
    """Raw-size files -> pad_img.pad (images and labels) -> tta_vessel.test_tta on the padded folders: the
    reference's two-step vessel recipe.  Ground truth is drawn from the oracle's own probabilities so that the ROC
    is informative for a random-init network; AUC-ROC of the product (either precision) within 1e-3 of sklearn on
    the oracle's fp32 maps, masks on disk equal to the oracle's up to threshold-boundary pixels."""
    monkeypatch.setenv("EDS_PRECISION", precision)
    name, cfg = "unetplusplusstar", star_cfg(base_dim)
    model = helpers.build_product_model(name, cfg)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    logdir = tmp_path / "models" / dataset / "Vessel" / "vexp"
    (logdir / "checkpoints").mkdir(parents=True)
    raw_img, raw_lab = tmp_path / "raw" / "images", tmp_path / "raw" / "labels"
    raw_img.mkdir(parents=True)
    raw_lab.mkdir(parents=True)
    h, w = raw_hw
    top, bottom, left, right = pad_img.pad_geometry(raw_hw, size)
    mean, std = pipeline.DATASET_STATS["IDRiD"]               # tta_vessel.py:73 passes dataset_name=None
    # vessel file lists are ``*.jpg`` (base_utils.py:81-84); labels are 8x8 blocks so that JPEG keeps them binary
    names, oracle_prob = [f"{i:02d}_test.jpg" for i in range(2)], {}
    for i, n in enumerate(names):
        Image.fromarray(_vessel_like(h, w, 90 + i)).save(raw_img / n, quality=95)
    pad_dir = tmp_path / "pad_ver" / "test"
    pad_img.pad(str(raw_img), str(pad_dir / "images"), desired_size=size)
    first = np.asarray(Image.open(pad_dir / "images" / names[0]).convert("RGB")).astype("uint8")
    _calibrate_head(name, cfg, sd, torch.from_numpy(pipeline.preprocess(first, mean, std).transpose(2, 0, 1)).float()[None])
    torch.save({"model_state_dict": sd}, logdir / "checkpoints" / "best.pth")
    sd_cuda = _cuda_sd(sd)
    for i, n in enumerate(names):
        padded = np.asarray(Image.open(pad_dir / "images" / n).convert("RGB")).astype("uint8")
        assert padded.shape == (size, size, 3)
        x = torch.from_numpy(pipeline.preprocess(padded, mean, std).transpose(2, 0, 1)).float()[None]
        oracle_prob[n] = _oracle_tta_prob(name, cfg, sd_cuda, x, "d4")[0].numpy()
        rng = np.random.default_rng(95 + i)
        p_raw = oracle_prob[n][top:top + h, left:left + w]
        hb, wb = -(-h // 8), -(-w // 8)
        p_blk = np.zeros((hb * 8, wb * 8), dtype=np.float64)
        p_blk[:h, :w] = p_raw
        p_blk = p_blk.reshape(hb, 8, wb, 8).mean(axis=(1, 3))
        lab = np.kron(rng.random((hb, wb)) < p_blk, np.ones((8, 8)))[:h, :w].astype(np.uint8) * 255
        Image.fromarray(lab, "L").save(raw_lab / n, quality=100)
    pad_img.pad(str(raw_lab), str(pad_dir / "labels"), desired_size=size, is_mask=True)
    for n in names:                                           # geometry of SURVEY 8a-3
        lab = np.asarray(Image.open(pad_dir / "labels" / n).convert("L")) > 50
        assert lab.shape == (size, size) and not lab[:top].any() and not lab[:, :left].any()
        assert not lab[top + h:].any() and not lab[:, left + w:].any() and lab.any()

    seen = {}
    real = eds_tta_vessel.get_aucroc
    monkeypatch.setattr(eds_tta_vessel, "get_aucroc", lambda gen, config: seen.setdefault("roc", real(gen, config)))
    out_dir = tmp_path / "vout"
    config = {"dataset_name": dataset, "lesion_type": "Vessel", "gray": False, "scale_size": size, "val_batch_size": 1,
              "model_name": name, "model_params": dict(cfg), "test_img_path": pad_dir / "images",
              "test_mask_path": pad_dir / "labels", "out_dir": str(out_dir), "data_type": "all"}
    eds_tta_vessel.test_tta(str(logdir), config, {"best": "true", "tta": "d4"})

    items = [(oracle_prob[n], (np.asarray(Image.open(pad_dir / "labels" / n).convert("L")) > 50).astype(np.uint8), n)
             for n in names]
    assert abs(seen["roc"] - scoring.get_aucroc(items)) < 1e-3, (seen["roc"], scoring.get_aucroc(items))
    t = scoring.roc_curve(items)["threshold"]
    written = out_dir / dataset / "tta" / "Vessel" / "vexp"
    assert sorted(p.name for p in written.iterdir()) == names
    flip_budget = 5e-3 if precision == "fp32" else 3e-2       # bf16 moves probabilities by up to 2e-2 around the cut
    for pred, _, n in items:
        got = np.asarray(Image.open(written / n).convert("L")) > 127
        assert got.shape == (size, size)
        assert 0.02 < (pred > t).mean() < 0.98, "degenerate test image"
        assert np.mean(got != (pred > t)) < flip_budget, n


# ------------------------------------------------------------------------------ AUC in product precision
def test_tta_patches_bf16_auc_within_1e3_of_reference_path(tmp_path, monkeypatch):
    """north_star: 'AUC-PR is within 1e-3' of the reference PyTorch path -- asserted end to end on the DEFAULT
    precision: JPEG files -> tta_patches (tiles, D4, bf16 tensor-core network, merge, paste, GPU histogram + scan) vs
    sklearn average_precision_score / roc_auc_score on the oracle's fp32 probability maps of the same files."""
    monkeypatch.delenv("EDS_PRECISION", raising=False)
    S = 256
    name, cfg = "unetplusplusstar", star_cfg(8)
    model = helpers.build_product_model(name, cfg)
    assert model.precision == "bf16"
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    _calibrate_head(name, cfg, sd, helpers.golden_input(1, S, seed=77), mean=-1.5, std=2.0)
    logdir = tmp_path / "models" / "IDRiD" / "EX" / "auc"
    (logdir / "checkpoints").mkdir(parents=True)
    torch.save({"model_state_dict": sd}, logdir / "checkpoints" / "best.pth")
    img_dir = tmp_path / "data" / "images"
    mask_root = tmp_path / "data" / "masks"
    mask_dir = mask_root / "3. Hard Exudates"
    img_dir.mkdir(parents=True)
    mask_dir.mkdir(parents=True)
    mean, std = pipeline.DATASET_STATS["IDRiD"]
    sd_cuda = _cuda_sd(sd)
    net = lambda t: nets.forward(name, sd_cuda, t.cuda(), cfg).cpu()      # noqa: E731
    items = []
    for i, (h, w) in enumerate([(560, 640), (512, 700), (600, 520)]):
        rng = np.random.default_rng(200 + i)
        img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        yy, xx = np.mgrid[:h, :w]
        img[(yy - h / 2) ** 2 + (xx - w / 2) ** 2 > (0.48 * min(h, w)) ** 2] = 0
        Image.fromarray(img).save(img_dir / f"IDRiD_{i:02d}.jpg", quality=95)
        image = np.asarray(Image.open(img_dir / f"IDRiD_{i:02d}.jpg").convert("RGB")).astype("uint8")
        pred = pipeline.tiled_probability_map(image, net, S, mean, std, "d4")
        gt = (rng.random((h, w)) < pred).astype(np.uint8)
        if i == 2:
            gt[:] = 0                                           # skipped by get_auc (aucpr.py:22)
        Image.fromarray(gt * 255, "L").save(mask_dir / f"IDRiD_{i:02d}_EX.tif")
        items.append((pred, gt, f"IDRiD_{i:02d}_EX.tif"))

    seen = {}
    real_auc = eds_tta.get_auc
    monkeypatch.setattr(eds_tta, "get_auc", lambda gen, config: seen.setdefault("pr", real_auc(gen, config)))
    real_curve = eds_tta.plot_aucpr_curve

    def curve(gen, exp_name, config):
        seen["roc"] = eds_aucpr.get_aucroc([it for it in gen if np.asarray(it[1]).any()], config)
        return real_curve(gen, exp_name, config)
    monkeypatch.setattr(eds_tta, "plot_aucpr_curve", curve)
    config = {"dataset_name": "IDRiD", "lesion_type": "EX", "gray": False, "scale_size": S, "val_batch_size": 2,
              "model_name": name, "model_params": dict(cfg), "test_img_path": img_dir, "test_mask_path": mask_root,
              "out_dir": str(tmp_path / "out"), "data_type": "tile"}
    eds_tta.tta_patches(str(logdir), config, {"best": "true", "tta": "d4", "createprob": "false", "optim_thres": 0})

    want_pr = scoring.get_auc(items)
    want_roc = scoring.get_aucroc(items[:2])
    assert 0.05 < want_pr < 0.995, "degenerate test set"
    assert abs(seen["pr"] - want_pr) < 1e-3, (seen["pr"], want_pr)
    assert abs(seen["roc"] - want_roc) < 1e-3, (seen["roc"], want_roc)


def test_bench_dump_outputs_hold_the_last_timed_image(tmp_path):
    """cfg-4 (the bench workload) with ``--dump-outputs``: one JSON line on stdout, and DIR holds float32 / float64
    arrays, 64 MB at most -- per lesion model a probability sample in [0, 1] and the scores of the last timed image;
    with one timed image the dumped AP is the line's mean AP.  ``--warmup 0`` runs no warm-up set."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dump = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "0",
                          "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=1800)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, res.stdout
    line = json.loads(lines[0])
    assert line["steps"] == 1 and line["warmup"] == 0
    lesions = ("EX", "HE", "MA", "SE")
    fields = ("prob_sample", "ap", "roc", "threshold_counts", "totals")
    assert sorted(os.listdir(dump)) == sorted(f"{les}_{f}.npy" for les in lesions for f in fields)
    assert sum(p.stat().st_size for p in dump.iterdir()) <= 64 << 20
    for i, les in enumerate(lesions):
        prob = np.load(dump / f"{les}_prob_sample.npy")
        assert prob.dtype == np.float32 and prob.shape == (1 << 20,)
        assert np.isfinite(prob).all() and prob.min() >= 0 and prob.max() <= 1 and prob.std() > 0
        got = {f: np.load(dump / f"{les}_{f}.npy") for f in fields[1:]}
        assert all(a.dtype == np.float64 for a in got.values())
        assert got["threshold_counts"].shape == (19, 2) and got["totals"].sum() == 2848 * 4288
        assert float(got["ap"]) == pytest.approx(line["config"]["mean_ap_per_lesion"][i], abs=1e-12)
