"""CPU tests of the host side: C-ABI surface, TTA view algebra, scoring curves from counts,
prediction caching, and the world_size-2 reduction (gloo) that stands in for the NCCL
all-reduce of the GPU box."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from eyediseasesegmentation_b200 import _lib, aucpr, ttach_compat as tta
from eyediseasesegmentation_b200._driver import CachedPredictions, longest_max_size, pad_to_square
from eyediseasesegmentation_b200.util import make_grid, multigen
from oracle import nets, scoring
import helpers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ C ABI
def test_library_loads_and_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "eds_b200.h")).read()
    declared = sorted(set(re.findall(r"EDS_API\s+[\w\s\*]+?\b(eds_\w+)\s*\(", header)))
    assert declared, "no declarations parsed"
    lib = _lib.load()                      # dlopen only; no CUDA call
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, missing
    assert declared == _lib.EXPORTS        # the ctypes table covers exactly the header
    assert lib.eds_version() >= 100


def test_small_conv_eligibility_is_a_host_decision():
    """eds_conv3x3_small_supported needs no GPU: the mma.sync tail kernel takes 16 input channels and 16 or 32
    output channels; 32-channel inputs go to the tcgen05 kernels (kernels.conv2d)."""
    lib = _lib.load()
    assert lib.eds_conv3x3_small_supported(16, 16) and lib.eds_conv3x3_small_supported(16, 32)
    assert not lib.eds_conv3x3_small_supported(32, 16) and not lib.eds_conv3x3_small_supported(32, 32)


def test_compute_entries_fail_loudly_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib.load()
    assert lib.eds_device_ok() == 0
    assert lib.eds_init() != 0 and b"no CPU fallback" in lib.eds_last_error()
    with pytest.raises(_lib.EdsError):
        _lib.lib()
    model = helpers.build_product_model("Unet", dict(encoder_name="resnet34", encoder_weights=None, classes=1))
    with pytest.raises(RuntimeError, match="CUDA"):
        model(torch.zeros(1, 3, 64, 64))
    # the drivers added on top of the path keep the rule: no silent CPU route
    from types import SimpleNamespace
    from eyediseasesegmentation_b200 import ensemble
    from eyediseasesegmentation_b200.aucpr_cb import AucPRMetricCallback
    cb = AucPRMetricCallback()
    cb.on_loader_start(None)
    runner = SimpleNamespace(output={"logits": torch.zeros(1, 1, 8, 8)}, input={"targets": torch.zeros(1, 1, 8, 8)},
                             loader_metrics={})
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cb.on_batch_end(runner)
    with pytest.raises(ValueError):
        cb.on_loader_end(runner)                       # nothing was accumulated (np.concatenate([]) in the reference)
    with pytest.raises(ValueError, match="no CPU path"):
        ensemble.ensemble_mean(torch.zeros(2, 1, 64, 64))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "eyediseasesegmentation_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "/root/reference" not in src, f


# ------------------------------------------------------------------ TTA algebra
@pytest.mark.parametrize("alias,kind,n", [("d4_transform", "d4", 8), ("flip_transform", "flip", 4),
                                          ("hflip_transform", "hflip", 2)])
def test_view_maps_agree_with_transform_chains(alias, kind, n):
    tfm = getattr(tta.aliases, alias)()
    assert len(tfm) == n
    S = 12
    x = torch.randn(2, 3, S, S)
    aug, deaug = tta.view_maps(tfm, S, S)
    ii, jj = torch.meshgrid(torch.arange(S), torch.arange(S), indexing="ij")
    oracle_views = nets.tta_views(kind)
    for v, t in enumerate(tfm):
        a, b, c, d, e, f = aug[v]
        assert torch.equal(t.augment_image(x), x[:, :, a * ii + b * jj + c, d * ii + e * jj + f])
        assert torch.equal(t.augment_image(x), oracle_views[v][0](x))       # independent restatement
        a, b, c, d, e, f = deaug[v]
        y = torch.randn(2, 1, S, S)
        assert torch.equal(t.deaugment_mask(y), y[:, :, a * ii + b * jj + c, d * ii + e * jj + f])
        assert torch.equal(t.deaugment_mask(y), oracle_views[v][1](y))
        assert torch.equal(t.deaugment_mask(t.augment_image(x)), x)


def test_generic_wrapper_equals_oracle_tta_mean():
    net = torch.nn.Conv2d(3, 1, 3, padding=1).eval()
    x = torch.randn(2, 3, 16, 16)
    with torch.no_grad():
        for alias, kind in (("d4_transform", "d4"), ("flip_transform", "flip")):
            w = tta.SegmentationTTAWrapper(net, getattr(tta.aliases, alias)(), merge_mode="mean")
            assert torch.equal(w(x), nets.tta_mean_logits(net, x, kind))


def test_multiscale_alias_is_not_fused():
    t = tta.aliases.multiscale_transform(scales=[1, 2, 4])
    assert len(t) == 3 and not tta.is_fusable(t)


# ------------------------------------------------------------------ scoring host logic
def _as_scored(items):
    """Attach oracle-computed ImageScores so the aucpr entry points run without a GPU."""
    out = []
    for pred, gt, name in items:
        tp, ap, pp = scoring.threshold_counts(pred, gt)
        from sklearn.metrics import average_precision_score, roc_auc_score
        pos = int(gt.sum())
        s = aucpr.ImageScores(average_precision_score(gt.ravel(), pred.ravel()) if pos else float("nan"),
                              roc_auc_score(gt.ravel(), pred.ravel()) if pos else float("nan"), tp, pp, pos,
                              int(gt.size - pos))
        out.append((aucpr.ScoredArray(pred, s), gt, name))
    return out


def test_aucpr_entry_points_from_counts_match_oracle(tmp_path):
    cfg = {"out_dir": str(tmp_path), "dataset_name": "IDRiD", "lesion_type": "EX"}
    for seed in (0, 1):
        items = helpers.synth_scoring_case(seed)
        scored = _as_scored(items)
        assert aucpr.get_auc(scored, cfg) == pytest.approx(scoring.get_auc(items), abs=1e-15)
        assert aucpr.get_aucroc(scored, cfg) == pytest.approx(scoring.get_aucroc(items), abs=1e-15)
        assert aucpr.plot_aucpr_curve(scored, "exp", cfg) == scoring.pr_curve(items)["thresholds"]
        assert aucpr.plot_aucroc_curve(scored, "exp", cfg) == scoring.roc_curve(items)["threshold"]
        tp, pp, ap, an = aucpr._pooled_counts(scored)
        o = scoring.pr_curve(items)
        assert np.array_equal(tp, o["tp"]) and np.array_equal(pp, o["pp"]) and ap == o["ap"]
        assert aucpr.pr_curve_from_counts(tp, pp, ap)[3] == pytest.approx(o["aucpr"], abs=1e-15)
    assert os.path.isdir(os.path.join(str(tmp_path), "IDRiD", "figures", "EX"))
    with pytest.raises(ZeroDivisionError):
        aucpr.get_auc(_as_scored([helpers.synth_scoring_case(0)[-1]]), cfg)      # no image has positives


def test_scored_array_does_not_leak_scores_to_derived_arrays():
    a = aucpr.ScoredArray(np.zeros((4, 4), np.float32), aucpr.ImageScores(1.0, 1.0, None, None, 1, 15))
    assert a._eds_scores is not None
    assert getattr(a > 0.5, "_eds_scores", None) is None and getattr(a[1:], "_eds_scores", None) is None


def test_cached_predictions_run_inference_once():
    calls = []

    def produce():
        calls.append(1)
        for i in range(3):
            yield i, i, str(i)

    gen = CachedPredictions(produce)
    assert list(gen()) == list(gen()) == list(gen) == [(i, i, str(i)) for i in range(3)]
    assert len(calls) == 1

    @multigen
    def g(n):
        for i in range(n):
            yield i
    r = g(3)
    assert list(r) == list(r) == [0, 1, 2]


def test_whole_image_geometry_idrid():
    img = np.zeros((2848, 4288, 3), np.uint8)
    import cv2
    small = longest_max_size(img, 1024, cv2.INTER_LINEAR)
    assert small.shape[:2] == (680, 1024)                  # SURVEY.md 3.3
    padded = pad_to_square(small, 1024)
    assert padded.shape[:2] == (1024, 1024)
    marker = pad_to_square(np.ones((680, 1024), np.uint8), 1024)
    assert marker[:172].sum() == 0 and marker[172:852].all() and marker[852:].sum() == 0


# ------------------------------------------------------------------ world_size 2 (gloo)
_WORKER = r"""
import os, sys, json
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, 'tests'))
import torch.distributed as dist
import helpers, test_host_logic as T
from eyediseasesegmentation_b200 import aucpr, _driver
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:{port}', rank=int(sys.argv[1]), world_size=2)
items = T._as_scored(helpers.synth_scoring_case(3, n_images=5))
mine = _driver.shard(items)
cfg = dict(out_dir={out!r}, dataset_name='IDRiD', lesion_type='EX')
res = dict(n=len(mine), auc=aucpr.get_auc(mine, cfg), roc=aucpr.get_aucroc(mine, cfg),
           pr=list(aucpr.plot_aucpr_curve(mine, 'e', cfg)), rocthr=aucpr.plot_aucroc_curve(mine, 'e', cfg))
print('RESULT' + json.dumps(res)); dist.destroy_process_group()
"""


def test_two_rank_sharding_reduces_to_single_process_answer(tmp_path):
    import json
    port = 29600 + os.getpid() % 300
    code = _WORKER.format(root=ROOT, port=port, out=str(tmp_path))
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True) for r in range(2)]
    outs = []
    for p in procs:
        o, e = p.communicate(timeout=240)
        assert p.returncode == 0, e[-2000:]
        outs.append(json.loads([l for l in o.splitlines() if l.startswith("RESULT")][0][6:]))
    items = helpers.synth_scoring_case(3, n_images=5)
    assert sorted(r["n"] for r in outs) == [2, 3]
    for r in outs:                                   # every rank holds the global answer
        assert r["auc"] == pytest.approx(scoring.get_auc(items), abs=1e-12)
        assert r["roc"] == pytest.approx(scoring.get_aucroc(items), abs=1e-12)
        assert tuple(r["pr"]) == scoring.pr_curve(items)["thresholds"]
        assert r["rocthr"] == scoring.roc_curve(items)["threshold"]


def test_stat_metrics_from_counts_follow_the_reference_formulas():
    """Host half of export_result: the five metrics from (true_p, actual_p, pred_p, n) -- including the
    empty-mask branches -- equal the reference's expressions evaluated on numpy masks (stat_result.py:55-79)."""
    import numpy as np
    from eyediseasesegmentation_b200.stat_result import metrics_from_counts, EPS
    rng = np.random.default_rng(3)
    cases = [(rng.random((40, 56)) < 0.2, rng.random((40, 56)) < 0.3), (np.zeros((8, 8), bool), rng.random((8, 8)) < 0.5),
             (rng.random((8, 8)) < 0.5, np.zeros((8, 8), bool)), (np.zeros((8, 8), bool), np.zeros((8, 8), bool)),
             (np.ones((8, 8), bool), rng.random((8, 8)) < 0.5)]
    for gt_b, pred_b in cases:
        arr_gt, arr_pred = gt_b.astype(np.uint8), pred_b.astype(np.uint8)
        true_p, actual_p, pred_p = np.sum(arr_gt & arr_pred), np.sum(arr_gt), np.sum(arr_pred)
        false_p = pred_p - true_p
        actual_n = arr_gt.size - actual_p
        true_n = actual_n - false_p
        union = actual_p + false_p
        want = (1 if actual_p == 0 else float(true_p) / float(actual_p),
                1 if pred_p == 0 else float(true_p) / float(pred_p),
                1 if actual_n == 0 else float(true_n) / float(actual_n),
                (true_p + EPS * (union == 0).astype("float")) / (actual_p + false_p + EPS),
                (2 * true_p + EPS * (union == 0).astype("float")) / (true_p + actual_p + false_p + EPS))
        got = metrics_from_counts(int(true_p), int(actual_p), int(pred_p), arr_gt.size)
        assert all(str(float(a)) == str(float(b)) for a, b in zip(got, want))


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the reference's CPU path = the oracle port, on the host cores): exactly one
    JSON line on stdout with the keys the driver reads; nothing else on stdout."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-views", "1", "--ref-size", "256"], capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, res.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_callback_pr_auc_readout_matches_sklearn():
    """aucpr_cb mirror: the histogram read-out is sklearn's precision_recall_curve + auc on key-quantised scores
    exactly (ties = shared bins), and within 1e-4 of the raw-score value (BASELINE budget: 1e-3)."""
    from eyediseasesegmentation_b200 import _lib
    from eyediseasesegmentation_b200.aucpr_cb import pr_auc_from_hist
    from oracle import scoring
    rng = np.random.default_rng(21)
    for prevalence, sharp in [(0.02, 4.0), (0.3, 1.0)]:
        gt = (rng.random(200_000) < prevalence).astype(np.float32)
        logit = rng.normal(size=gt.size) * sharp + (gt * 2 - 1) * 1.5
        pred = (1.0 / (1.0 + np.exp(-logit))).astype(np.float32)
        key = scoring.score_key(pred)
        neg = np.bincount(key[gt == 0], minlength=_lib.PR_BINS)
        pos = np.bincount(key[gt == 1], minlength=_lib.PR_BINS)
        got = pr_auc_from_hist(neg, pos)
        assert abs(got - scoring.callback_pr_auc([gt], [key.astype(np.float64)])) < 1e-12
        assert abs(got - scoring.callback_pr_auc([gt[:1000], gt[1000:]], [pred[:1000], pred[1000:]])) < 1e-4
    assert np.isnan(pr_auc_from_hist(np.ones(_lib.PR_BINS, dtype=np.int64), np.zeros(_lib.PR_BINS, dtype=np.int64)))


def test_cached_predictions_spill_beyond_the_byte_budget():
    """The three-consumer cache keeps at most EDS_CACHE_BYTES of maps in RAM and spills the rest to memmap files;
    replayed items are identical and keep their device-computed scores."""
    from eyediseasesegmentation_b200._driver import CachedPredictions
    from eyediseasesegmentation_b200.aucpr import ScoredArray, ImageScores
    calls = []

    def produce():
        calls.append(1)
        for i in range(4):
            s = ImageScores(0.1 * i, 0.5, np.zeros(19, dtype=np.int64), np.zeros(19, dtype=np.int64), 1, 2)
            yield ScoredArray(np.full((6, 7), i, np.float32), s), np.full((6, 7), i % 2, np.uint8), f"img{i}"

    cache = CachedPredictions(produce, budget_bytes=6 * 7 * 5 + 10)          # room for exactly one image
    first, second, third = list(cache), list(cache), list(cache())
    assert len(calls) == 1
    for a, b, c in zip(first, second, third):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2] == c[2]
        assert b[0]._eds_scores.ap == a[0]._eds_scores.ap and b[0].dtype == np.float32 and b[1].dtype == np.uint8
    assert cache._spill_dir is not None and len(os.listdir(cache._spill_dir.name)) == 6


def test_load_checkpoint_accepts_catalyst_style_dicts(tmp_path):
    """Reference checkpoints are catalyst dicts (optimizer state, metric dicts with numpy scalars ...): the
    restricted loader of torch >= 2.6 refuses some of them, the driver then loads them the reference's way."""
    import collections
    import torch
    from eyediseasesegmentation_b200._driver import load_checkpoint
    ckpt = {"model_state_dict": {"w": torch.arange(4.0)}, "epoch": 3,
            "valid_metrics": collections.defaultdict(float, {"auc_pr": np.float64(0.5)}),
            "checkpoint_data": {"best": np.array([1, 2, 3])}}
    torch.save(ckpt, tmp_path / "best.pth")
    got = load_checkpoint(tmp_path / "best.pth")
    assert torch.equal(got["model_state_dict"]["w"], torch.arange(4.0)) and got["epoch"] == 3


# ------------------------------------------------------------------ (image, tile) partition (SURVEY.md 8e)
def test_owned_cells_equal_last_writer_wins_map():
    """partition.owned_cells against a brute-force replay of the paste loop (preds[y1:y2, x1:x2] = tile, in order):
    IDRiD's 6-tile grid, ragged grids, the degenerate grids of make_grid (4 identical windows for 1024^2 @1024) and
    arbitrary overlapping windows."""
    from eyediseasesegmentation_b200 import partition
    cases = [((2848, 4288), 2048), ((300, 420), 128), ((608, 608), 512), ((1024, 1024), 1024), ((330, 290), 256)]
    lists = [([tuple(int(v) for v in s) for s in make_grid(shape, window=w, min_overlap=32)], shape) for shape, w in cases]
    rng = np.random.default_rng(0)
    for _ in range(5):
        wins = []
        for _ in range(7):
            y, x = int(rng.integers(-10, 90)), int(rng.integers(-10, 120))
            wins.append((y, y + int(rng.integers(1, 60)), x, x + int(rng.integers(1, 70))))
        lists.append((wins, (100, 130)))
    for slices, shape in lists:
        cells = partition.owned_cells(slices, shape)
        want = partition.owner_map(slices, shape)
        got = np.full(shape, -1, dtype=np.int32)
        for t, rects in enumerate(cells):
            for (y, x, h, w) in rects:
                assert h > 0 and w > 0 and (got[y:y + h, x:x + w] == -1).all()      # disjoint
                got[y:y + h, x:x + w] = t
        assert np.array_equal(got, want)
    # IDRiD: tile origins and the 27 * 6 = 162 units balance to within one unit on 8 ranks
    sizes = [len(partition.tile_units(27, 6, r, 8)) for r in range(8)]
    assert sum(sizes) == 162 and max(sizes) - min(sizes) <= 1
    assert partition.batches(list(range(15)), 6) == [list(range(0, 5)), list(range(5, 10)), list(range(10, 15))]
    assert partition.batches([], 6) == [] and [len(b) for b in partition.batches(list(range(13)), 6)] == [5, 4, 4]


_PART_WORKER = r"""
import os, sys, json
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, 'tests'))
import numpy as np, torch, torch.distributed as dist
from eyediseasesegmentation_b200 import partition, _lib
from eyediseasesegmentation_b200.util import make_grid
from oracle import scoring
rank = int(sys.argv[1])
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:{port}', rank=rank, world_size=2)
# every rank builds the same synthetic maps; each bins (numpy stand-in for eds_pr_hist_rects_f32: same key, same
# layout) only the pixels its (image, tile) units own; ONE all-reduce of [n_img, 2, bins] int32
shapes = [(150, 210), (140, 130), (150, 210)]
rng = np.random.default_rng(5)
maps = [rng.random(s, dtype=np.float32) for s in shapes]
gts = [(rng.random(s) < 0.2).astype(np.uint8) for s in shapes]
hist = torch.zeros((len(shapes), 2, _lib.PR_BINS), dtype=torch.int32)
unit = 0
for i, shape in enumerate(shapes):
    slices = [tuple(int(v) for v in s) for s in make_grid(shape, window=64, min_overlap=32)]
    cells = partition.owned_cells(slices, shape)
    for t in range(len(slices)):
        if unit % 2 == rank:
            for (y, x, h, w) in cells[t]:
                key = scoring.score_key(maps[i][y:y + h, x:x + w]).ravel()
                g = gts[i][y:y + h, x:x + w].ravel()
                for cls in (0, 1):
                    hist[i, cls] += torch.from_numpy(np.bincount(key[g == cls], minlength=_lib.PR_BINS).astype(np.int32))
        unit += 1
partition.allreduce_sum_(hist)
full = [[np.bincount(scoring.score_key(maps[i]).ravel()[gts[i].ravel() == cls], minlength=_lib.PR_BINS)
         for cls in (0, 1)] for i in range(len(shapes))]
ok = all(np.array_equal(hist[i, cls].numpy(), full[i][cls]) for i in range(len(shapes)) for cls in (0, 1))
print('RESULT' + json.dumps(dict(ok=bool(ok), total=int(hist.sum())))); dist.destroy_process_group()
"""


def test_two_rank_tile_partition_histograms_sum_to_single_process(tmp_path):
    import json
    port = 29950 + os.getpid() % 300
    code = _PART_WORKER.format(root=ROOT, port=port)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True) for r in range(2)]
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        res = json.loads([ln for ln in out.splitlines() if ln.startswith("RESULT")][0][6:])
        assert res["ok"] and res["total"] == 150 * 210 * 2 + 140 * 130


def test_skip_consumer_plan_of_the_dense_decoder():
    """Engine._plan_skip_consumers (host logic of eds_gated_stats_multi): which SCSE attention1 blocks read a skip
    source at its own resolution, and at which channel offset of their concat -- derived from the block list and
    checked here against the concat order of unetplusplusstar.py:239-263 ([x_up, dense skips by depth, encoder
    feature]); MHCA blocks (x_0_0, x_0_1, x_1_1) take no statistics and sources with one consumer are left out."""
    from eyediseasesegmentation_b200.archs.engine import Engine
    from eyediseasesegmentation_b200.archs.spec import dense_decoder_blocks
    eng = Engine.__new__(Engine)
    eng.blocks = dense_decoder_blocks((3, 64, 256, 512, 1024, 2048))
    scse = ["x_2_2", "x_3_3", "x_1_2", "x_2_3", "x_0_2", "x_1_3", "x_0_3", "x_0_4"]
    eng.w = {f"decoder.blocks.{n}.attention1.sse": 1 for n in scse}
    feats = [torch.empty(1, 1, 1, c) for c in (64, 256, 512, 1024, 2048)]
    plan = eng._plan_skip_consumers(feats)
    a1 = lambda n: f"decoder.blocks.{n}.attention1"      # noqa: E731
    assert plan["f1"] == [(a1("x_3_3"), 256, 320), (a1("x_2_3"), 320, 384), (a1("x_1_3"), 384, 448), (a1("x_0_3"), 256, 320)]
    assert plan["x_3_3"] == [(a1("x_2_3"), 256, 384), (a1("x_1_3"), 320, 448), (a1("x_0_3"), 192, 320)]
    assert plan["x_2_3"] == [(a1("x_1_3"), 256, 448), (a1("x_0_3"), 128, 320)]
    assert plan["f2"] == [(a1("x_2_2"), 512, 768), (a1("x_1_2"), 768, 1024), (a1("x_0_2"), 640, 896)]
    assert plan["x_2_2"] == [(a1("x_1_2"), 512, 1024), (a1("x_0_2"), 384, 896)]
    assert set(plan) == {"f1", "f2", "x_3_3", "x_2_3", "x_2_2"}          # x_1_3, x_1_2, f3, f4: one SCSE consumer or none
    # every offset + source width stays inside the consumer's concat, offsets are multiples of 8 (vector loads)
    ch = {"f1": 64, "f2": 256, "x_3_3": 64, "x_2_3": 64, "x_2_2": 256}
    for src, cons in plan.items():
        for (_, off, ctot) in cons:
            assert off % 8 == 0 and off + ch[src] <= ctot


def test_fused_blend_eligibility_is_a_host_decision():
    """eds_tta_blend_supported needs no GPU: the one-kernel blend is taken for flip / rot90 views of a square tile
    whose size is a multiple of 64 and a canvas whose rows are 16-byte aligned; everything else falls back to
    eds_tta_merge + paste (``_driver.fused_blend_views``)."""
    from eyediseasesegmentation_b200 import kernels as K, _driver as drv
    for alias, n in (("d4_transform", 8), ("flip_transform", 4), ("hflip_transform", 2)):
        _, deaug = tta.view_maps(getattr(tta.aliases, alias)(), 1024, 1024)
        assert len(deaug) == n
        assert K.tta_blend_supported(n, 1024, deaug, 4288)
        assert not K.tta_blend_supported(n, 1024, deaug, 4290)           # canvas rows not 16-byte aligned
    _, deaug96 = tta.view_maps(tta.aliases.d4_transform(), 96, 96)
    assert not K.tta_blend_supported(8, 96, deaug96, 4288)               # tile size not a multiple of 64
    assert drv.fused_blend_views(torch.nn.Identity(), tta.aliases.d4_transform(), 1024, 4288) is None   # no forward_tta
    assert drv.tile_blend_mode(None) == "overwrite"


_GROUP_WORKER = r"""
import os, sys, json
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, 'tests'))
import cv2, numpy as np, torch, torch.distributed as dist
from eyediseasesegmentation_b200 import _driver as drv, kernels as K, partition, _lib, ttach_compat as tta
from oracle import pipeline, scoring
rank = int(sys.argv[1])
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:{port}', rank=rank, world_size=2)

# ---- numpy stand-ins for the CUDA entry points the driver calls (same arithmetic as the kernels' contracts) so that
# ---- the REAL _driver.partitioned_group runs on CPU tensors: units, batches, ownership, canvases, histogram rows
def preprocess_tile(img, y0, x0, S, mean, std, out=None):
    win = img.numpy()[y0:y0 + 2 * S, x0:x0 + 2 * S]
    small = cv2.resize(win, (S, S), interpolation=cv2.INTER_LINEAR)
    out.copy_(torch.from_numpy(pipeline.preprocess(small, mean, std).transpose(2, 0, 1)).float())
    return out
def paste_tiles_owned_x2(src, first_tile, dst, origins):
    S = src.shape[1]
    H, W = dst.shape
    cells = partition.owned_cells([(y, y + 2 * S, x, x + 2 * S) for (y, x) in origins], (H, W))
    for j in range(src.shape[0]):
        t = first_tile + j
        up = cv2.resize(src[j].numpy(), (2 * S, 2 * S), interpolation=cv2.INTER_LINEAR)
        for (y, x, h, w) in cells[t]:
            dst[y:y + h, x:x + w] = torch.from_numpy(up[y - origins[t][0]:y - origins[t][0] + h, x - origins[t][1]:x - origins[t][1] + w])
def _bin(prob, gt, hist):
    key = scoring.score_key(prob).ravel()
    for cls in (0, 1):
        hist[cls] += torch.from_numpy(np.bincount(key[gt.ravel() == cls], minlength=_lib.PR_BINS).astype(np.int32))
def pr_hist_rects(prob, gt, rects, hist, strad):
    for (y, x, h, w) in rects:
        _bin(prob.numpy()[y:y + h, x:x + w], gt.numpy()[y:y + h, x:x + w], hist)
def pr_hist(prob, gt, hist=None, strad=None, splits=0):
    _bin(prob.numpy(), gt.numpy(), hist[0])
    return hist, strad
K.preprocess_tile, K.paste_tiles_owned_x2, K.pr_hist_rects, K.pr_hist = preprocess_tile, paste_tiles_owned_x2, pr_hist_rects, pr_hist

class Pointwise(torch.nn.Module):
    def forward(self, x):
        return x[:, 0:1] * 0.7 - x[:, 1:2] * 0.3 + x[:, 2:3] * 0.1
model, tfm = Pointwise(), tta.aliases.d4_transform()
S = 64
mean, std = pipeline.DATASET_STATS['IDRiD']
rng = np.random.default_rng(8)
shapes = [(300, 420), (280, 302), (330, 290)]
images = [torch.from_numpy(rng.integers(0, 256, size=s + (3,), dtype=np.uint8)) for s in shapes]
gts = [torch.from_numpy((rng.random(s) < 0.2).astype(np.uint8)) for s in shapes]
hist = torch.zeros((len(shapes), 2, _lib.PR_BINS), dtype=torch.int32)
strad = torch.zeros((len(shapes), _lib.PR_NTHRESH, 2), dtype=torch.int32)
canvases, nxt = drv.partitioned_group(model, tfm, images, gts, S, mean, std, hist, strad, 0, rank, 2, tiles_per_batch=4)
partition.allreduce_sum_(hist)
for c in canvases:
    dist.all_reduce(c)
ok_units = nxt == sum(drv.tile_plan(s[0], s[1], S).n for s in shapes)
ok_map, ok_hist = True, True
for k, s in enumerate(shapes):
    want = pipeline.tiled_probability_map(images[k].numpy(), model, S, mean, std, 'd4')
    ok_map &= bool(np.abs(canvases[k].numpy() - want).max() < 1e-6)
    full = torch.zeros((2, _lib.PR_BINS), dtype=torch.int32)
    _bin(canvases[k].numpy(), gts[k].numpy(), full)
    ok_hist &= bool(torch.equal(hist[k], full))
mine = len([u for u in range(nxt) if u % 2 == rank])
print('RESULT' + json.dumps(dict(ok_units=bool(ok_units), ok_map=ok_map, ok_hist=ok_hist, mine=mine, total=int(nxt))))
dist.destroy_process_group()
"""


def test_two_rank_partitioned_group_on_cpu_equals_the_oracle_pipeline(tmp_path):
    """The REAL _driver.partitioned_group under gloo, world size 2, with numpy stand-ins for the five CUDA entry
    points it calls: the two ranks' canvases sum to oracle/pipeline.py's single-process map (the reference's tile
    loop restated), the all-reduced integer histograms equal the histogram of that map bin for bin, and the
    (image, tile) units split evenly."""
    import json
    port = 29120 + os.getpid() % 300
    code = _GROUP_WORKER.format(root=ROOT, port=port)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True) for r in range(2)]
    seen = []
    for p in procs:
        out, err = p.communicate(timeout=600)
        assert p.returncode == 0, err[-3000:]
        res = json.loads([ln for ln in out.splitlines() if ln.startswith("RESULT")][0][6:])
        assert res["ok_units"] and res["ok_map"] and res["ok_hist"], res
        seen.append(res["mine"])
    assert sum(seen) == res["total"] and abs(seen[0] - seen[1]) <= 1


_PRODUCER_WORKER = _GROUP_WORKER.split("class Pointwise")[0] + r"""
def pr_scan(hist, strad):
    # totals exact, AP / ROC read off the bins as sklearn does on key-quantised scores
    from sklearn.metrics import average_precision_score, roc_auc_score
    n = hist.shape[0]
    ap, roc = np.full(n, np.nan), np.full(n, np.nan)
    counts = torch.zeros((n, _lib.PR_NTHRESH, 2), dtype=torch.int64)
    totals = torch.zeros((n, 2), dtype=torch.int64)
    for i in range(n):
        neg, pos = hist[i, 0].numpy().astype(np.int64), hist[i, 1].numpy().astype(np.int64)
        totals[i, 0], totals[i, 1] = int(pos.sum()), int(neg.sum())
        if pos.sum() and neg.sum():
            keys = np.arange(_lib.PR_BINS)
            y = np.concatenate([np.ones(_lib.PR_BINS), np.zeros(_lib.PR_BINS)])
            s = np.concatenate([keys, keys]); w = np.concatenate([pos, neg]).astype(float)
            ap[i] = average_precision_score(y, s, sample_weight=w)
            roc[i] = roc_auc_score(y, s, sample_weight=w)
    return torch.from_numpy(ap), torch.from_numpy(roc), counts, totals
K.pr_scan = pr_scan
drv.device = lambda: torch.device('cpu')
_reduce = dist.reduce
class Pointwise(torch.nn.Module):
    def forward(self, x):
        return x[:, 0:1] * 0.7 - x[:, 1:2] * 0.3 + x[:, 2:3] * 0.1
model, tfm = Pointwise(), tta.aliases.d4_transform()
S = 64
mean, std = pipeline.DATASET_STATS['IDRiD']
rng = np.random.default_rng(8)
shapes = [(300, 420), (280, 302), (330, 290)]          # three images, two ranks: a ragged last group
data = {{f'img{{i}}': (rng.integers(0, 256, size=s + (3,), dtype=np.uint8), (rng.random(s) < 0.2).astype(np.uint8))
        for i, s in enumerate(shapes)}}
if {empty_last}:
    data['img2'][1][:] = 0                              # an image without positives
loads = []
def load(key):
    loads.append(key)
    return data[key]
produce = drv.partitioned_producer(model, tfm, sorted(data), load, S, mean, std, tiles_per_batch=4)
items = list(produce())
from eyediseasesegmentation_b200 import aucpr
auc = aucpr.get_auc(items, dict())
want = {{k: pipeline.tiled_probability_map(v[0], model, S, mean, std, 'd4') for k, v in data.items()}}
ok = True
held = []
for (pred, gt, name) in items:
    assert pred._eds_scores.replicated
    if np.asarray(pred).size:
        held.append(name)
        ok &= bool(np.abs(np.asarray(pred) - want[name]).max() < 1e-6) and bool(np.array_equal(gt, data[name][1]))
    else:
        ok &= gt is None
ref = scoring.get_auc([(scoring.score_key(want[k]).astype(np.float64), data[k][1], k) for k in sorted(data)])
print('RESULT' + json.dumps(dict(ok=bool(ok), names=[n for _, _, n in items], held=held, loads=loads, auc=auc, ref=ref)))
dist.destroy_process_group()
"""


@pytest.mark.parametrize("empty_last", [False, True])
def test_two_rank_partitioned_producer_on_cpu(tmp_path, empty_last):
    """_driver.partitioned_producer (the generator behind tta_patches under torchrun) on two gloo ranks with numpy
    stand-ins for the CUDA entry points: each rank decodes only its images of a group, every rank yields EVERY image
    with the global (replicated) scores, the full-resolution map lives on exactly one rank and equals the oracle's
    tile loop, and get_auc returns the same global mean on both ranks without summing over ranks again."""
    import json
    port = 29420 + os.getpid() % 300 + (7 if empty_last else 0)
    code = _PRODUCER_WORKER.format(root=ROOT, port=port, empty_last=empty_last)
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                              text=True) for r in range(2)]
    results = []
    for p in procs:
        out, err = p.communicate(timeout=600)
        assert p.returncode == 0, err[-3000:]
        results.append(json.loads([ln for ln in out.splitlines() if ln.startswith("RESULT")][0][6:]))
    for r in results:
        assert r["ok"] and r["names"] == ["img0", "img1", "img2"]
        assert abs(r["auc"] - r["ref"]) < 1e-9 and abs(r["auc"] - results[0]["auc"]) < 1e-15
    assert sorted(results[0]["held"] + results[1]["held"]) == ["img0", "img1", "img2"]
    assert results[0]["loads"] == ["img0", "img2"] and results[1]["loads"] == ["img1"]
