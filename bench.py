#!/usr/bin/env python
"""Benchmark of the inference-and-scoring hot path (BASELINE.json metric).

Workload ("cfg4", SURVEY.md 8d-4): a FIXED SET of synthetic IDRiD-shaped 2848x4288 RGB fundus images (one per
step), four single-class lesion models (EX/HE/MA/SE) of the proposed UNet++* (base_dim 32), sliding window
(2048 px windows -> 1024^2 tiles, 6 tiles per image), D4 8-view TTA, sigmoid, x2 bilinear paste, per-image
PR/ROC histogram + scan.  One step = one image through all four lesion models (6 * 8 * 4 = 192 network
forwards = 359.5 algorithmic TFLOP).  metric = images per second.

Multi-GPU (SURVEY.md 8e): STRONG scaling -- the same `steps` images whatever N is; their (image, tile) units are
dealt round-robin to the ranks, every rank pastes / histograms only the pixels its tiles own, and ONE all-reduce
sums the per-image integer histograms before every rank scans them.

  python bench.py [--gpus N --steps K --warmup W]          B200 path (one rank per GPU under torchrun)
  python bench.py [...] --dump-outputs DIR                 + the last timed image's maps (sample) and scores as .npy
  python bench.py --impl reference [...]                   the reference's CPU path (oracle port) on host cores

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how each field is obtained.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

H, W, S = 2848, 4288, 1024
LESIONS = ("EX", "HE", "MA", "SE")
PREVALENCE = {"EX": 0.01, "HE": 0.01, "MA": 0.001, "SE": 0.005}
TILES, VIEWS = 6, 8
GFLOP_PER_FORWARD = 1872.19                      # BASELINE.md section 2 (reference modules, FLOP = 2*MAC)
TFLOP_PER_IMAGE = TILES * VIEWS * len(LESIONS) * GFLOP_PER_FORWARD / 1e3
METRIC = "IDRiD-size (2848x4288) fundus images/s, 4 lesion models, sliding-window + 8-view D4 TTA + AUC-PR"
WORKLOAD = ("cfg4: fixed set of `steps` distinct 2848x4288 images x 4 lesion models (proposed UNet++*, base_dim 32, "
            "random init), 6 tiles of 1024^2 x 8 D4 views each, sigmoid + x2 paste + PR histogram/scan")
# DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu --set full captures
TRAFFIC = {
    "conv": {"bytes": 1115.83e6 + 252.90e6, "source": "profiles/r02_kernels_full.md #0 (conv_igemm 1024->256 @256^2 x8: "
             "1074 MB algorithmic)"},
    "hist": {"bytes": 1653.80e6 + 4.69e6, "source": "profiles/r02_hist_full.md #0 (27 images, 1648.7 MB algorithmic)"},
    "blend": {"bytes": 108.50e6 + 18.03e6, "source": "profiles/r02_blend_fused_full.md #0 (tta_blend_x2: blocks under a later "
              "tile are not read; most of the 48.8 MB of stores are still in L2 when the kernel ends)"},
}


def star_cfg(base_dim=32):
    return dict(classes=1, decoder_attention_type="scse", decoder_use_batchnorm=True, base_dim=base_dim,
                encoder_depth=5, encoder_name="BoTSER50_Axial_scratch", deep_supervision=False,
                drop_block_prob=0.0, clf_head=False)


def synth_image_device(seed, dev):
    """uint8 noise inside a centred disc of radius 1400, black outside (fundus-like), + 4 blob masks, generated on
    the device from a seed: every rank builds the SAME image i (the partition needs identical inputs everywhere)."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(1999 + seed)
    img = torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, device=dev, generator=g)
    yy = torch.arange(H, device=dev, dtype=torch.float32).view(H, 1) - H / 2
    xx = torch.arange(W, device=dev, dtype=torch.float32).view(1, W) - W / 2
    disc = (yy * yy + xx * xx) <= 1400.0 ** 2
    img = img * disc.unsqueeze(-1).to(torch.uint8)
    masks = {}
    for les in LESIONS:
        coarse = torch.rand((H // 16, W // 16), device=dev, generator=g) < PREVALENCE[les]    # Bernoulli blobs of 16x16 px
        m = coarse.repeat_interleave(16, dim=0).repeat_interleave(16, dim=1) & disc
        if les == "SE" and seed % 9 == 4:
            m = torch.zeros_like(m)                # a few images without soft exudates (aucpr.py:22 skips them)
        masks[les] = m.to(torch.uint8).contiguous()
    return img.contiguous(), masks


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ B200 arm
def _claim_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line there.
    Point fd 1 at stderr for the whole run and return a handle on the real stdout for the final line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def run_b200(args):
    real_stdout = _claim_stdout()
    import torch
    import torch.distributed as dist
    from eyediseasesegmentation_b200 import archs, kernels as K, _driver as drv, _lib, partition, ttach_compat as tta
    from eyediseasesegmentation_b200.archs import get_preprocessing_fn

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)

    _, mean, std = get_preprocessing_fn("IDRiD", False)
    tfm = tta.aliases.d4_transform()
    models = {}
    for i, les in enumerate(LESIONS):
        torch.manual_seed(1999 + i)
        m = archs.get_model("unetplusplusstar", star_cfg(32), training=False).to(dev).eval()
        m.precision = "bf16"
        m.engine()
        models[les] = m

    # the fixed image set: `steps` distinct images for the timed region, `warmup` more for the warm-up set
    n_set = max(args.steps, args.warmup)
    dev_imgs, dev_masks = [], []
    for j in range(n_set):
        img, masks = synth_image_device(j, dev)
        dev_imgs.append(img)
        dev_masks.append(masks)
    host_imgs = [t.cpu().pin_memory() for t in dev_imgs]
    host_masks = [{les: t.cpu().pin_memory() for les, t in d.items()} for d in dev_masks]
    pinned_out = {les: [torch.empty((H, W), dtype=torch.float32).pin_memory() for _ in range(2)] for les in LESIONS}
    pinned_scores = torch.empty((len(LESIONS), n_set, 2 + 2 * 19 + 2), dtype=torch.float64).pin_memory()
    allreduce_ms = []
    up_stream, down_stream = torch.cuda.Stream(), torch.cuda.Stream()

    # images whose (image, tile) units are dealt together: the whole set while its canvases fit comfortably (the
    # units then balance to within one tile per rank and the batches have one shape); the file drivers use
    # groups of `world` images because they decode and broadcast as they go
    group_size = args.group if args.group > 0 else (n_set if n_set <= 64 else world)

    def run_set(count, host):
        """`count` images of the set (strong scaling: the same images for every N), (image, tile) units over
        the ranks in groups of `world` images.  host=False: inputs resident in HBM, results stay on the device
        (value).  host=True: each group's images + masks come from pinned host memory, the assembled
        probability maps and the scores go back to pinned host memory (e2e).
        -> (scores per lesion model, {lesion: this rank's pieces of the probability map of image count-1})"""
        hist = torch.zeros((len(LESIONS), count, 2, _lib.PR_BINS), dtype=torch.int32, device=dev)
        strad = torch.zeros((len(LESIONS), count, _lib.PR_NTHRESH, 2), dtype=torch.int32, device=dev)
        main = torch.cuda.current_stream()
        # host mode: groups of max(N, 4) images so that the upload of group g+1 (copy stream) and the download of
        # finished maps (another copy stream) overlap the compute of group g; the units of a group still balance
        gs = group_size if not host else max(world, 4)
        starts = list(range(0, count, gs))

        def upload(g):
            group = list(range(g, min(g + gs, count)))
            with torch.cuda.stream(up_stream):
                imgs = [host_imgs[i].to(dev, non_blocking=True) for i in group]
                gts = {les: [host_masks[i][les].to(dev, non_blocking=True) for i in group] for les in LESIONS}
                ev = torch.cuda.Event()
                ev.record(up_stream)
            return group, imgs, gts, ev

        pending = upload(starts[0]) if host else None
        last_maps = {}
        for gi, g in enumerate(starts):
            if host:
                group, imgs, gts, ev = pending
                main.wait_event(ev)
                for t_ in imgs + [m for les in LESIONS for m in gts[les]]:
                    t_.record_stream(main)
                pending = upload(starts[gi + 1]) if gi + 1 < len(starts) else None
            else:
                group = list(range(g, min(g + gs, count)))
                imgs = [dev_imgs[i] for i in group]
                gts = {les: [dev_masks[i][les] for i in group] for les in LESIONS}
            for li, les in enumerate(LESIONS):
                canvases, _ = drv.partitioned_group(models[les], tfm, imgs, gts[les], S, mean, std, hist[li], strad[li],
                                                    g, rank, world, args.tiles, unit_offset=g * TILES)
                if group[-1] == count - 1:
                    last_maps[les] = canvases[-1]
                if host:
                    for r, i in enumerate(group):
                        if world > 1:
                            dist.reduce(canvases[r], dst=i % world, op=dist.ReduceOp.SUM)   # pieces -> the writer rank
                    down_stream.wait_stream(main)
                    with torch.cuda.stream(down_stream):
                        for r, i in enumerate(group):
                            if i % world == rank:
                                pinned_out[les][(i // world) % 2].copy_(canvases[r], non_blocking=True)
                                canvases[r].record_stream(down_stream)
        if host:
            main.wait_stream(down_stream)
        if world > 1:                              # the path's single data collective: per-image integer histograms
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            partition.allreduce_sum_(hist, strad)
            a1.record()
        out = [K.pr_scan(hist[li], strad[li]) for li in range(len(LESIONS))]
        if host:
            for li, (ap, roc, counts, totals) in enumerate(out):
                pinned_scores[li, :count, 0].copy_(ap, non_blocking=True)
                pinned_scores[li, :count, 1].copy_(roc, non_blocking=True)
                pinned_scores[li, :count, 2:40].copy_(counts.reshape(count, -1).to(torch.float64), non_blocking=True)
                pinned_scores[li, :count, 40:42].copy_(totals.to(torch.float64), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        if world > 1:
            torch.cuda.current_stream().synchronize()
            allreduce_ms.append(a0.elapsed_time(a1))
        return out, last_maps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def prewarm():
        """Untimed: every batch shape of the timed plan runs three times per model (eager, graph capture, replay),
        so that no CUDA graph is captured inside a timed region."""
        sizes = set()
        for count in {args.steps, args.warmup}:
            for gs in {group_size, max(world, 4)}:          # resident run / host run (see run_set)
                for g in range(0, count, gs):
                    n_units = (min(g + gs, count) - g) * TILES
                    mine = [u for u in range(n_units) if (g * TILES + u) % world == rank]
                    sizes |= {len(b) for b in partition.batches(mine, args.tiles)}
        deaug = drv.fused_blend_views(models[LESIONS[0]], tfm, S, W)       # the forward the tile path will call
        for les in LESIONS:
            for b in sorted(sizes):
                x = torch.zeros((b, 3, S, S), device=dev)
                for _ in range(3):
                    if deaug is not None:
                        models[les].forward_tta(x, tfm, merge=False)
                    else:
                        drv.predict_probs(models[les], tfm, x)
        if world > 1:                              # lazy NCCL channel set-up of the collectives used below
            w0 = torch.zeros((4, 4), dtype=torch.int32, device=dev)
            partition.allreduce_sum_(w0)
            dist.reduce(torch.zeros((4, 4), device=dev), dst=0)

    def timed(host):
        if args.warmup:
            run_set(args.warmup, host)             # W warm-up steps (images)
        barrier()
        before = K.LAUNCHES[0]
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        out, maps = run_set(args.steps, host)      # EXACTLY `steps` images
        t1.record()
        barrier()
        launches = K.LAUNCHES[0] - before
        ms = torch.tensor([t0.elapsed_time(t1), float(launches)], dtype=torch.float64, device=dev)
        if world > 1:
            mx = ms.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(ms, op=dist.ReduceOp.SUM)
            return float(mx[0]), int(ms[1]), out, maps
        return float(ms[0]), int(ms[1]), out, maps

    # the two HBM-bound kernels are timed ALONE, before the long tensor-bound run puts the GPU under its power cap
    # (their denominator is the burst copy bandwidth of MEASURED_PEAKS.json, also measured on an otherwise idle GPU)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tensor_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "measured (MEASURED_PEAKS.json; sustained bf16 figure, HBM copy figure)" if peaks else \
        "fallback (B200_PROFILING.md)"
    hist_roof = blend_roof = None
    if rank == 0:
        hist_roof = hist_roofline(dev, hbm_peak, peak_src)
        blend_roof = blend_roofline(dev, hbm_peak, peak_src)
    prewarm()
    sampler = ClockSampler(local) if rank == 0 else None
    ms_total, launches, out, maps = timed(False)
    clocks = sampler.stop() if sampler else None
    ar_ms = allreduce_ms[-1] if allreduce_ms else 0.0
    ms_e2e, _, _, _ = timed(True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, maps, rank, world)

    line = None
    if rank == 0:
        value = args.steps / (ms_total / 1e3)
        e2e = args.steps / (ms_e2e / 1e3)
        roof, shares = conv_roofline(models["EX"], tfm, dev_imgs[0], mean, std, args.tiles, tensor_peak, peak_src)
        ap_mean = [float(torch.nanmean(o[0]).item()) for o in out]
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "tiles_per_batch": args.tiles,
                       "algorithmic_tflop_per_image": TFLOP_PER_IMAGE,
                       "achieved_algorithmic_tflops_per_gpu": TFLOP_PER_IMAGE * value / world,
                       "l2": "working set per tile batch (>5 GB of activations) far exceeds the 126 MB L2; every image of "
                             "the set is distinct",
                       "parallelism": f"(image, tile) units round-robin over {world} rank(s); ONE all-reduce of the "
                                      f"per-image integer histograms [4 x {args.steps} x 2 x {_lib.PR_BINS}] int32",
                       "images_per_group": group_size, "allreduce_ms": ar_ms,
                       "allreduce_ms_note": "device time of the collective on rank 0: transfer (~0.2 ms) + waiting for the "
                                            "slowest rank",
                       "mean_ap_per_lesion": ap_mean},
            "e2e": {"value": e2e, "unit": "images/s",
                    "h2d_bytes_per_step": world * (H * W * 3 + len(LESIONS) * H * W),
                    "d2h_bytes_per_step": len(LESIONS) * (H * W * 4 + 42 * 8),
                    "what": "groups of max(N, 4) images: each rank uploads the group's images + masks from pinned host "
                            "memory (copy stream, one group ahead); the owned pieces of the probability maps are summed "
                            "onto one rank per image (NCCL) and copied to pinned host memory (second copy stream) with "
                            "the scores"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_hist": hist_roof,
            "roofline_blend": blend_roof, "time_shares": shares,
        }
        if not args.no_extra and world == 1:
            line["other_configs"] = other_configs(dev)
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), file=real_stdout, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


DUMP_SAMPLE = 1 << 20                            # pixels per probability map in --dump-outputs (4 MB each)


def dump_outputs(directory, out, maps, rank, world):
    """--dump-outputs: what the resident timed run returned for its last image (step `steps`), per lesion model:
    the same fixed sample of DUMP_SAMPLE pixels (numpy default_rng(0), row-major order) of the full-resolution
    probability map as <lesion>_prob_sample.npy (float32), and the image's scores as float64: <lesion>_ap.npy,
    <lesion>_roc.npy, <lesion>_threshold_counts.npy ([19, 2]: tp, pp per threshold), <lesion>_totals.npy
    (n_pos, n_neg).  Under torchrun every rank holds only the pixels its tiles own: the pieces are summed onto
    rank 0, which writes.  Two runs of one build are not bit-identical: the SE / SCSE channel means are summed with
    float atomics in varying order (measured on a B200 at 1000 W, --steps 3 --warmup 2: up to 1.9e-3 in a
    probability, 23 pixels in a threshold count, 1.2e-6 in an AP)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    idx = np.sort(np.random.default_rng(0).choice(H * W, DUMP_SAMPLE, replace=False))
    arrays = {}
    for li, les in enumerate(LESIONS):
        canvas = maps[les]
        if world > 1:
            dist.reduce(canvas, dst=0, op=dist.ReduceOp.SUM)
        if rank != 0:
            continue
        flat = canvas[:, :W].reshape(-1)           # canvas rows are padded to a multiple of 4 columns
        ap, roc, counts, totals = (t[-1] for t in out[li])
        arrays[f"{les}_prob_sample"] = flat[torch.from_numpy(idx).to(flat.device)].float().cpu().numpy()
        arrays[f"{les}_ap"] = ap.cpu().numpy()
        arrays[f"{les}_roc"] = roc.cpu().numpy()
        arrays[f"{les}_threshold_counts"] = counts.to(torch.float64).cpu().numpy()
        arrays[f"{les}_totals"] = totals.to(torch.float64).cpu().numpy()
    if rank == 0:
        os.makedirs(directory, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(directory, name + ".npy"), a)


def conv_roofline(model, tfm, image, mean, std, tiles, peak, peak_src):
    """Dominant kernels = the tcgen05 convolutions.  One instrumented (eager) tile batch with a CUDA event after
    every launch on the launching stream: achieved = algorithmic FLOPs of the conv launches (2*M*Cout*K with M =
    real output pixels) / their summed device time; the same trace gives the time share of every kernel class."""
    import torch
    from eyediseasesegmentation_b200 import kernels as K, _driver as drv
    drv.tiled_probability_map(model, tfm, image, S, mean, std, tiles_per_batch=tiles)   # warm
    torch.cuda.synchronize()
    K.CONV_TRACE = []
    drv.tiled_probability_map(model, tfm, image, S, mean, std, tiles_per_batch=tiles)
    torch.cuda.synchronize()
    trace, K.CONV_TRACE = K.CONV_TRACE, None
    flops = sum(t[0] for t in trace)
    ms = sum(t[1].elapsed_time(t[2]) for t in trace)
    achieved = flops / (ms / 1e3) / 1e12
    # per-class shares: consecutive events on the stream
    K.KERNEL_TRACE = []
    start = torch.cuda.Event(enable_timing=True)
    start.record()
    drv.tiled_probability_map(model, tfm, image, S, mean, std, tiles_per_batch=tiles)
    torch.cuda.synchronize()
    ktrace, K.KERNEL_TRACE = K.KERNEL_TRACE, None
    per, prev = {}, start
    for name, ev in ktrace:
        per[name] = per.get(name, 0.0) + prev.elapsed_time(ev)
        prev = ev
    total = sum(per.values()) or 1.0
    shares = {k: round(v / total, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}
    shares["_note"] = ("device time between consecutive launch events of ONE eager tile batch (48 maps), by wrapper; "
                       f"total {total:.1f} ms")
    roof = {"kernel": "conv_igemm_kernel + conv3x3_wide_kernel + conv3x3_halo_kernel (tcgen05 implicit GEMM) + "
                      "conv3x3_small_kernel (16-channel tail): every convolution launch of a pass",
            "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": TRAFFIC["conv"]["bytes"], "traffic_source": TRAFFIC["conv"]["source"],
            "launches": len(trace), "avg_launch_ms": ms / max(1, len(trace)), "peak_source": peak_src,
            "flops_counted": flops}
    return roof, shares


def hist_roofline(dev, peak, peak_src):
    """AUC-PR kernel GB/s: the whole 27-image test set in one launch (SURVEY.md 8d), algorithmic bytes =
    n_px * (4 B score + 1 B label); uniform random scores (every pixel its own bin: the hardest case)."""
    import torch
    from eyediseasesegmentation_b200 import kernels as K
    n_img = 27
    prob = torch.rand((n_img, H * W), device=dev)
    gt = (torch.rand((n_img, H * W), device=dev) < 0.01).to(torch.uint8)
    hist, strad = K.pr_hist(prob, gt)
    torch.cuda.synchronize()
    times = []
    for _ in range(5):
        hist.zero_(); strad.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        K.pr_hist(prob, gt, hist, strad)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    ms = sorted(times)[len(times) // 2]
    gbs = n_img * H * W * 5 / (ms / 1e3) / 1e9
    return {"kernel": "pr_hist_kernel", "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s",
            "frac": gbs / peak, "traffic": TRAFFIC["hist"]["bytes"], "traffic_source": TRAFFIC["hist"]["source"],
            "launch_ms": ms, "images_per_launch": n_img, "algorithmic_bytes": n_img * H * W * 5, "peak_source": peak_src}


def blend_roofline(dev, peak, peak_src):
    """The blend of SURVEY.md 8d: TTA de-augment + mean + sigmoid over V*B logit maps, x2 bilinear, overwrite-paste of
    the B tiles -- ONE kernel (tta_blend_x2_kernel) at the bench shape (V=8, B=6, S=1024) for the 4 lesion models of
    one image, back to back as in a step (4 x 201 MB of logits: larger than L2, and L2 is flushed before each
    repetition).  Algorithmic bytes per tile (8d) = V*S^2*4 read + (2S)^2*4 write = 50.3 MB, x 6 tiles per launch.
    `moved` = what the kernel really touches: blocks under a later tile are neither read nor written.  The
    two-kernel form (tta_merge64 + paste_tiles_x2, the fallback for tile sizes that are not multiples of 64) and
    the device's pure-write bandwidth (memset) are timed beside it."""
    import torch
    from eyediseasesegmentation_b200 import kernels as K, partition, ttach_compat as tta
    from eyediseasesegmentation_b200.util import make_grid
    V, B, M = VIEWS, TILES, len(LESIONS)
    _, deaug = tta.view_maps(tta.aliases.d4_transform(), S, S)
    logits = [torch.randn((V, B, S, S), device=dev) for _ in range(M)]
    prob = [torch.empty((B, S, S), device=dev) for _ in range(M)]
    preds = [torch.zeros((H, W), device=dev) for _ in range(M)]
    slices = make_grid((H, W), window=2 * S, min_overlap=32)
    origins = [(int(x1), int(y1)) for (x1, _, y1, _) in slices]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)        # > L2

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / M)
        return sorted(ts)[2]

    def fused():
        for m in range(M):
            K.tta_blend_x2(logits[m], deaug, preds[m], origins)

    def pair():
        for m in range(M):
            K.tta_merge(logits[m], deaug, True, out=prob[m])
            K.paste_tiles_x2(prob[m], preds[m], origins)

    def merge_only():
        for m in range(M):
            K.tta_merge(logits[m], deaug, True, out=prob[m])

    ms_fused, ms_pair, ms_merge = timed(fused), timed(pair), timed(merge_only)
    big = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    M1 = M
    M = 1
    ms_write = timed(lambda: big.zero_())
    M = M1
    bytes_8d = B * (V * S * S * 4 + (2 * S) * (2 * S) * 4)
    # blocks (64 x 64 of a tile = 128 x 128 of its window) not completely under a later tile, and owned pixels
    cells = partition.owned_cells([(y, y + 2 * S, x, x + 2 * S) for (y, x) in origins], (H, W))
    owned_px = sum(h * w for rects in cells for (_, _, h, w) in rects)
    live_blocks = 0
    for t, (y, x) in enumerate(origins):
        for by in range(0, 2 * S, 128):
            for bx in range(0, 2 * S, 128):
                covered = any(y + by >= ly and y + by + 128 <= ly + 2 * S and x + bx >= lx and x + bx + 128 <= lx + 2 * S
                              for (ly, lx) in origins[t + 1:])
                live_blocks += 0 if covered else 1
    moved = live_blocks * 64 * 64 * 4 * V + owned_px * 4
    gbs = bytes_8d / (ms_fused / 1e3) / 1e9
    return {"kernel": "tta_blend_x2_kernel (views -> preds: de-augment + mean + sigmoid + x2 bilinear + ownership, one launch "
                      "per image and lesion model)",
            "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
            "traffic": TRAFFIC["blend"]["bytes"], "traffic_source": TRAFFIC["blend"]["source"],
            "moved_bytes": moved, "moved_note": "computed: logits of the blocks not under a later tile + owned pixels written",
            "launch_ms": ms_fused, "algorithmic_bytes": bytes_8d, "launches_timed": M, "peak_source": peak_src,
            "moved_gbs": moved / (ms_fused / 1e3) / 1e9,
            "l2": "256 MB written before each repetition (flush); 4 x 201 MB of logits per repetition",
            "two_kernel_form": {"kernels": "tta_merge64_kernel + paste_tiles_x2_kernel", "ms": ms_pair,
                                "achieved": bytes_8d / (ms_pair / 1e3) / 1e9, "unit": "GB/s",
                                "merge_only_ms": ms_merge,
                                "merge_only_gbs": (V * B * S * S * 4 + B * S * S * 4) / (ms_merge / 1e3) / 1e9},
            "pure_write_gbs": (1 << 30) / (ms_write / 1e3) / 1e9}


def other_configs(dev):
    """The other BASELINE.json configurations at their stated sizes on one GPU (parity: tests/test_configs_gpu.py):
    cfg-1 smp.Unet(resnet34) fp32 1x3x512x512; cfg-2 UNet++ se_resnet50 + scse, 16 x 1024^2, 4-view flip, bf16;
    cfg-5 vessel: proposed net at 608^2 (base_dim 19) and 1024^2, D4, ROC + PR histogram."""
    import torch
    import helpers
    from eyediseasesegmentation_b200 import kernels as K, ttach_compat as tta

    def timeit(fn, n=3):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    out = {}
    m = helpers.build_product_model("Unet", dict(encoder_name="resnet34", encoder_weights=None, classes=1)).to(dev)
    m.precision = "fp32"
    x = torch.randn(1, 3, 512, 512, device=dev)
    ms = timeit(lambda: m(x), n=5)
    out["cfg1_unet_r34_fp32_512"] = {"ms_per_forward": ms, "gflop": 62.51, "tflops": 62.51 / ms}
    del m
    se50 = dict(encoder_name="se_resnet50", encoder_weights=None, classes=1, decoder_attention_type="scse",
                deep_supervision=True)
    m = helpers.build_product_model("unetplusplus_deepsup", se50).to(dev)
    m.precision = "bf16"
    x = torch.randn(16, 3, 1024, 1024, device=dev)
    flip = tta.aliases.flip_transform()
    ms = timeit(lambda: m.forward_tta(x, flip, apply_sigmoid=True), n=3)
    out["cfg2_uppse50_bf16_16x1024_flip"] = {"ms_per_batch": ms, "images_per_s": 16 / (ms / 1e3), "tflop_per_batch": 117.1,
                                             "tflops": 117.1 / (ms / 1e3)}
    del m, x
    d4 = tta.aliases.d4_transform()
    for size, bd, gflop in ((608, 19, 659.73), (1024, 32, 1872.19)):
        m = helpers.build_product_model("unetplusplusstar", star_cfg(bd)).to(dev)
        m.precision = "bf16"
        x = torch.randn(1, 3, size, size, device=dev)
        gt = (torch.rand(1, size * size, device=dev) < 0.1).to(torch.uint8)

        def one():
            prob = m.forward_tta(x, d4, apply_sigmoid=True)
            h, s = K.pr_hist(prob.reshape(1, -1), gt)
            return K.pr_scan(h, s)
        ms = timeit(one, n=5)
        out[f"cfg5_vessel_star_bd{bd}_{size}_d4"] = {"ms_per_image": ms, "images_per_s": 1e3 / ms,
                                                    "tflops": 8 * gflop / ms}
        del m
    out["e2e_from_files"] = from_files(dev)
    return out


def from_files(dev, n_images=4):
    """JPEG files on disk -> scores (SURVEY.md 8f-2): the per-image loop of tta_patches for ONE lesion model --
    PIL decode of image and mask on the host, upload, 6 tiles x 8 views, paste, histogram + scan, map and scores back
    -- with the decode of image k+1 prefetched on a background thread (the product path) and serial (as the
    reference does it, tta.py:192-203).  Smooth synthetic fundus images (JPEG of white noise decodes atypically)."""
    import tempfile
    import numpy as np
    import torch
    from PIL import Image
    import helpers
    from eyediseasesegmentation_b200 import _driver as drv, ttach_compat as tta
    from eyediseasesegmentation_b200.archs import get_preprocessing_fn
    _, mean, std = get_preprocessing_fn("IDRiD", False)
    tfm = tta.aliases.d4_transform()
    model = helpers.build_product_model("unetplusplusstar", star_cfg(32)).to(dev)
    model.precision = "bf16"
    rng = np.random.default_rng(0)
    with tempfile.TemporaryDirectory() as tmp:
        paths = []
        yy, xx = np.mgrid[:H, :W]
        disc = (yy - H / 2) ** 2 + (xx - W / 2) ** 2 <= 1400 ** 2
        for i in range(n_images):
            low = rng.integers(0, 256, size=(H // 32, W // 32, 3), dtype=np.uint8)
            img = np.asarray(Image.fromarray(low).resize((W, H), Image.BICUBIC)).copy()
            img[~disc] = 0
            m = (np.kron(rng.random((H // 16, W // 16)) < 0.01, np.ones((16, 16), dtype=bool)) & disc).astype(np.uint8) * 255
            Image.fromarray(img).save(os.path.join(tmp, f"img{i}.jpg"), quality=92)
            Image.fromarray(m, "L").save(os.path.join(tmp, f"img{i}_EX.tif"))
            paths.append((os.path.join(tmp, f"img{i}.jpg"), os.path.join(tmp, f"img{i}_EX.tif")))

        def load(p):
            return drv.read_rgb(p[0]), drv.read_mask(p[1], 0)

        def run(prefetch):
            loaded = drv.prefetched([(lambda p=p: load(p)) for p in paths]) if prefetch else (load(p) for p in paths)
            t0 = time.perf_counter()
            for image, gt in loaded:
                drv.infer_image_host(model, tfm, torch.from_numpy(image), torch.from_numpy(gt), S, mean, std, copy=False)
            torch.cuda.synchronize()
            return time.perf_counter() - t0

        t0 = time.perf_counter()
        for p in paths:
            load(p)
        decode_s = (time.perf_counter() - t0) / n_images
        run(True)                                   # warm (graph capture)
        serial, overlapped = run(False), run(True)
    return {"what": "one lesion model, JPEG + TIFF files on disk -> probability map and scores on the host",
            "decode_s_per_image": decode_s, "images_per_s_serial_decode": n_images / serial,
            "images_per_s_prefetched_decode": n_images / overlapped, "images": n_images}


# ------------------------------------------------------------------------------ CPU baseline / reference arm
_CPU_STATE = {}


def _cpu_setup(threads, size=S):
    import torch
    from oracle import nets
    import helpers
    if "sd" not in _CPU_STATE:
        torch.set_num_threads(threads)
        # the proposed network ties its attention length to the input size: base_dim = size / 32 (32 <-> 1024^2)
        model = helpers.build_product_model("unetplusplusstar", star_cfg(size // 32), seed=1999)
        _CPU_STATE["sd"] = model.state_dict()
        _CPU_STATE["x"] = torch.randn(1, 3, size, size, generator=torch.Generator().manual_seed(0))
    return _CPU_STATE["sd"], _CPU_STATE["x"]


def cpu_tile_sample(threads, views=VIEWS, size=S):
    """One REAL unit of the workload on the host cores with the oracle (the reference's PyTorch path restated,
    oracle/nets.py + sklearn): ONE 1024^2 tile through all `views` D4 views of the proposed network with the TTA mean
    and the sigmoid (tta.py:209-210) -> seconds."""
    import torch
    from oracle import nets
    sd, x = _cpu_setup(threads, size)
    kind = "d4" if views == 8 else "none"
    t0 = time.perf_counter()
    with torch.no_grad():
        torch.sigmoid(nets.tta_mean_logits(lambda t: nets.unetplusplusstar_forward(sd, t, size // 32), x, kind))
    return time.perf_counter() - t0


def cpu_score_sample():
    """Reference scoring of ONE full 2848x4288 lesion map: sklearn average_precision_score (aucpr.py:24) + the 19
    threshold passes (aucpr.py:60-81) -> seconds."""
    import numpy as np
    from oracle import scoring
    rng = np.random.default_rng(0)
    prob = rng.random((H, W), dtype=np.float32)
    gt = (rng.random((H, W)) < 0.01).astype(np.uint8)
    t0 = time.perf_counter()
    scoring.get_auc([(prob, gt, "full")])
    scoring.threshold_counts(prob, gt)
    return time.perf_counter() - t0


def cpu_cfg1(threads):
    """BASELINE.md 3.1: config 1 in full -- smp.Unet(resnet34) fp32 on 1x3x512x512, best of 5 on the host cores."""
    import torch
    from oracle import nets
    import helpers
    torch.set_num_threads(threads)
    model = helpers.build_product_model("Unet", dict(encoder_name="resnet34", encoder_weights=None, classes=1))
    sd = model.state_dict()
    x = torch.randn(1, 3, 512, 512, generator=torch.Generator().manual_seed(0))
    best = 1e9
    with torch.no_grad():
        for _ in range(5):
            t0 = time.perf_counter()
            nets.unet_forward(sd, x)
            best = min(best, time.perf_counter() - t0)
    return best


def cpu_baseline():
    threads = os.cpu_count() or 1
    cpu_tile_sample(threads, views=1)                              # warm the allocator / thread pool
    t_tile = cpu_tile_sample(threads)
    t_score = cpu_score_sample()
    per_image = TILES * len(LESIONS) * t_tile + len(LESIONS) * t_score
    return {"value": 1.0 / per_image, "unit": "images/s", "cores": threads, "kind": "port",
            "sample": f"oracle (reference PyTorch path restated) on CPU fp32, RUN in full: one 1024^2 tile through all 8 "
                      f"D4 views + TTA mean + sigmoid ({t_tile:.1f} s) and the reference scoring of one full 2848x4288 "
                      f"map (sklearn AP + 19 threshold passes, {t_score:.1f} s); an image is 6 tiles x 4 lesion models "
                      f"= 24 such tiles + 4 such scorings (factor stated, not run); the reference additionally repeats "
                      f"inference 3x (tta.py:218,221,225), not counted",
            "tile_seconds": t_tile, "score_seconds": t_score,
            "cfg1_unet_r34_fp32_512_forward_s": cpu_cfg1(threads)}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (here the oracle port) on all host
    threads.  Each of the `steps` steps RUNS one whole tile (8 D4 views, TTA mean, sigmoid) and one full-image
    scoring; an image is 24 such tiles + 4 such scorings (stated in `config`).  Warm-up = `warmup` single
    forwards."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    for _ in range(args.warmup):
        cpu_tile_sample(threads, views=1, size=args.ref_size)
    tiles, scores = [], []
    for _ in range(args.steps):
        tiles.append(cpu_tile_sample(threads, views=args.ref_views, size=args.ref_size) * (VIEWS / args.ref_views))
        scores.append(cpu_score_sample())
    t_tile, t_score = sum(tiles) / len(tiles), sum(scores) / len(scores)
    sec = TILES * len(LESIONS) * t_tile + len(LESIONS) * t_score
    value = 1.0 / sec
    sample = (f"each step RUNS one 1024^2 tile (8 D4 views of the proposed net, TTA mean, sigmoid: {t_tile:.1f} s) + the "
              f"reference scoring of one full 2848x4288 map ({t_score:.1f} s) on {threads} host threads; images/s = "
              f"1 / (24 tiles + 4 scorings)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "images/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": len(tiles), "warmup": args.warmup,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": sample, "sample_seconds": t_tile + t_score,
                       "samples_per_step": {"tiles": TILES * len(LESIONS), "scorings": len(LESIONS)}},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tiles", type=int, default=6, help="tiles per forward batch (x8 views)")
    ap.add_argument("--group", type=int, default=0, help="images per unit-dealing group (0 = the whole set)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg-1 / cfg-2 / cfg-5 side measurements")
    ap.add_argument("--ref-size", type=int, default=S,
                    help="--impl reference: tile edge of the sampled forward (1024 = the workload; smaller only for "
                         "quick contract tests, the printed value is then not a measurement)")
    ap.add_argument("--ref-views", type=int, default=VIEWS, choices=[1, VIEWS],
                    help="--impl reference: TTA views per sampled tile (8 = the workload; 1 only for quick contract tests)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the probability maps (fixed sample) and scores of the last timed image to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
