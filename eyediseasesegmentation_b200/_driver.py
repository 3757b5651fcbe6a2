"""Shared core of the inference drivers (``tta.py`` / ``tta_vessel.py`` mirrors).

One pass per image does everything the reference's three generator passes redo
(src/main/tta.py:218,221,225): forward of all TTA views, merge, sigmoid, paste, and -- while
the probability map is still in HBM -- the PR/ROC histogram.  The yielded arrays carry their
scores (:class:`aucpr.ScoredArray`), so ``get_auc`` / ``plot_*`` / the mask writer reuse them.

Multi-GPU (SURVEY.md 8e): with ``torch.distributed`` initialised (torchrun, one process per
GPU) the image list is sharded ``images[rank::world_size]``; no activation crosses ranks.
The only exchange is the all-reduce of the pooled integer counts / AP sums in ``aucpr``.
"""
from __future__ import annotations

import logging
import os
import re
from pathlib import Path
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from . import archs, kernels as K, ttach_compat as tta
from .aucpr import ScoredArray, score_device
from .util import lesion_dict, make_grid

logging.basicConfig(level=logging.INFO)


class _Smp:
    """Stand-in for the ``segmentation_models_pytorch`` namespace probed by
    ``hasattr(smp, config['model_name'])`` (tta.py:62,155)."""
    Unet = staticmethod(archs.Unet)


smp = _Smp()


def get_model(params, model_name):
    """tta.py:40-46."""
    params["encoder_weights"] = None
    return getattr(smp, model_name)(**params)


def str_2_bool(value: str):
    if value.lower() in ["1", "true"]:
        return True
    elif value.lower() in ["0", "false"]:
        return False
    else:
        raise ValueError("Invalid value, should be one of these 1, true, 0, false")


def device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("the B200 inference drivers need a CUDA device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def ensure_distributed() -> None:
    """Under torchrun (WORLD_SIZE > 1 in the environment) make this process one rank of the NCCL group on its
    own GPU, unless the caller already did: the reference's ``pipeline.py`` knows nothing about ranks, so the
    drop-in drivers join the group themselves (``torchrun --nproc-per-node N pipeline.py ...`` just works)."""
    import torch.distributed as dist
    if int(os.environ.get("WORLD_SIZE", "1")) <= 1 or not dist.is_available():
        return
    if not torch.cuda.is_available():
        raise RuntimeError("the B200 inference drivers need a CUDA device; there is no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if dist.is_initialized():
        if dist.get_backend() == "nccl":
            torch.cuda.set_device(local)
        return
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))


def build_model(config, logdir, args):
    ensure_distributed()
    """Model dispatch + checkpoint load of tta.py:61-72,86-88 / 155-171."""
    if hasattr(smp, config["model_name"]):
        model = get_model(config["model_params"], config["model_name"])
    elif config["model_name"] == "TransUnet":
        raise NotImplementedError("TransUnet is outside the B200 hot path")
    else:
        model = archs.get_model(model_name=config["model_name"], params=config["model_params"], training=False)
    ckpt = load_checkpoint(f"{logdir}/checkpoints/{'best' if str_2_bool(args['best']) else 'last'}.pth")
    model.load_state_dict(ckpt["model_state_dict"])
    model = model.to(device())
    model.eval()
    return model


def load_checkpoint(path):
    """``torch.load`` of a reference checkpoint (tta.py:86,168).  catalyst checkpoints also carry optimizer /
    scheduler state and metric dicts with numpy scalars, which the ``weights_only=True`` default of torch >= 2.6
    refuses; the reference loads them unrestricted, so a checkpoint the restricted loader rejects is re-read the
    reference's way (checkpoints are the user's own training output)."""
    import pickle
    try:
        return torch.load(path, map_location="cpu", weights_only=True)
    except (pickle.UnpicklingError, RuntimeError, AttributeError) as e:
        logging.info(f"checkpoint {path} needs the unrestricted unpickler ({type(e).__name__}); loading with "
                     "weights_only=False")
        return torch.load(path, map_location="cpu", weights_only=False)


def tta_transforms(args):
    """tta.py:92-99: ``getattr(tta.aliases, args['tta'] + '_transform')``."""
    factory = getattr(tta.aliases, args["tta"] + "_transform")
    return factory(scales=[1, 2, 4]) if args["tta"] == "multiscale" else factory()


def shard(items: Sequence, what: str = "images") -> List:
    """This rank's slice of the work list (round-robin by index)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return list(items)[dist.get_rank()::dist.get_world_size()]
    return list(items)


def fused_blend_views(model, transforms, S: int, dst_w: int):
    """De-augment maps for the one-kernel blend (``eds_tta_blend_x2_f32``) when model, TTA alias, tile size and
    canvas width qualify, else None (the drivers then merge and paste with two kernels)."""
    if getattr(model, "forward_tta", None) is None or not tta.is_fusable(transforms):
        return None
    _, deaug = tta.view_maps(transforms, S, S)
    return deaug if K.tta_blend_supported(len(deaug), S, deaug, dst_w) else None


def predict_probs(model, transforms, x: torch.Tensor) -> torch.Tensor:
    """x [B,3,S,S] on the device -> probabilities [B,S,S] (sigmoid of the TTA-mean logits)."""
    fused = getattr(model, "forward_tta", None)
    if fused is not None and tta.is_fusable(transforms) and x.shape[2] == x.shape[3]:
        return fused(x, transforms, apply_sigmoid=True)[:, 0]
    wrapped = tta.SegmentationTTAWrapper(model, transforms, merge_mode="mean")
    return torch.sigmoid(wrapped(x))[:, 0].contiguous()


class CachedPredictions:
    """Re-iterable ``(pred, gt, name)`` source: the first iteration runs ``produce`` (inference
    + scoring) and keeps the results on the host; later iterations replay them.  This is what
    makes the reference's ``@multigen`` pattern cost one pass instead of three.

    Memory: the reference streams its three passes in O(1) memory; a cache of full-resolution fp32 maps is
    ~61 MB per IDRiD image and tens of GB on DDR / FGADR.  Up to ``EDS_CACHE_BYTES`` (default 8 GiB) stay in
    RAM; beyond that the arrays are spilled to ``np.memmap`` files in a temporary directory (the scores, which
    is all the first two consumers read, always stay in memory)."""

    def __init__(self, produce: Callable, budget_bytes: Optional[int] = None):
        self._produce = produce
        self._items: Optional[list] = None
        self._budget = int(os.environ.get("EDS_CACHE_BYTES", 8 << 30)) if budget_bytes is None else budget_bytes
        self._held = 0
        self._spill_dir = None

    def __iter__(self):
        if self._items is not None:
            return iter(self._items)
        return self._first_pass()

    def _spill(self, arr: np.ndarray, tag: str) -> np.ndarray:
        import tempfile
        if self._spill_dir is None:
            self._spill_dir = tempfile.TemporaryDirectory(prefix="eds_cache_")
        mm = np.lib.format.open_memmap(os.path.join(self._spill_dir.name, tag + ".npy"), mode="w+",
                                       dtype=arr.dtype, shape=arr.shape)
        mm[...] = arr
        mm.flush()
        return mm

    def _keep(self, item, index: int):
        pred, gt, name = item
        nbytes = getattr(pred, "nbytes", 0) + getattr(gt, "nbytes", 0)
        if self._held + nbytes <= self._budget:
            self._held += nbytes
            return item
        scores = getattr(pred, "_eds_scores", None)
        spilled = self._spill(np.asarray(pred), f"pred{index}")
        if scores is not None:
            spilled = ScoredArray(spilled, scores)
        return spilled, self._spill(np.asarray(gt), f"gt{index}"), name

    def _first_pass(self):
        items = []
        for item in self._produce():
            items.append(self._keep(item, len(items)))
            yield item
        self._items = items

    def __call__(self):   # ``predict_generator()`` call sites keep working
        return self


def read_rgb(path) -> np.ndarray:
    from PIL import Image
    return np.asarray(Image.open(path).convert("RGB")).astype("uint8")


def read_mask(path, threshold: int) -> np.ndarray:
    """PIL 'L' -> (x > threshold) -> {0,1} uint8 (tta.py:192-194 uses 0, the datasets use 50)."""
    from PIL import Image
    m = np.asarray(Image.open(path).convert("L"))
    return (m > threshold).astype(np.uint8)


def longest_max_size(img: np.ndarray, max_size: int, interpolation) -> np.ndarray:
    """albumentations 1.0 ``F.longest_max_size`` (3P): scale so the longest side == max_size."""
    import cv2
    h, w = img.shape[:2]
    scale = max_size / float(max(h, w))
    if scale == 1.0:
        return img
    new_h, new_w = int(round(h * scale)), int(round(w * scale))
    return cv2.resize(img, (new_w, new_h), interpolation=interpolation)


def pad_to_square(img: np.ndarray, size: int) -> np.ndarray:
    """albumentations ``PadIfNeeded(size, size, BORDER_CONSTANT, 0)`` (3P): centred zero pad."""
    h, w = img.shape[:2]
    top = int((size - h) / 2.0) if h < size else 0
    left = int((size - w) / 2.0) if w < size else 0
    out = np.zeros((max(size, h), max(size, w)) + img.shape[2:], dtype=img.dtype)
    out[top:top + h, left:left + w] = img
    return out


def tile_blend_mode(config=None) -> str:
    """"overwrite" (the reference's paste, tta.py:213: last writer wins -- default and parity mode) or "gaussian"
    (opt-in, no reference counterpart: Gaussian-weighted mean of the overlapping tiles); from
    ``config["tile_blend"]`` or the EDS_TILE_BLEND environment variable."""
    mode = (config or {}).get("tile_blend") or os.environ.get("EDS_TILE_BLEND", "overwrite")
    if mode not in ("overwrite", "gaussian"):
        raise ValueError(f"tile_blend must be 'overwrite' or 'gaussian', got {mode!r}")
    return mode


def tiled_probability_map(model, transforms, image_dev: torch.Tensor, S: int, mean, std,
                          tiles_per_batch: int = 6, blend: str = "overwrite") -> torch.Tensor:
    """Sliding-window inference of tta.py:196-213 on one decoded image (``[H,W,3]`` u8 on the
    device): window 2S, min_overlap 32, each window box-averaged to SxS, all TTA views, sigmoid,
    bilinear x2, overwrite-paste in ``make_grid`` order (last writer wins).  ``blend="gaussian"`` (opt-in, not
    the reference's behaviour) replaces the overwrite by a Gaussian-weighted mean of the overlapping tiles."""
    H, W = int(image_dev.shape[0]), int(image_dev.shape[1])
    slices = make_grid((H, W), window=2 * S, min_overlap=32)
    preds = torch.zeros((H, W), dtype=torch.float32, device=image_dev.device)
    if blend == "gaussian":
        wsum = torch.zeros_like(preds)
        window = K.gaussian_window(2 * S, device=image_dev.device)
    for (x1, x2, y1, y2) in slices:
        if x1 < 0 or y1 < 0 or x2 - x1 != 2 * S or y2 - y1 != 2 * S:
            raise ValueError(f"could not broadcast input array from shape ({2 * S},{2 * S}) into shape "
                             f"({max(x2 - max(x1, 0), 0)},{max(y2 - max(y1, 0), 0)}): window larger than the image")
    deaug = fused_blend_views(model, transforms, S, W) if blend == "overwrite" and len(slices) <= 32 else None
    origins = [(int(x1), int(y1)) for (x1, _, y1, _) in slices]
    for i in range(0, len(slices), tiles_per_batch):
        group = slices[i:i + tiles_per_batch]
        x = torch.empty((len(group), 3, S, S), dtype=torch.float32, device=image_dev.device)
        for j, (x1, _, y1, _) in enumerate(group):
            K.preprocess_tile(image_dev, int(x1), int(y1), S, mean, std, out=x[j])
        if deaug is not None:                         # views -> preds in one kernel, no [B,S,S] intermediate
            K.tta_blend_x2(model.forward_tta(x, transforms, merge=False), deaug, preds, origins, first_tile=i)
            continue
        prob = predict_probs(model, transforms, x)
        if blend == "gaussian":
            prob = prob.contiguous()
            for j, (x1, _, y1, _) in enumerate(group):
                K.blend_tile_gaussian_x2(prob[j], (int(x1), int(y1)), window, preds, wsum)
        elif len(group) <= 32 and W % 4 == 0:         # one launch, 128-bit stores (rows of preds 16-byte aligned)
            K.paste_tiles_x2(prob.contiguous(), preds, [(int(x1), int(y1)) for (x1, _, y1, _) in group])
        else:
            for j, (x1, _, y1, _) in enumerate(group):
                K.resize_paste(prob[j], preds, (0, 0, S, S), (int(x1), int(y1)), (2 * S, 2 * S))
    if blend == "gaussian":
        K.blend_finalize(preds, wsum, out=preds)
    return preds


# ------------------------------------------------------------------ (image, tile) partition (SURVEY.md 8e)
class TilePlan:
    """Static tile geometry of one image shape: paste origins in make_grid order and the rectangles each
    tile owns under last-writer-wins."""

    def __init__(self, H: int, W: int, S: int):
        from . import partition
        self.slices = make_grid((H, W), window=2 * S, min_overlap=32)
        for (x1, x2, y1, y2) in self.slices:
            if x1 < 0 or y1 < 0 or x2 - x1 != 2 * S or y2 - y1 != 2 * S:
                raise ValueError(f"could not broadcast input array from shape ({2 * S},{2 * S}) into shape "
                                 f"({max(x2 - max(x1, 0), 0)},{max(y2 - max(y1, 0), 0)}): window larger than the image")
        self.origins = [(int(x1), int(y1)) for (x1, _, y1, _) in self.slices]       # (row, column) of each window
        self.cells = partition.owned_cells([(x1, x2, y1, y2) for (x1, x2, y1, y2) in self.slices], (H, W))
        self.n = len(self.origins)


_PLANS = {}


def tile_plan(H: int, W: int, S: int) -> TilePlan:
    key = (int(H), int(W), int(S))
    if key not in _PLANS:
        _PLANS[key] = TilePlan(*key)
    return _PLANS[key]


def partitioned_group(model, transforms, images, gts, S: int, mean, std, hist: torch.Tensor, strad: torch.Tensor,
                      first_row: int, rank: int, world_size: int, tiles_per_batch: int = 6, unit_offset: int = 0):
    """This rank's share of the sliding-window inference of a GROUP of images (every rank holds the same
    decoded images ``[H,W,3]`` u8 and masks ``[H,Wp]`` u8 on its device, Wp = W rounded up to 4).

    Units ``(image, tile)`` are dealt round-robin (unit number = unit_offset + running index); the rank runs its
    tiles in batches, writes only the pixels they own into one zero-initialised canvas ``[H,Wp]`` per image and
    adds the histogram of those pixels to ``hist[first_row + k]`` / ``strad[first_row + k]``.  Returns
    (canvases, next unit_offset).  Summing canvases / histograms over ranks gives the single-process results."""
    from . import partition
    dev = images[0].device
    plans = [tile_plan(int(im.shape[0]), int(im.shape[1]), S) for im in images]
    units = [(k, t) for k, p in enumerate(plans) for t in range(p.n)]
    mine = [u for j, u in enumerate(units) if (unit_offset + j) % world_size == rank]
    canvases = [torch.zeros((int(im.shape[0]), int(g.shape[1])), dtype=torch.float32, device=dev)
                for im, g in zip(images, gts)]
    deaug = fused_blend_views(model, transforms, S, int(gts[0].shape[1])) if all(p.n <= 32 for p in plans) else None
    for batch in partition.batches(mine, tiles_per_batch):
        x = torch.empty((len(batch), 3, S, S), dtype=torch.float32, device=dev)
        for j, (k, t) in enumerate(batch):
            y0, x0 = plans[k].origins[t]
            K.preprocess_tile(images[k], y0, x0, S, mean, std, out=x[j])
        if deaug is not None:
            logits = model.forward_tta(x, transforms, merge=False)
            for j, (k, t) in enumerate(batch):
                K.tta_blend_x2(logits, deaug, canvases[k], plans[k].origins, first_tile=t, b0=j, n_src=1)
            continue
        prob = predict_probs(model, transforms, x).contiguous()
        for j, (k, t) in enumerate(batch):
            K.paste_tiles_owned_x2(prob[j:j + 1], t, canvases[k], plans[k].origins)
    for k, p in enumerate(plans):
        tiles_here = [t for (kk, t) in mine if kk == k]
        if len(tiles_here) == p.n and int(gts[k].shape[1]) == int(images[k].shape[1]):
            # this rank holds every tile of the image (one GPU, or more images than units): the streaming kernel
            K.pr_hist(canvases[k].view(1, -1), gts[k].view(1, -1), hist[first_row + k:first_row + k + 1],
                      strad[first_row + k:first_row + k + 1])
            continue
        rects = [r for t in tiles_here for r in p.cells[t]]
        if rects:
            K.pr_hist_rects(canvases[k], gts[k], rects, hist[first_row + k], strad[first_row + k])
    return canvases, unit_offset + len(units)


def partitioned_producer(model, transforms, keys, load, S: int, mean, std, tiles_per_batch: int = 6):
    """``produce()`` of the sliding-window drivers under torchrun (world size > 1).

    ``keys`` lists the images (same order on every rank), ``load(key) -> (image [H,W,3] u8, gt [H,W] u8)`` decodes
    one on the host.  Images are taken in groups of ``world_size``: rank r decodes the r-th image of the group
    (on a background thread, one group ahead) and broadcasts it; every rank then runs its ``(image, tile)``
    units of the group (``partitioned_group``); the canvases are summed onto the rank that decoded the image,
    which keeps the full-resolution map for the mask writer.  After the last group ONE all-reduce sums the
    per-image integer histograms, every rank scans them, and the generator yields, for every image, the global
    scores (``replicated=True``) with the map on its writer rank and an empty array elsewhere."""
    import torch.distributed as dist
    from . import partition
    from . import _lib
    from .aucpr import ImageScores

    def produce():
        rank, ws = partition.world()
        dev = device()
        n = len(keys)
        hist = torch.zeros((max(n, 1), 2, _lib.PR_BINS), dtype=torch.int32, device=dev)
        strad = torch.zeros((max(n, 1), _lib.PR_NTHRESH, 2), dtype=torch.int32, device=dev)
        kept = {}
        unit_offset = 0
        starts = list(range(0, n, ws))
        def guarded(g):
            # a decode error on one rank must reach every rank BEFORE the next collective, or the others hang in it
            try:
                return load(keys[g + rank]) if g + rank < n else None
            except Exception as e:                      # noqa: BLE001 -- re-raised on every rank below
                return e

        mine = prefetched([(lambda g=g: guarded(g)) for g in starts])
        for g, loaded in zip(starts, mine):
            group = list(range(g, min(g + ws, n)))
            shapes = [None] * ws
            failed = isinstance(loaded, Exception)
            dist.all_gather_object(shapes, ("error", f"rank {rank}: {loaded!r}") if failed else
                                   (None if loaded is None else tuple(loaded[0].shape[:2])))
            errors = [s_[1] for s_ in shapes if isinstance(s_, tuple) and s_ and s_[0] == "error"]
            if errors:
                raise RuntimeError("image loading failed: " + "; ".join(errors))
            images, gts = [], []
            for r, i in enumerate(group):
                H, W = shapes[r]
                img = torch.empty((H, W, 3), dtype=torch.uint8, device=dev)
                gt = torch.zeros((H, (W + 3) // 4 * 4), dtype=torch.uint8, device=dev)
                if r == rank:
                    img.copy_(torch.from_numpy(np.ascontiguousarray(loaded[0])))
                    gt[:, :W].copy_(torch.from_numpy(np.ascontiguousarray(loaded[1])))
                dist.broadcast(img, src=r)
                dist.broadcast(gt, src=r)
                images.append(img)
                gts.append(gt)
            canvases, unit_offset = partitioned_group(model, transforms, images, gts, S, mean, std, hist, strad, g,
                                                      rank, ws, tiles_per_batch, unit_offset)
            for r, i in enumerate(group):
                dist.reduce(canvases[r], dst=r, op=dist.ReduceOp.SUM)       # pieces -> the rank that wrote image i
                if r == rank:
                    W = shapes[r][1]
                    kept[i] = (canvases[r][:, :W].cpu().numpy(), loaded[1])
        partition.allreduce_sum_(hist, strad)                                # the path's one data collective
        if n:
            ap, roc, counts, totals = [t.cpu().numpy() for t in K.pr_scan(hist[:n], strad[:n])]
        for i in range(n):
            scores = ImageScores(float(ap[i]), float(roc[i]), counts[i, :, 0].copy(), counts[i, :, 1].copy(),
                                 int(totals[i, 0]), int(totals[i, 1]), replicated=True)
            name = getattr(keys[i], "name", str(keys[i]))
            if i in kept:
                yield ScoredArray(kept[i][0], scores), kept[i][1], name
            else:
                yield ScoredArray(np.zeros((0, 0), dtype=np.float32), scores), None, name

    return produce


def pad_width4(t: torch.Tensor) -> torch.Tensor:
    """[H,W] -> [H,Wp] with Wp = W rounded up to a multiple of 4 (zero columns): rows of the canvases and masks of
    the partitioned path start 16-byte aligned for the 128-bit paste stores."""
    H, W = t.shape
    if W % 4 == 0:
        return t
    out = torch.zeros((H, (W + 3) // 4 * 4), dtype=t.dtype, device=t.device)
    out[:, :W] = t
    return out


def prefetched(thunks, depth: int = 2):
    """Run ``thunk()`` for every element of ``thunks`` on ONE background thread, ``depth`` ahead of the consumer,
    and yield the results in order: JPEG decode (PIL releases the GIL) and pinned staging of image k+1 hide
    behind the GPU work of image k (SURVEY.md 8f-2; the reference decodes inside the loop, tta.py:196-203)."""
    import collections
    from concurrent.futures import ThreadPoolExecutor
    it = iter(thunks)
    with ThreadPoolExecutor(max_workers=1) as pool:
        q = collections.deque()
        for _ in range(max(1, depth)):
            t = next(it, None)
            if t is not None:
                q.append(pool.submit(t))
        while q:
            fut = q.popleft()
            t = next(it, None)
            if t is not None:
                q.append(pool.submit(t))
            yield fut.result()


_PINNED = {}


def _pinned(shape, dtype, tag="") -> torch.Tensor:
    """Reusable page-locked staging buffer (cudaHostAlloc is milliseconds; the copy engine needs
    pinned memory to run asynchronously at full PCIe rate)."""
    key = (tuple(shape), dtype, tag)
    buf = _PINNED.get(key)
    if buf is None:
        buf = torch.empty(tuple(shape), dtype=dtype).pin_memory()
        _PINNED[key] = buf
    return buf


def score_to_host(preds_dev: torch.Tensor, gt_dev: torch.Tensor, copy: bool = True, slot: str = ""):
    """Histogram + scan while the probability map is in HBM, then ONE synchronisation: the map and the
    packed scores travel device -> pinned host asynchronously on the current stream.
    Returns (probability map on the host [ScoredArray], ImageScores); with ``copy=False`` the array
    aliases the staging buffer of ``slot`` (valid until the next call with the same slot)."""
    from .aucpr import ImageScores
    hist, strad = K.pr_hist(preds_dev.reshape(1, -1), gt_dev.reshape(1, -1))
    ap, roc, counts, totals = K.pr_scan(hist, strad)
    h_pred = _pinned(preds_dev.shape, torch.float32, "pred" + slot)
    h_f = _pinned((2,), torch.float64, "apr" + slot)
    h_c = _pinned(counts.shape, torch.int64, "cnt" + slot)
    h_t = _pinned(totals.shape, torch.int64, "tot" + slot)
    h_pred.copy_(preds_dev, non_blocking=True)
    h_f[0:1].copy_(ap, non_blocking=True)
    h_f[1:2].copy_(roc, non_blocking=True)
    h_c.copy_(counts, non_blocking=True)
    h_t.copy_(totals, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    c = h_c.numpy()
    scores = ImageScores(float(h_f[0]), float(h_f[1]), c[0, :, 0].copy(), c[0, :, 1].copy(), int(h_t[0, 0]),
                         int(h_t[0, 1]))
    arr = h_pred.numpy()
    return ScoredArray(arr.copy() if copy else arr, scores), scores


def infer_image_host(model, transforms, image_host: torch.Tensor, gt_host: torch.Tensor, S: int, mean, std,
                     tiles_per_batch: int = 6, copy: bool = True, slot: str = "", blend: str = "overwrite"):
    """Host-facing unit of the sliding-window path (one iteration of tta.py:190-215 plus its scoring):
    decoded image ``[H,W,3]`` u8 and mask ``[H,W]`` u8 on the HOST (pinned memory makes the uploads
    asynchronous) -> (probability map on the host, ImageScores)."""
    dev = device()
    image = image_host.to(dev, non_blocking=True)
    gt = gt_host.to(dev, non_blocking=True)
    preds = tiled_probability_map(model, transforms, image, S, mean, std, tiles_per_batch, blend=blend)
    return score_to_host(preds, gt, copy=copy, slot=slot)


def scored(preds_dev: torch.Tensor, gt: np.ndarray) -> ScoredArray:
    gt_dev = torch.from_numpy(np.ascontiguousarray(gt)).to(preds_dev.device)
    return score_to_host(preds_dev, gt_dev)[0]


def output_dir(config, logdir) -> Path:
    out_path = Path(config["out_dir"]) / config["dataset_name"] / "tta" / config["lesion_type"] / Path(logdir).name
    if not os.path.isdir(out_path):
        os.makedirs(out_path, exist_ok=True)
    return out_path
