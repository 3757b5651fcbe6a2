"""Torch-tensor wrappers around the C ABI.

PyTorch is used for device memory and streams only; every operation here is one call
into ``libeds_b200.so``.  Activations are NHWC tensors ``[N, H, W, C]`` (bf16 or fp32).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import EDS_BF16, EDS_F32
from ._lib import check as _check

#: number of kernel launches issued through this module (every wrapper below is one launch)
LAUNCHES = [0]
#: when set to a list, conv2d(impl="tc") appends (algorithmic_flops, start_event, end_event)
CONV_TRACE = None
#: 3x3 s1 p1 convolutions with Cout <= 128 on maps at least this large take the halo-reuse kernel
HALO_MIN_HW = 64
#: 3x3 layers with Cout <= 64 run on the dw-grouped wide-N kernel (conv3x3_wide_sm100.cu) when the map is at
#: least WIDE_MIN_HW on its short side and the reduction has at least WIDE_MIN_CIN channels
WIDE_MIN_HW = 64
WIDE_MIN_CIN = 16


#: when set to a list, every launch appends (kernel class, CUDA event recorded right after it on the launching
#: stream): consecutive events give per-launch device times of an EAGER pass (bench.py: time shares per class)
KERNEL_TRACE = None
_TAG = [None]


def check(rc: int) -> None:
    LAUNCHES[0] += 1
    _check(rc)
    if KERNEL_TRACE is not None:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        KERNEL_TRACE.append((_TAG[0] or __import__("sys")._getframe(1).f_code.co_name, ev))
    _TAG[0] = None


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.bfloat16:
        return EDS_BF16
    if t.dtype == torch.float32:
        return EDS_F32
    raise TypeError(f"unsupported activation dtype {t.dtype}")


def _chk(*tensors: Optional[torch.Tensor]) -> None:
    cur = -1
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise ValueError("libeds_b200 kernels need CUDA tensors (there is no CPU path)")
        if not t.is_contiguous():
            raise ValueError("tensor must be contiguous")
        if cur < 0:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            # the launch goes to the CURRENT device's stream: a tensor of another GPU would be dereferenced there
            raise ValueError(f"tensor lives on cuda:{t.device.index} but the current device is cuda:{cur}; wrap the call "
                             "in `with torch.cuda.device(tensor.device):` (B200SegModel.forward does)")


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# ------------------------------------------------------------------ scoring
def pr_hist(prob: torch.Tensor, gt: torch.Tensor, hist: Optional[torch.Tensor] = None,
            straddle: Optional[torch.Tensor] = None, splits: int = 0):
    """prob [n_img, n_px] fp32, gt [n_img, n_px] u8 -> (hist [n_img,2,BINS] i32, straddle [n_img,19,2] i32)."""
    _chk(prob, gt)
    assert prob.dtype == torch.float32 and gt.dtype == torch.uint8 and prob.shape == gt.shape and prob.dim() == 2
    n_img, n_px = prob.shape
    if hist is None:
        hist = torch.zeros((n_img, 2, _lib.PR_BINS), dtype=torch.int32, device=prob.device)
    if straddle is None:
        straddle = torch.zeros((n_img, _lib.PR_NTHRESH, 2), dtype=torch.int32, device=prob.device)
    check(_lib.lib().eds_pr_hist_f32(_p(prob), _p(gt), n_px, n_img, _p(hist), _p(straddle), splits, _stream()))
    return hist, straddle


def pr_hist_rects(prob: torch.Tensor, gt: torch.Tensor, rects, hist: torch.Tensor, straddle: torch.Tensor) -> None:
    """prob [H,W] fp32, gt [H,W] u8, rects: [(y, x, h, w), ...] (<= 32) -> accumulates the histogram of those
    rectangles into hist [2,BINS] i32 / straddle [19,2] i32 of that image (one rank's owned pixels)."""
    _chk(prob, gt, hist, straddle)
    assert prob.dtype == torch.float32 and gt.dtype == torch.uint8 and prob.shape == gt.shape and prob.dim() == 2
    assert hist.shape == (2, _lib.PR_BINS) and straddle.shape == (_lib.PR_NTHRESH, 2)
    rects = [r for r in rects if r[2] > 0 and r[3] > 0]
    for i in range(0, len(rects), 32):
        part = rects[i:i + 32]
        flat = _lib.int_array([int(v) for r in part for v in r])
        check(_lib.lib().eds_pr_hist_rects_f32(_p(prob), _p(gt), prob.shape[0], prob.shape[1], len(part), flat,
                                               _p(hist), _p(straddle), _stream()))


def pr_scan(hist: torch.Tensor, straddle: torch.Tensor):
    """-> ap [n] f64, roc [n] f64, counts [n,19,2] i64 (tp, pp), totals [n,2] i64 (n_pos, n_neg)."""
    _chk(hist, straddle)
    n = hist.shape[0]
    dev = hist.device
    ap = torch.empty(n, dtype=torch.float64, device=dev)
    roc = torch.empty(n, dtype=torch.float64, device=dev)
    counts = torch.empty((n, _lib.PR_NTHRESH, 2), dtype=torch.int64, device=dev)
    totals = torch.empty((n, 2), dtype=torch.int64, device=dev)
    check(_lib.lib().eds_pr_scan(_p(hist), _p(straddle), n, _p(ap), _p(roc), _p(counts), _p(totals), _stream()))
    return ap, roc, counts, totals


def confusion_counts(pred: torch.Tensor, gt: torch.Tensor, thr_pred: int = 50, thr_gt: int = 50,
                     counts: Optional[torch.Tensor] = None) -> torch.Tensor:
    """pred, gt [n_img, n_px] u8 -> counts [n_img, 3] i64 = (true_p, actual_p, pred_p) of the masks
    binarised with ``x > thr`` (accumulates into ``counts`` when given)."""
    _chk(pred, gt, counts)
    assert pred.dtype == torch.uint8 and gt.dtype == torch.uint8 and pred.shape == gt.shape and pred.dim() == 2
    n_img, n_px = pred.shape
    if counts is None:
        counts = torch.zeros((n_img, 3), dtype=torch.int64, device=pred.device)
    check(_lib.lib().eds_confusion_u8(_p(pred), _p(gt), n_px, n_img, int(thr_pred), int(thr_gt), _p(counts), _stream()))
    return counts


# ------------------------------------------------------------- TTA and paste
def tta_merge(logits: torch.Tensor, deaug_maps: Sequence[Sequence[int]], apply_sigmoid: bool = True,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """logits [V,B,S,S] fp32 -> prob [B,S,S] fp32."""
    _chk(logits, out)
    V, B, S, S2 = logits.shape
    assert S == S2 and logits.dtype == torch.float32 and len(deaug_maps) == V
    if out is None:
        out = torch.empty((B, S, S), dtype=torch.float32, device=logits.device)
    flat = _lib.int_array([v for m in deaug_maps for v in m])
    check(_lib.lib().eds_tta_merge(_p(logits), V, B, S, flat, int(apply_sigmoid), _p(out), _stream()))
    return out


def resize_paste(src: torch.Tensor, dst: torch.Tensor, crop, dst_yx, out_hw) -> None:
    """Bilinear resize of src[crop] (y, x, h, w) to out_hw, written over dst at dst_yx."""
    _chk(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == torch.float32 and src.dim() == 2 and dst.dim() == 2
    cy, cx, ch, cw = crop
    check(_lib.lib().eds_resize_paste_f32(_p(src), src.shape[0], src.shape[1], cy, cx, ch, cw, _p(dst), dst.shape[0],
                                          dst.shape[1], dst_yx[0], dst_yx[1], out_hw[0], out_hw[1], _stream()))


def paste_tiles_x2(src: torch.Tensor, dst: torch.Tensor, origins) -> None:
    """src [B,S,S] fp32 tiles, each upsampled x2 (bilinear, cv2 arithmetic) and written over dst at
    origins[b] = (y, x), in index order with last-writer-wins -- one launch for the whole batch."""
    _chk(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == torch.float32 and src.dim() == 3 and dst.dim() == 2
    B, S, S2 = src.shape
    assert S == S2 and len(origins) == B
    ys = _lib.int_array([int(o[0]) for o in origins])
    xs = _lib.int_array([int(o[1]) for o in origins])
    check(_lib.lib().eds_paste_tiles_x2_f32(_p(src), B, S, ys, xs, _p(dst), dst.shape[0], dst.shape[1], _stream()))


def paste_tiles_owned_x2(src: torch.Tensor, first_tile: int, dst: torch.Tensor, origins) -> None:
    """src [n,S,S] = tiles first_tile .. first_tile+n-1 of the image whose FULL tile list (make_grid order) is
    ``origins``; writes only the pixels those tiles own (no later tile of the list covers them)."""
    _chk(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == torch.float32 and src.dim() == 3 and dst.dim() == 2
    n, S, S2 = src.shape
    assert S == S2 and 0 <= first_tile and first_tile + n <= len(origins)
    ys = _lib.int_array([int(o[0]) for o in origins])
    xs = _lib.int_array([int(o[1]) for o in origins])
    check(_lib.lib().eds_paste_tiles_owned_x2_f32(_p(src), n, first_tile, len(origins), S, ys, xs, _p(dst),
                                                  dst.shape[0], dst.shape[1], _stream()))


def tta_blend_supported(V: int, S: int, deaug_maps, dst_w: int) -> bool:
    flat = _lib.int_array([v for m in deaug_maps for v in m])
    return bool(_lib.load().eds_tta_blend_supported(int(V), int(S), flat, int(dst_w)))


def tta_blend_x2(logits: torch.Tensor, deaug_maps, dst: torch.Tensor, origins, first_tile: int = 0, b0: int = 0,
                 n_src: Optional[int] = None) -> None:
    """logits [V,Bt,S,S] fp32 -> de-augment + mean + sigmoid + bilinear x2 + overwrite-paste of tiles b0 .. b0+n_src-1
    of the batch (= tiles first_tile .. of the image's list ``origins``) into dst [H,W], one launch; only the
    pixels no later tile of the list covers are written (and only the blocks that own some are read)."""
    _chk(logits, dst)
    V, Bt, S, S2 = logits.shape
    assert S == S2 and logits.dtype == torch.float32 and dst.dtype == torch.float32 and dst.dim() == 2
    n_src = Bt - b0 if n_src is None else n_src
    flat = _lib.int_array([v for m in deaug_maps for v in m])
    ys = _lib.int_array([int(o[0]) for o in origins])
    xs = _lib.int_array([int(o[1]) for o in origins])
    check(_lib.lib().eds_tta_blend_x2_f32(_p(logits), V, Bt, b0, n_src, S, flat, first_tile, len(origins), ys, xs,
                                          _p(dst), dst.shape[0], dst.shape[1], _stream()))


def gaussian_window(S2: int, sigma_scale: float = 0.25, device=None) -> torch.Tensor:
    """Separable blend window of the opt-in Gaussian mode: g[t] = exp(-(t - c)^2 / (2 sigma^2)), c = (S2 - 1) / 2,
    sigma = sigma_scale * S2, evaluated in float64 and rounded once to float32."""
    import numpy as np
    t = np.arange(S2, dtype=np.float64)
    g = np.exp(-((t - (S2 - 1) / 2.0) ** 2) / (2.0 * (sigma_scale * S2) ** 2)).astype(np.float32)
    return torch.from_numpy(g).to(device) if device is not None else torch.from_numpy(g)


def blend_tile_gaussian_x2(src: torch.Tensor, origin, window: torch.Tensor, acc: torch.Tensor, wsum: torch.Tensor) -> None:
    """src [S,S] fp32: acc += w * up2x(src), wsum += w over the tile's window at origin (y, x); opt-in mode."""
    _chk(src, window, acc, wsum)
    S = src.shape[0]
    assert src.shape == (S, S) and window.shape == (2 * S,) and acc.shape == wsum.shape and acc.dim() == 2
    assert src.dtype == window.dtype == acc.dtype == wsum.dtype == torch.float32
    check(_lib.lib().eds_blend_tile_gaussian_x2_f32(_p(src), S, int(origin[0]), int(origin[1]), _p(window), _p(acc),
                                                    _p(wsum), acc.shape[0], acc.shape[1], _stream()))


def blend_finalize(acc: torch.Tensor, wsum: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(acc, wsum, out)
    if out is None:
        out = torch.empty_like(acc)
    check(_lib.lib().eds_blend_finalize_f32(_p(acc), _p(wsum), acc.numel(), _p(out), _stream()))
    return out


def preprocess_tile(img: torch.Tensor, y0: int, x0: int, S: int, mean, std,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """img [H,W,3] u8 -> normalised half-resolution window [3,S,S] fp32."""
    _chk(img, out)
    assert img.dtype == torch.uint8 and img.dim() == 3 and img.shape[2] == 3
    if out is None:
        out = torch.empty((3, S, S), dtype=torch.float32, device=img.device)
    m = (C.c_double * 3)(*[float(v) for v in mean])
    s = (C.c_double * 3)(*[float(v) for v in std])
    check(_lib.lib().eds_preprocess_tile_u8(_p(img), img.shape[0], img.shape[1], y0, x0, S, m, s, _p(out), _stream()))
    return out


# -------------------------------------------------------------- network ops
def stem_conv(x: torch.Tensor, aug_maps, w: torch.Tensor, bias: torch.Tensor, dtype: torch.dtype,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [B,3,H,W] fp32 NCHW -> [V*B, H/2, W/2, 64]."""
    _chk(x, w, bias, out)
    B, Cin, H, W = x.shape
    assert Cin == 3 and x.dtype == torch.float32 and w.shape == (7, 7, 3, 64) and w.dtype == torch.float32
    V = len(aug_maps)
    if out is None:
        out = torch.empty((V * B, H // 2, W // 2, 64), dtype=dtype, device=x.device)
    flat = _lib.int_array([v for m in aug_maps for v in m])
    check(_lib.lib().eds_stem_conv7x7s2(_p(x), B, H, W, V, flat, _p(w), _p(bias), _p(out), _dt(out), _stream()))
    return out


def stem_pack_weights(w: torch.Tensor) -> torch.Tensor:
    """w [7,7,3,64] fp32 -> packed bf16 operand of the tensor-core stem (once per model)."""
    _chk(w)
    assert w.shape == (7, 7, 3, 64) and w.dtype == torch.float32
    out = torch.empty(_lib.STEM_PACKED_ELEMS, dtype=torch.bfloat16, device=w.device)
    check(_lib.lib().eds_stem_pack_weights(_p(w), _p(out), _stream()))
    return out


def stem_conv_mma(x: torch.Tensor, aug_maps, w_packed: torch.Tensor, bias: torch.Tensor,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [B,3,H,W] fp32 NCHW -> [V*B, H/2, W/2, 64] bf16 on the tensor cores."""
    _chk(x, w_packed, bias, out)
    B, Cin, H, W = x.shape
    assert Cin == 3 and x.dtype == torch.float32 and w_packed.dtype == torch.bfloat16
    assert w_packed.numel() == _lib.STEM_PACKED_ELEMS
    V = len(aug_maps)
    if out is None:
        out = torch.empty((V * B, H // 2, W // 2, 64), dtype=torch.bfloat16, device=x.device)
    flat = _lib.int_array([v for m in aug_maps for v in m])
    check(_lib.lib().eds_stem_conv7x7s2_mma(_p(x), B, H, W, V, flat, _p(w_packed), _p(bias), _p(out), _stream()))
    return out


def conv_out_hw(H: int, W: int, R: int, stride: int, pad: int):
    return (H + 2 * pad - R) // stride + 1, (W + 2 * pad - R) // stride + 1


def pack_grouped_weights(w: torch.Tensor) -> torch.Tensor:
    """Grouped filter w [Cout,R,S,C/groups] (C == Cout, the channels per group dividing 64) -> the block-diagonal
    [Cout,R,S,64] operand of eds_conv2d_igemm_bf16_grouped: row co holds the 64 input channels of its 64-channel
    chunk, zero outside co's group.  Same dtype and device as w (pack in fp32, then cast)."""
    Cout, R, S, cpg = w.shape
    assert 64 % cpg == 0 and Cout % 64 == 0, (Cout, cpg)
    packed = torch.zeros((Cout, R, S, 64), dtype=w.dtype, device=w.device)
    off = (torch.arange(Cout, device=w.device) // cpg * cpg) % 64           # first channel of co's group in its chunk
    idx = (off.view(Cout, 1) + torch.arange(cpg, device=w.device).view(1, cpg)).view(Cout, 1, 1, cpg)
    packed.scatter_(3, idx.expand(Cout, R, S, cpg), w)
    return packed


def conv2d(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], stride: int = 1, pad: int = 0,
           relu: bool = False, residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
           impl: str = "auto", x1: Optional[torch.Tensor] = None, groups: int = 1) -> torch.Tensor:
    """x [N,H,W,C], w [Cout,R,S,C] (same dtype as x) -> [N,Ho,Wo,Cout].

    impl: "tc" = bf16 kernels picked by layer shape (the mma.sync kernel of conv3x3_small.cu for the 16-channel
    tail, else the tcgen05 generic, halo-reuse or dw-grouped wide-N implicit GEMM), "igemm" / "halo" / "wide" =
    force that tcgen05 kernel, "simt" = CUDA-core kernel, "auto" = tc for bf16 activations, simt for fp32 (the
    fp32 parity mode).

    groups > 1 (ResNeXt 3x3): always the grouped kernels, w [Cout,R,S,64] from pack_grouped_weights on the tensor
    cores, w [Cout,R,S,C/groups] on the CUDA cores.  A shape the grouped tcgen05 kernel does not take raises.
    """
    if groups > 1:
        return _conv2d_grouped(x, w, bias, groups, stride, pad, relu, residual, out, impl)
    _chk(x, w, bias, residual, out, x1)
    N, H, W_, Cin = x.shape
    Cout, R, S, Cw = w.shape
    C1 = 0
    if x1 is not None:          # convolution of cat([x, x1], channel) without building it (tensor-core kernels)
        assert x1.shape[:3] == x.shape[:3] and x1.dtype == x.dtype and stride == 1
        C1 = x1.shape[3]
    assert Cw == Cin + C1 and w.dtype == x.dtype
    Ho, Wo = conv_out_hw(H, W_, R, stride, pad)
    if out is None:
        out = torch.empty((N, Ho, Wo, Cout), dtype=x.dtype, device=x.device)
    if impl == "auto":
        impl = "tc" if x.dtype == torch.bfloat16 else "simt"
    if impl in ("tc", "igemm", "halo", "wide"):
        if x.dtype != torch.bfloat16:
            raise TypeError("the tcgen05 kernel takes bf16 activations")
        trace = CONV_TRACE
        if trace is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        # measured (48 maps): 16 -> 16 @1024^2 1.7 ms here vs 2.4 ms on the tcgen05 halo kernel; with 32 input
        # channels the legacy mma.sync pipe (~100 TFLOP/s in these kernels) loses to tcgen05 (32 -> 32 @512^2:
        # 2.2 ms vs 0.6 ms), so the small kernel takes only 16 input channels
        if (impl == "tc" and x1 is None and residual is None and R == 3 and S == 3 and stride == 1 and pad == 1 and
                _lib.load().eds_conv3x3_small_supported(Cin, Cout)):
            return conv3x3_small(x, w, bias, relu, out=out)
        # measured at 48 maps (scripts/dev_wide_probe.py, wide vs halo): 448 -> 64 @512^2 5.17 ms vs 6.02, 320 -> 32
        # 2.38 vs 4.31, 896 -> 64 @256^2 2.47 vs 2.92, 64 -> 64 @512^2 (weights resident) 1.33 vs 1.51, 32 -> 32 0.57
        # vs 0.67, 32 -> 16 @1024^2 1.00 vs 1.24
        wide = impl == "wide" or (impl == "tc" and min(H, W_) >= WIDE_MIN_HW and
                                  Cin + C1 >= WIDE_MIN_CIN and
                                  _lib.load().eds_conv3x3_wide_supported(Cin + C1, Cout, R, S, stride, pad))
        halo = not wide and (impl == "halo" or (impl == "tc" and min(H, W_) >= HALO_MIN_HW and
                                                _lib.load().eds_conv3x3_halo_supported(Cin + C1, Cout, R, S, stride, pad)))
        _TAG[0] = "conv3x3_wide (tcgen05)" if wide else "conv3x3_halo (tcgen05)" if halo else \
            f"conv_igemm {R}x{R} (tcgen05)"
        if wide:
            if x1 is not None:
                check(_lib.lib().eds_conv3x3_wide_bf16_2src(_p(x), Cin, _p(x1), C1, N, H, W_, _p(w), _p(bias), Cout,
                                                            int(relu), _p(residual), _p(out), _stream()))
            else:
                check(_lib.lib().eds_conv3x3_wide_bf16(_p(x), N, H, W_, Cin, _p(w), _p(bias), Cout, int(relu),
                                                       _p(residual), _p(out), _stream()))
        elif x1 is not None:
            if halo:
                check(_lib.lib().eds_conv3x3_halo_bf16_2src(_p(x), Cin, _p(x1), C1, N, H, W_, _p(w), _p(bias), Cout,
                                                            int(relu), _p(residual), _p(out), _stream()))
            else:
                check(_lib.lib().eds_conv2d_igemm_bf16_2src(_p(x), Cin, _p(x1), C1, N, H, W_, _p(w), _p(bias), Cout,
                                                            R, S, pad, int(relu), _p(residual), _p(out), _stream()))
        elif halo:
            check(_lib.lib().eds_conv3x3_halo_bf16(_p(x), N, H, W_, Cin, _p(w), _p(bias), Cout, int(relu),
                                                   _p(residual), _p(out), _stream()))
        else:
            check(_lib.lib().eds_conv2d_igemm_bf16(_p(x), N, H, W_, Cin, _p(w), _p(bias), Cout, R, S, stride, pad,
                                                   int(relu), _p(residual), _p(out), _stream()))
        if trace is not None:
            ev1.record()
            trace.append((2.0 * N * Ho * Wo * Cout * R * S * (Cin + C1), ev0, ev1,
                          (N, H, W_, Cin + C1, Cout, R, stride)))
    elif impl == "simt":
        if x1 is not None:
            raise ValueError("the CUDA-core kernel takes one input: concatenate first")
        check(_lib.lib().eds_conv2d_simt(_p(x), N, H, W_, Cin, _p(w), _p(bias), Cout, R, S, stride, pad, int(relu),
                                         _p(residual), _p(out), _dt(x), _stream()))
    else:
        raise ValueError(impl)
    return out


def _conv2d_grouped(x, w, bias, groups, stride, pad, relu, residual, out, impl):
    _chk(x, w, bias, residual, out)
    N, H, W_, Cin = x.shape
    Cout, R, S, Cw = w.shape
    assert w.dtype == x.dtype and Cin % groups == 0
    Ho, Wo = conv_out_hw(H, W_, R, stride, pad)
    if out is None:
        out = torch.empty((N, Ho, Wo, Cout), dtype=x.dtype, device=x.device)
    if impl == "auto":
        impl = "tc" if x.dtype == torch.bfloat16 else "simt"
    if impl == "tc":
        if x.dtype != torch.bfloat16:
            raise TypeError("the tcgen05 kernel takes bf16 activations")
        if not _lib.load().eds_conv2d_igemm_grouped_supported(Cin, Cout, groups, R, S, stride):
            raise ValueError(f"grouped convolution C={Cin} Cout={Cout} groups={groups} {R}x{S} stride {stride} is not "
                             "supported by the tcgen05 kernel (C == Cout, C % 64 == 0, C / groups dividing 64)")
        assert Cw == 64, "tensor-core grouped weights are the packed [Cout,R,S,64] operand (pack_grouped_weights)"
        trace = CONV_TRACE
        if trace is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        _TAG[0] = f"conv_igemm {R}x{R} grouped (tcgen05)"
        check(_lib.lib().eds_conv2d_igemm_bf16_grouped(_p(x), N, H, W_, Cin, _p(w), _p(bias), groups, Cout, R, S,
                                                       stride, pad, int(relu), _p(residual), _p(out), _stream()))
        if trace is not None:
            ev1.record()
            trace.append((2.0 * N * Ho * Wo * Cout * R * S * (Cin // groups), ev0, ev1,
                          (N, H, W_, Cin, Cout, R, stride, groups)))
    elif impl == "simt":
        assert Cw == Cin // groups
        check(_lib.lib().eds_conv2d_simt_grouped(_p(x), N, H, W_, Cin, _p(w), _p(bias), groups, Cout, R, S, stride,
                                                 pad, int(relu), _p(residual), _p(out), _dt(x), _stream()))
    else:
        raise ValueError(f"grouped convolutions run on the grouped tcgen05 or CUDA-core kernel, not {impl!r}")
    return out


def conv1x1_se(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], gate: torch.Tensor,
               residual: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """SE bottleneck tail in the convolution's epilogue: relu((conv1x1(x) + bias) * gate[n, co] + residual), bf16 on
    the tcgen05 kernel.  x [N,H,W,C], w [Cout,1,1,C], gate [N,Cout] fp32, residual [N,H,W,Cout]."""
    _chk(x, w, bias, gate, residual, out)
    N, H, W_, Cin = x.shape
    Cout = w.shape[0]
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and w.shape == (Cout, 1, 1, Cin)
    assert gate.shape == (N, Cout) and gate.dtype == torch.float32 and residual.shape == (N, H, W_, Cout)
    if out is None:
        out = torch.empty((N, H, W_, Cout), dtype=x.dtype, device=x.device)
    trace = CONV_TRACE
    if trace is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    _TAG[0] = "conv_igemm 1x1 (tcgen05)"
    check(_lib.lib().eds_conv2d_igemm_bf16_gated(_p(x), N, H, W_, Cin, _p(w), _p(bias), _p(gate), Cout, 1, 1, 1, 0, 1,
                                                 _p(residual), _p(out), _stream()))
    if trace is not None:
        ev1.record()
        trace.append((2.0 * N * H * W_ * Cout * Cin, ev0, ev1, (N, H, W_, Cin, Cout, 1, 1)))
    return out


def affine_rows(m: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], out: Optional[torch.Tensor] = None):
    """m [N,Cin] fp32, w [Cout,Cin] fp32 -> [N,Cout] = m @ w.T + b."""
    _chk(m, w, b, out)
    N, Cin = m.shape
    Cout = w.shape[0]
    assert w.shape == (Cout, Cin) and m.dtype == torch.float32 and w.dtype == torch.float32
    if out is None:
        out = torch.empty((N, Cout), dtype=torch.float32, device=m.device)
    check(_lib.lib().eds_affine_rows(_p(m), N, Cin, _p(w), _p(b), Cout, _p(out), _stream()))
    return out


def conv3x3_small(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], relu: bool = True,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Decoder-tail 3x3 s1 p1 convolution on mma.sync: x [N,H,W,16] bf16, w [Cout,3,3,16] with Cout in {16, 32}
    -> [N, H, W, Cout]."""
    _chk(x, w, bias, out)
    N, H, W_, Cin = x.shape
    Cout = w.shape[0]
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and w.shape == (Cout, 3, 3, Cin)
    if out is None:
        out = torch.empty((N, H, W_, Cout), dtype=x.dtype, device=x.device)
    trace = CONV_TRACE
    if trace is not None:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    _TAG[0] = "conv3x3_small (mma.sync)"
    check(_lib.lib().eds_conv3x3_small_bf16(_p(x), N, H, W_, Cin, _p(w), _p(bias), Cout, int(relu), _p(out),
                                            _stream()))
    if trace is not None:
        ev1.record()
        trace.append((2.0 * N * H * W_ * Cout * 9 * Cin, ev0, ev1, (N, H, W_, Cin, Cout, 3, 1)))
    return out


def head_conv3x3(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor],
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [N,H,W,C], w [classes,3,3,C] fp32 -> logits [N,classes,H,W] fp32."""
    _chk(x, w, bias, out)
    N, H, W_, Cin = x.shape
    classes = w.shape[0]
    assert w.dtype == torch.float32 and w.shape[1:] == (3, 3, Cin)
    if out is None:
        out = torch.empty((N, classes, H, W_), dtype=torch.float32, device=x.device)
    check(_lib.lib().eds_head_conv3x3(_p(x), N, H, W_, Cin, _p(w), _p(bias), classes, _p(out), _dt(x), _stream()))
    return out


def pool_out(size: int, k: int, stride: int, pad: int, ceil_mode: bool) -> int:
    num = size + 2 * pad - k
    o = (-(-num // stride) if ceil_mode else num // stride) + 1
    if ceil_mode and (o - 1) * stride >= size + pad:
        o -= 1
    return o


def maxpool2d(x: torch.Tensor, k: int, stride: int, pad: int = 0, ceil_mode: bool = False,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(x, out)
    N, H, W_, Cc = x.shape
    Ho, Wo = pool_out(H, k, stride, pad, ceil_mode), pool_out(W_, k, stride, pad, ceil_mode)
    if out is None:
        out = torch.empty((N, Ho, Wo, Cc), dtype=x.dtype, device=x.device)
    check(_lib.lib().eds_maxpool2d(_p(x), N, H, W_, Cc, k, stride, pad, int(ceil_mode), _p(out), _dt(x), _stream()))
    return out


def avgpool2_affine(x: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, relu: bool,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(x, scale, shift, out)
    N, H, W_, Cc = x.shape
    if out is None:
        out = torch.empty((N, H // 2, W_ // 2, Cc), dtype=x.dtype, device=x.device)
    check(_lib.lib().eds_avgpool2_affine(_p(x), N, H, W_, Cc, _p(scale), _p(shift), int(relu), _p(out), _dt(x),
                                         _stream()))
    return out


def channel_mean(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(x, out)
    N, H, W_, Cc = x.shape
    if out is None:
        out = torch.empty((N, Cc), dtype=torch.float32, device=x.device)
    check(_lib.lib().eds_channel_mean(_p(x), N, H * W_, Cc, _p(out), _dt(x), _stream()))
    return out


def se_gate(mean: torch.Tensor, w1, b1, w2, b2, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(mean, w1, b1, w2, b2, out)
    N, Cc = mean.shape
    Cr = w1.shape[0]
    assert w1.shape == (Cr, Cc) and w2.shape == (Cc, Cr)
    if out is None:
        out = torch.empty((N, Cc), dtype=torch.float32, device=mean.device)
    check(_lib.lib().eds_se_gate(_p(mean), N, Cc, Cr, _p(w1), _p(b1), _p(w2), _p(b2), _p(out), _stream()))
    return out


def se_scale_add_relu(x: torch.Tensor, gate: torch.Tensor, residual: torch.Tensor,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(x, gate, residual, out)
    N, H, W_, Cc = x.shape
    if out is None:
        out = torch.empty_like(x)
    check(_lib.lib().eds_se_scale_add_relu(_p(x), _p(gate), _p(residual), N, H * W_, Cc, _p(out), _dt(x), _stream()))
    return out


def upsample2x_concat(x0: torch.Tensor, skips: Sequence[torch.Tensor], mode: int,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(x0, out, *skips)
    N, h, w, C0 = x0.shape
    ctot = C0 + sum(s.shape[3] for s in skips)
    up = 1 if mode == _lib.UP_NONE else 2
    for s in skips:
        assert s.shape[:3] == (N, up * h, up * w) and s.dtype == x0.dtype
    if out is None:
        out = torch.empty((N, up * h, up * w, ctot), dtype=x0.dtype, device=x0.device)
    n = len(skips)
    ptrs = (C.c_void_p * max(n, 1))(*[s.data_ptr() for s in skips])
    chans = (C.c_int * max(n, 1))(*[s.shape[3] for s in skips])
    check(_lib.lib().eds_upsample2x_concat(_p(x0), N, h, w, C0, mode, ptrs, chans, n, _p(out), _dt(x0), _stream()))
    return out


def gated_stats(x: torch.Tensor, cgate: Optional[torch.Tensor], sgate: Optional[torch.Tensor],
                w_sse: Optional[torch.Tensor], mean: torch.Tensor, c_off: int = 0, zero_mean: bool = False,
                dot: Optional[torch.Tensor] = None, accumulate: bool = False) -> None:
    """Pass A over one (possibly gated) source [N,h,w,C]: mean[:, c_off:c_off+C] += channel means of the
    gated values; dot [N,h,w] (+)= per-pixel dot with w_sse (this source's slice, contiguous)."""
    _chk(x, cgate, sgate, w_sse, mean, dot)
    N, h, w, Cc = x.shape
    assert mean.dtype == torch.float32 and mean.shape[0] == N
    if w_sse is not None:
        assert w_sse.numel() == Cc and w_sse.dtype == torch.float32
    if dot is not None:
        assert dot.shape == (N, h, w) and dot.dtype == torch.float32
    check(_lib.lib().eds_gated_stats(_p(x), _p(cgate), _p(sgate), N, h * w, Cc, _p(w_sse), _p(mean), mean.shape[1],
                                     c_off, int(zero_mean), _p(dot), int(accumulate), _dt(x), _stream()))


def gated_stats_multi(x: torch.Tensor, cgate: Optional[torch.Tensor], sgate: Optional[torch.Tensor], consumers) -> None:
    """One read of a same-resolution skip source [N,h,w,C] for ALL its consumers: ``consumers`` is a list (<= 4) of
    ``(w_sse slice [C] fp32, mean [N,stride] fp32, c_off, dot [N,h,w] fp32)``; the (gated) channel means are ADDED
    into ``mean[:, c_off:c_off+C]`` and the per-pixel dots ADDED into ``dot`` (the caller zeroes both once)."""
    _chk(x, cgate, sgate)
    N, h, w, Cc = x.shape
    n = len(consumers)
    assert 1 <= n <= 4
    for (ws, mean, off, dot) in consumers:
        _chk(ws, mean, dot)
        assert ws.numel() == Cc and ws.dtype == torch.float32 and mean.dtype == torch.float32 and mean.shape[0] == N
        assert dot.shape == (N, h, w) and dot.dtype == torch.float32
    ws = (C.c_void_p * n)(*[c[0].data_ptr() for c in consumers])
    means = (C.c_void_p * n)(*[c[1].data_ptr() for c in consumers])
    strides = (C.c_int * n)(*[c[1].shape[1] for c in consumers])
    offs = (C.c_int * n)(*[int(c[2]) for c in consumers])
    dots = (C.c_void_p * n)(*[c[3].data_ptr() for c in consumers])
    check(_lib.lib().eds_gated_stats_multi(_p(x), _p(cgate), _p(sgate), N, h * w, Cc, n, ws, means, strides, offs, dots,
                                           _dt(x), _stream()))


def sse_finalize(dot0: Optional[torch.Tensor], dot1: Optional[torch.Tensor], mode: int, b_sse: float,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """sigmoid(up(dot0) + dot1 + b) -> [N,H,W] fp32 (in place over dot1 by default)."""
    _chk(dot0, dot1, out)
    up = 1 if mode == _lib.UP_NONE else 2
    if dot0 is not None:
        N, h, w = dot0.shape
    else:
        N, H, W_ = dot1.shape
        h, w = H // up, W_ // up
    if out is None:
        out = dot1 if dot1 is not None else torch.empty((N, up * h, up * w), dtype=torch.float32, device=dot0.device)
    assert out.shape == (N, up * h, up * w)
    check(_lib.lib().eds_sse_finalize(_p(dot0), _p(dot1), N, h, w, mode, float(b_sse), _p(out), _stream()))
    return out


def concat_gated_split(srcs, mode: int, cgate: Optional[torch.Tensor] = None, sgate: Optional[torch.Tensor] = None):
    """Like concat_gated but into TWO dense maps: (up2x(src 0) [N,2h,2w,C0], cat(src 1..) [N,2h,2w,sum Ck]),
    each gated with its channel slice of cgate; the pair feeds conv2d(x, ..., x1=...)."""
    x0 = srcs[0][0]
    N, h, w, C0 = x0.shape
    assert len(srcs) >= 2
    c_skip = sum(t[0].shape[3] for t in srcs[1:])
    arr = (_lib.GatedSrc * len(srcs))()
    for k, (x, cg, sg) in enumerate(srcs):
        _chk(x, cg, sg)
        assert x.dtype == x0.dtype and x.shape[:3] == ((N, h, w) if k == 0 else (N, 2 * h, 2 * w))
        arr[k].x, arr[k].cgate, arr[k].sgate, arr[k].C = _p(x), _p(cg), _p(sg), x.shape[3]
    _chk(cgate, sgate)
    y_up = torch.empty((N, 2 * h, 2 * w, C0), dtype=x0.dtype, device=x0.device)
    y_skip = torch.empty((N, 2 * h, 2 * w, c_skip), dtype=x0.dtype, device=x0.device)
    check(_lib.lib().eds_concat_gated_split(arr, len(srcs), N, h, w, mode, _p(cgate), _p(sgate), _p(y_up), _p(y_skip),
                                            _dt(x0), _stream()))
    LAUNCHES[0] += 1            # two kernels
    return y_up, y_skip


def concat_gated(srcs, mode: int, cgate: Optional[torch.Tensor] = None, sgate: Optional[torch.Tensor] = None,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """srcs: [(x, cgate or None, sgate or None), ...]; source 0 [N,h,w,C0] is upsampled x2, the others are
    [N,2h,2w,Ck].  -> cat(...) * (cgate[n,c] + sgate[n,p]) as one write."""
    x0 = srcs[0][0]
    N, h, w, _ = x0.shape
    ctot = sum(t[0].shape[3] for t in srcs)
    arr = (_lib.GatedSrc * len(srcs))()
    for k, (x, cg, sg) in enumerate(srcs):
        _chk(x, cg, sg)
        assert x.dtype == x0.dtype and x.shape[:3] == ((N, h, w) if k == 0 else (N, 2 * h, 2 * w))
        arr[k].x, arr[k].cgate, arr[k].sgate, arr[k].C = _p(x), _p(cg), _p(sg), x.shape[3]
    _chk(cgate, sgate, out)
    if out is None:
        out = torch.empty((N, 2 * h, 2 * w, ctot), dtype=x0.dtype, device=x0.device)
    check(_lib.lib().eds_concat_gated(arr, len(srcs), N, h, w, mode, _p(cgate), _p(sgate), _p(out), _dt(x0),
                                      _stream()))
    return out


def apply_gate(x: torch.Tensor, cgate: torch.Tensor, sgate: torch.Tensor, out: Optional[torch.Tensor] = None):
    _chk(x, cgate, sgate, out)
    N, H, W_, Cc = x.shape
    if out is None:
        out = torch.empty_like(x)
    check(_lib.lib().eds_apply_gate(_p(x), _p(cgate), _p(sgate), N, H * W_, Cc, _p(out), _dt(x), _stream()))
    return out


def axial_attention(qk: torch.Tensor, v: Optional[torch.Tensor], axis: int, heads: int, dqk: int, dv: int,
                    rel: torch.Tensor, sim_scale: torch.Tensor, out_scale: torch.Tensor, out_shift: torch.Tensor,
                    relu: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(qk, v, rel, sim_scale, out_scale, out_shift, out)
    N, H, W_, Cq = qk.shape
    L = H if axis == 0 else W_
    assert rel.shape == (2 * dqk + dv, 2 * L - 1) and rel.dtype == torch.float32
    assert Cq == heads * (2 * dqk + (0 if v is not None else dv))
    if v is not None:
        assert v.shape == (N, H, W_, heads * dv) and v.dtype == qk.dtype
    if out is None:
        out = torch.empty((N, H, W_, heads * dv), dtype=qk.dtype, device=qk.device)
    check(_lib.lib().eds_axial_attention(_p(qk), Cq, _p(v), heads * dv, N, H, W_, axis, heads, dqk, dv, _p(rel),
                                         _p(sim_scale), _p(out_scale), _p(out_shift), int(relu), _p(out), _dt(qk),
                                         _stream()))
    return out


def mhca_gate(ori: torch.Tensor, att: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _chk(ori, att, out)
    N, h, w, Cc = att.shape
    assert ori.shape == (N, 2 * h, 2 * w, Cc)
    if out is None:
        out = torch.empty_like(ori)
    check(_lib.lib().eds_mhca_gate(_p(ori), _p(att), N, h, w, Cc, _p(out), _dt(ori), _stream()))
    return out
