"""Residual 1x1 convolutions of the encoder at 48 maps (dev tool): the SE bottleneck tails (conv3 plain, with a
residual, with gate + residual in its epilogue, and as conv3 + se_scale_add_relu) and the axial block's `out`
projection with its residual.  CUDA-event times, the bytes each variant must move (bf16 maps; gate and weights
are negligible) and the rate that makes.  Outputs and residuals are larger than the 126 MB L2; the inputs of
layer3 (100 MB) and of the axial projection (6 MB) fit in it."""
import os, sys, math, subprocess
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from eyediseasesegmentation_b200 import kernels as K
N = 48


def timeit(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def row(what, ms, nbytes):
    print(f"  {what:<34s} {ms:7.3f} ms  {nbytes / 1e9:6.3f} GB  {nbytes / ms / 1e6:6.0f} GB/s", flush=True)


print(f"card: {card()}  (N = {N} maps, bf16)")
for name, H, Cin, Cout in [("layer1 conv3", 256, 64, 256), ("layer2 conv3", 128, 128, 512),
                           ("layer3 conv3", 64, 256, 1024), ("axial out", 32, 64, 2048)]:
    x = torch.randn(N, H, H, Cin, device="cuda").bfloat16()
    w = (torch.randn(Cout, 1, 1, Cin, device="cuda") / math.sqrt(Cin)).bfloat16()
    b = torch.zeros(Cout, device="cuda")
    res = torch.randn(N, H, H, Cout, device="cuda").bfloat16()
    gate = torch.rand(N, Cout, device="cuda")
    y = torch.empty(N, H, H, Cout, device="cuda", dtype=torch.bfloat16)
    bx, by = x.numel() * 2, y.numel() * 2
    print(f"{name}: {N} x {H}^2 x {Cin} -> {Cout}")
    t_plain = timeit(lambda: K.conv2d(x, w, b, 1, 0, False, None, out=y, impl="tc"))
    row("plain", t_plain, bx + by)
    row("+ residual + ReLU", timeit(lambda: K.conv2d(x, w, b, 1, 0, True, res, out=y, impl="tc")), bx + 2 * by)
    if name.startswith("axial"):
        continue
    row("fused (gate + residual + ReLU)", timeit(lambda: K.conv1x1_se(x, w, b, gate, res, out=y)), bx + 2 * by)
    t_scale = timeit(lambda: K.se_scale_add_relu(y, gate, res, out=y))
    row("se_scale_add_relu alone", t_scale, 3 * by)
    row("unfused (conv3 + se_scale_add_relu)", t_plain + t_scale, bx + 4 * by)
    del x, w, res, y
    torch.cuda.empty_cache()
