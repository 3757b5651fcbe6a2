"""Time the decoder concat (both parts, split destination) on the benchmark's layer shapes (dev tool)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from eyediseasesegmentation_b200 import kernels as K, _lib
N = 48
# name, low-res h, C0, x gated?, skips [(C, gated)]
layers = [("x_1_3", 256, 256, True, [(64, True), (64, True), (64, False)]),
          ("x_0_3", 256, 64, True, [(64, True), (64, True), (64, True), (64, False)]),
          ("x_2_3", 256, 256, True, [(64, True), (64, False)]),
          ("x_3_3", 256, 256, False, [(64, False)]),
          ("x_1_2", 128, 512, False, [(256, True), (256, False)]),
          ("x_0_2", 128, 128, False, [(256, True), (256, True), (256, False)]),
          ("x_2_2", 128, 512, False, [(256, False)])]
tot = 0.0
for name, h, C0, xg, skips in layers:
    def src(n, hh, C, gated):
        x = torch.randn(n, hh, hh, C, device="cuda").bfloat16()
        return (x, torch.rand(n, C, device="cuda"), torch.rand(n, hh, hh, device="cuda")) if gated else (x, None, None)
    srcs = [src(N, h, C0, xg)] + [src(N, 2 * h, C, g) for C, g in skips]
    Ctot = C0 + sum(C for C, _ in skips)
    cg1 = torch.rand(N, Ctot, device="cuda")
    sg1 = torch.rand(N, 2 * h, 2 * h, device="cuda")
    fn = lambda: K.concat_gated_split(srcs, _lib.UP_BILINEAR, cg1, sg1)
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(4):
        fn()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 4
    tot += ms
    out_b = N * (2 * h) ** 2 * Ctot * 2
    in_b = N * h * h * C0 * 2 + N * (2 * h) ** 2 * sum(C for C, _ in skips) * 2
    print(f"{name}: {ms:.3f} ms  ({(in_b + out_b) / ms / 1e6:.0f} GB/s read+write)", flush=True)
    del srcs, cg1, sg1
print(f"total {tot:.3f} ms")
