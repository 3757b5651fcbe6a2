import sys, os, math
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from eyediseasesegmentation_b200 import kernels as K
def timeit(fn, n=4, warm=2):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n): fn()
    e.record(); torch.cuda.synchronize()
    return s.elapsed_time(e) / n
N = 48
for (H, C, Cout, R) in [(256, 64, 256, 1), (128, 128, 512, 1), (64, 256, 1024, 1), (256, 256, 64, 1), (128, 512, 128, 1), (128, 256, 512, 1)]:
    x = torch.randn(N, H, H, C, device='cuda').bfloat16()
    w = (torch.randn(Cout, R, R, C, device='cuda') / math.sqrt(R*R*C)).bfloat16()
    b = torch.zeros(Cout, device='cuda')
    y = torch.empty(N, H, H, Cout, device='cuda', dtype=torch.bfloat16)
    ms = timeit(lambda: K.conv2d(x, w, b, 1, R // 2, True, None, out=y, impl='tc'))
    by = (x.numel() + y.numel()) * 2
    print(f"N{N} {H} C{C}->{Cout} k{R}: {ms:.3f} ms {by/ms/1e6:.0f} GB/s", flush=True)
    del x, w, y
