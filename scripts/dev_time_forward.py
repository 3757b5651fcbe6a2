"""Developer timing probe (not the benchmark): per-layer conv timings and a whole forward."""
import sys, os, time, math
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from eyediseasesegmentation_b200 import archs, kernels as K, ttach_compat as tta

def timeit(fn, n=5, warm=2):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n): fn()
    e.record(); torch.cuda.synchronize()
    return s.elapsed_time(e) / n

convs = [  # N,H,W,C,Cout,R  (decoder hot layers at 1024^2, 8 views)
    (8, 256, 256, 1024, 256, 3), (8, 128, 128, 1536, 512, 3), (8, 256, 256, 768, 256, 3), (8, 256, 256, 256, 256, 3),
    (8, 512, 512, 448, 64, 3), (8, 512, 512, 64, 64, 3), (8, 1024, 1024, 32, 16, 3), (8, 64, 64, 3072, 256, 3),
    (8, 64, 64, 1024, 512, 1), (8, 32, 32, 512, 2048, 1),
]
halo = [(8, 512, 512, 448, 64), (8, 512, 512, 320, 32), (8, 512, 512, 64, 64), (8, 1024, 1024, 32, 16),
        (8, 1024, 1024, 16, 16), (8, 256, 256, 896, 64), (8, 128, 128, 128, 128), (8, 256, 256, 64, 64)]
for (N, H, W, C, Cout) in halo:
    x = torch.randn(N, H, W, C, device='cuda').bfloat16()
    w = (torch.randn(Cout, 3, 3, C, device='cuda') / math.sqrt(9*C)).bfloat16()
    b = torch.zeros(Cout, device='cuda')
    y = torch.empty(N, H, W, Cout, device='cuda', dtype=torch.bfloat16)
    fl = 2.0 * N * H * W * C * Cout * 9
    ms0 = timeit(lambda: K.conv2d(x, w, b, 1, 1, True, None, out=y, impl='igemm'))
    ms1 = timeit(lambda: K.conv2d(x, w, b, 1, 1, True, None, out=y, impl='halo'))
    print(f"halo N{N} {H}x{W} C{C}->{Cout}: generic {ms0:.3f} ms {fl/ms0/1e9:.0f} TF | halo {ms1:.3f} ms {fl/ms1/1e9:.0f} TF", flush=True)
    del x, w, y
for (N, H, W, C, Cout, R) in convs:
    x = torch.randn(N, H, W, C, device='cuda').bfloat16()
    w = (torch.randn(Cout, R, R, C, device='cuda') / math.sqrt(R*R*C)).bfloat16()
    b = torch.zeros(Cout, device='cuda')
    y = torch.empty(N, H, W, Cout, device='cuda', dtype=torch.bfloat16)
    ms = timeit(lambda: K.conv2d(x, w, b, 1, R // 2, True, None, out=y, impl='tc'))
    fl = 2.0 * N * H * W * C * Cout * R * R
    print(f"conv N{N} {H}x{W} C{C}->{Cout} k{R}: {ms:.3f} ms  {fl/ms/1e9:.1f} TFLOP/s", flush=True)
    del x, w, y

cfg = dict(classes=1, decoder_attention_type="scse", decoder_use_batchnorm=True, base_dim=32, encoder_depth=5,
           encoder_name="BoTSER50_Axial_scratch", deep_supervision=False, drop_block_prob=0.0, clf_head=False)
torch.manual_seed(0)
model = archs.get_model("unetplusplusstar", cfg, training=False).to('cuda').eval()
x = torch.randn(1, 3, 1024, 1024, device='cuda')
t = tta.aliases.d4_transform()
ms = timeit(lambda: model.forward_tta(x, t, True), n=3, warm=2)
print(f"star 1024^2 d4 (8 views) eager: {ms:.2f} ms -> {8*1872.19/ms:.1f} TFLOP/s algorithmic", flush=True)
ms1 = timeit(lambda: model(x), n=3, warm=1)
print(f"star 1024^2 single view eager: {ms1:.2f} ms", flush=True)
print("max mem GB", torch.cuda.max_memory_allocated()/2**30)
K.CONV_TRACE = []
model.forward_tta(x, t, True); torch.cuda.synchronize()
tr, K.CONV_TRACE = K.CONV_TRACE, None
agg = {}
for f, a, b, shp in tr:
    e = agg.setdefault(shp, [0, 0.0, 0.0]); e[0] += 1; e[1] += a.elapsed_time(b); e[2] += f
tot = sum(v[1] for v in agg.values())
print(f"conv launches {len(tr)} total {tot:.2f} ms (event-bracketed, includes launch gaps)")
for shp, (n, ms, f) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    print(f"  N{shp[0]} {shp[1]}x{shp[2]} C{shp[3]}->{shp[4]} k{shp[5]} s{shp[6]}: x{n} {ms:.3f} ms {f/ms/1e9:.0f} TFLOP/s")
# per-kernel profile through torch profiler
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    model.forward_tta(x, t, True); torch.cuda.synchronize()
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=25, max_name_column_width=60))
