"""One 48-map pass (6 tiles x 8 D4 views, proposed net, bf16, CUDA graph) timed in isolation (dev tool; the line it
prints starts with the EDS_* environment it ran under)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
import helpers
from eyediseasesegmentation_b200 import ttach_compat as tta
m = helpers.build_product_model("unetplusplusstar", helpers.star_cfg(32)).to("cuda")
m.precision = "bf16"
x = torch.randn(6, 3, 1024, 1024, device="cuda")
t = tta.aliases.d4_transform()
for _ in range(3):
    m.forward_tta(x, t, merge=False)
torch.cuda.synchronize()
ts = []
for _ in range(8):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); m.forward_tta(x, t, merge=False); b.record(); torch.cuda.synchronize()
    ts.append(a.elapsed_time(b))
print(" ".join(f"{k}={v}" for k, v in os.environ.items() if k.startswith("EDS_")), f"pass: median {sorted(ts)[4]:.2f} ms  min {min(ts):.2f} ms")
