"""Tiny invocation of every kernel family for compute-sanitizer (memcheck)."""
import sys, os, math
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from eyediseasesegmentation_b200 import kernels as K, _lib, ttach_compat as tta
dev = "cuda"
torch.manual_seed(0)
def conv(N, H, W, C, Cout, R, impl, stride=1, x1c=0, res=False):
    x = torch.randn(N, H, W, C, device=dev).bfloat16()
    x1 = torch.randn(N, H, W, x1c, device=dev).bfloat16() if x1c else None
    w = (torch.randn(Cout, R, R, C + x1c, device=dev) / math.sqrt(R * R * (C + x1c))).bfloat16()
    b = torch.zeros(Cout, device=dev)
    Ho, Wo = K.conv_out_hw(H, W, R, stride, R // 2)
    r = torch.randn(N, Ho, Wo, Cout, device=dev).bfloat16() if res else None
    return K.conv2d(x, w, b, stride, R // 2, True, r, impl=impl, x1=x1)
conv(2, 20, 24, 64, 256, 3, "tc"); conv(1, 33, 17, 128, 80, 1, "tc", res=True); conv(2, 16, 16, 64, 128, 3, "tc", stride=2)
conv(1, 24, 24, 64, 512, 3, "tc", x1c=192); conv(3, 40, 20, 64, 32, 3, "halo", res=True); conv(1, 70, 13, 128, 64, 3, "halo", x1c=64)
conv(1, 66, 30, 16, 16, 3, "halo"); conv(2, 64, 64, 32, 16, 3, "halo")
K.conv3x3_small(torch.randn(2, 21, 19, 16, device=dev).bfloat16(), torch.randn(32, 3, 3, 16, device=dev).bfloat16(),
                torch.zeros(32, device=dev), True)
K.conv3x3_small(torch.randn(2, 37, 45, 16, device=dev).bfloat16(), torch.randn(16, 3, 3, 16, device=dev).bfloat16(), None, True)
srcs = [(torch.randn(2, 7, 5, 64, device=dev).bfloat16(), torch.rand(2, 64, device=dev), torch.rand(2, 7, 5, device=dev)),
        (torch.randn(2, 14, 10, 32, device=dev).bfloat16(), None, None)]
mean = torch.empty(2, 96, device=dev); d0 = torch.empty(2, 7, 5, device=dev); d1 = torch.empty(2, 14, 10, device=dev)
wv = torch.randn(96, device=dev)
K.gated_stats(srcs[0][0], srcs[0][1], srcs[0][2], wv[:64], mean, 0, True, d0, False)
K.gated_stats(srcs[1][0], None, None, wv[64:], mean, 64, False, d1, False)
sg = K.sse_finalize(d0, d1, _lib.UP_BILINEAR, 0.1)
K.concat_gated(srcs, _lib.UP_BILINEAR, torch.rand(2, 96, device=dev), sg)
K.concat_gated_split(srcs, _lib.UP_NEAREST, torch.rand(2, 96, device=dev), sg)
for (H, heads, dv, cross) in ((19, 8, 64, False), (38, 4, 8, True), (64, 8, 64, False)):
    G = 16 + (0 if cross else dv)
    qk = torch.randn(1, H, H, heads * G, device=dev).bfloat16()
    v = torch.randn(1, H, H, heads * dv, device=dev).bfloat16() if cross else None
    for ax in (0, 1):
        K.axial_attention(qk, v, ax, heads, 8, dv, torch.randn(16 + dv, 2 * H - 1, device=dev), torch.rand(heads, 3, device=dev),
                          torch.rand(2, heads * dv, device=dev), torch.rand(2, heads * dv, device=dev))
xin = torch.randn(2, 3, 96, 96, device=dev)
aug, deaug = tta.view_maps(tta.aliases.d4_transform(), 96, 96)
wst = torch.randn(7, 7, 3, 64, device=dev)
K.stem_conv_mma(xin, aug, K.stem_pack_weights(wst), torch.zeros(64, device=dev))
K.stem_conv(xin, aug, wst, torch.zeros(64, device=dev), torch.float32)
lg = torch.randn(8, 2, 96, 96, device=dev)
pr = K.tta_merge(lg, deaug, True)
full = torch.zeros(300, 420, device=dev)
K.resize_paste(pr[0], full, (0, 0, 96, 96), (100, 200), (192, 192))
img = torch.randint(0, 256, (300, 420, 3), device=dev, dtype=torch.uint8)
K.preprocess_tile(img, 10, 20, 96, [0.45, 0.22, 0.06], [0.33, 0.17, 0.09])
p8 = torch.rand(3, 12345 * 4, device=dev); g8 = (torch.rand(3, 12345 * 4, device=dev) < 0.1).to(torch.uint8)
h, st = K.pr_hist(p8, g8); K.pr_scan(h, st)
K.confusion_counts((p8 * 255).to(torch.uint8), g8 * 255)
y = torch.randn(2, 24, 24, 16, device=dev).bfloat16()
K.head_conv3x3(y, torch.randn(1, 3, 3, 16, device=dev), torch.zeros(1, device=dev))
K.maxpool2d(torch.randn(2, 33, 33, 64, device=dev).bfloat16(), 3, 2, 0, True)
torch.cuda.synchronize()
print("sanitize probe ok")
