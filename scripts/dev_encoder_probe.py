"""Encoder probe: UNet++ (unetplusplus_deepsup, SCSE decoder) at cfg-2's shape -- 16 images of 1024 x 1024, 4-view
flip TTA (64 maps per pass), bf16 -- with the se_resnet50 encoder (baseline) and the ResNet-50 family that runs its
32-group 3x3 convolutions on the grouped tcgen05 kernel (resnet50, resnext50_32x4d, se_resnext50_32x4d).

Per encoder it records
  * images/s of forward_tta (CUDA-graph replays, median of the timed passes);
  * every grouped convolution launch of one eager pass: CUDA-event time, algorithmic bytes (input + output + the
    group-sized weights, bf16) and their fraction of the device-to-device copy rate measured in the same run, the
    algorithmic FLOPs and the MMA work the tensor pipe actually does (the block-diagonal 64-channel K: 64 / cpg times
    the algorithmic work);
  * time shares by kernel class (device time between consecutive launch events of one eager pass).
The card name and power limit are read in the same run.  Writes one JSON file (default under profiles/).

  python scripts/dev_encoder_probe.py [--out profiles/r03_encoder_probe.json] [--passes 5]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import helpers  # noqa: E402
from eyediseasesegmentation_b200 import kernels as K, ttach_compat as tta  # noqa: E402

ENCODERS = ("se_resnet50", "resnet50", "resnext50_32x4d", "se_resnext50_32x4d")
BATCH, SIZE = 16, 1024


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                              "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:          # the numbers still say which device they come from
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


def copy_rate(nbytes=4 << 30, reps=20):
    """Device-to-device copy, bytes read + written per second (the HBM reference of the grouped layers)."""
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        b.copy_(a)
    t1.record()
    torch.cuda.synchronize()
    return 2.0 * nbytes * reps / (t0.elapsed_time(t1) / 1e3)


def probe(enc, passes, copy_bps):
    cfg = dict(encoder_name=enc, encoder_weights=None, classes=1, decoder_attention_type="scse")
    model = helpers.build_product_model("unetplusplus_deepsup", cfg).to("cuda")
    model.precision = "bf16"
    x = torch.randn(BATCH, 3, SIZE, SIZE, device="cuda")
    tfm = tta.aliases.flip_transform()
    for _ in range(3):                                 # eager, capture, replay
        model.forward_tta(x, tfm, merge=False)
    torch.cuda.synchronize()
    ts = []
    for _ in range(passes):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        model.forward_tta(x, tfm, merge=False)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    med = sorted(ts)[len(ts) // 2]

    K.CONV_TRACE = []                                  # a trace forces the eager path
    model.forward_tta(x, tfm, merge=False)
    torch.cuda.synchronize()
    trace, K.CONV_TRACE = K.CONV_TRACE, None
    layers = []
    for flops, e0, e1, shape in trace:
        if len(shape) < 8:
            continue
        N, H, W, C, Cout, R, stride, groups = shape
        cpg = C // groups
        Ho, Wo = K.conv_out_hw(H, W, R, stride, 1)
        ms = e0.elapsed_time(e1)
        nbytes = 2.0 * (N * H * W * C + N * Ho * Wo * Cout + Cout * R * R * cpg)
        mma = 2.0 * N * Ho * Wo * Cout * R * R * 64
        layers.append({"maps": N, "in_hw": [H, W], "channels": C, "cpg": cpg, "stride": stride, "ms": round(ms, 4),
                       "algorithmic_bytes": nbytes, "hbm_fraction_of_copy_rate": round(nbytes / (ms / 1e3) / copy_bps, 3),
                       "algorithmic_flops": flops, "mma_flops": mma,
                       "mma_tflops": round(mma / (ms / 1e3) / 1e12, 1)})

    K.KERNEL_TRACE = []
    start = torch.cuda.Event(enable_timing=True)
    start.record()
    model.forward_tta(x, tfm, merge=False)
    torch.cuda.synchronize()
    ktrace, K.KERNEL_TRACE = K.KERNEL_TRACE, None
    per, prev = {}, start
    for name, ev in ktrace:
        per[name] = per.get(name, 0.0) + prev.elapsed_time(ev)
        prev = ev
    total = sum(per.values()) or 1.0
    del model
    torch.cuda.empty_cache()
    return {"images_per_s": round(BATCH / (med / 1e3), 2), "pass_ms_median": round(med, 3),
            "pass_ms_all": [round(t, 3) for t in ts],
            "grouped_conv_ms_total": round(sum(l["ms"] for l in layers), 3), "grouped_layers": layers,
            "eager_pass_ms": round(total, 3),
            "shares": {k: round(v / total, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_encoder_probe.json"))
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--encoders", default=",".join(ENCODERS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dev_encoder_probe measures on a CUDA device; none is visible")
    torch.cuda.init()
    info = card()
    copy_bps = copy_rate()
    res = {"workload": f"unetplusplus_deepsup + scse, {BATCH} x {SIZE}^2, flip TTA (4 views, {4 * BATCH} maps), bf16",
           "card": info, "copy_rate_GBps": round(copy_bps / 1e9, 1),
           "notes": "images/s from CUDA-graph replays (median); per-layer times from one eager pass with CUDA "
                    "events around each grouped launch; shares from one eager pass",
           "encoders": {}}
    for enc in args.encoders.split(","):
        res["encoders"][enc] = probe(enc, args.passes, copy_bps)
        print(enc, res["encoders"][enc]["images_per_s"], "img/s", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "encoders"}))


if __name__ == "__main__":
    main()
