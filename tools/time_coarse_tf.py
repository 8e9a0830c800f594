"""Times the coarse LoFTR transformer (8 layers, d_model 256) on N pairs at 480x640 (60x80 = 4800 tokens per image;
default N = 64): the stock PyTorch modules in fp32 and cast to bf16, and the CUDA bf16 path (csrc/coarse_tf.cu); then
Matcher.forward from images with the default flags, with fine_cuda_bf16 and with both bf16 flags.  CUDA events, after
a warm-up of every timed shape; the inputs (N x 4800 x 256 per side) are larger than the 126 MB L2 at N = 64.
Prints the card's name and power limit and one JSON line (also written to the path given with --json)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pope_b200
from pope_b200 import ops, synth
from pope_b200.feature_net import LocalFeatureTransformer

# 4 * 2 * 256^2 (q, k, v, merge) + 2 * 512^2 + 2 * 512 * 256 (MLP) per token and layer, x 4800 tokens x 2 images x 8 layers
FLOP_PER_PAIR = 100.7e9
BF16_PEAK_TFLOPS = {"burst": 1659.8, "sustained": 1404.1}    # cuBLAS bf16 on one B200 (MEASURED_PEAKS.json, SURVEY.md)

ap = argparse.ArgumentParser()
ap.add_argument("--pairs", type=int, default=64)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--json", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("time_coarse_tf.py needs a CUDA device")
dev = torch.device("cuda:0")
N, H, W = args.pairs, 60, 80
L = H * W


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


torch.manual_seed(0)
cfg = pope_b200.make_default_cfg()
m = pope_b200.Matcher(cfg).eval().to(dev)
tf = m.loftr_coarse
f0, f1 = synth.coarse_features(1, N, L, L, dtype=torch.bfloat16)
f0, f1 = f0.to(dev), f1.to(dev)
res = {"card": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "pairs": N, "tokens_per_image": L}

with torch.no_grad():
    x0, x1 = f0.float(), f1.float()
    res["tf_stock_fp32_ms"] = timed(lambda: tf(x0, x1), args.reps)
    tb = LocalFeatureTransformer(cfg["coarse"]).eval().to(dev)
    tb.load_state_dict(tf.state_dict())
    tb = tb.to(torch.bfloat16)
    res["tf_stock_bf16_ms"] = timed(lambda: tb(f0, f1), args.reps)
    packed = tf._packed_weights(dev)
    ws = ops.coarse_tf_workspace(N, L, L, dev)
    a, b = f0.clone(), f1.clone()
    res["tf_cuda_bf16_ms"] = timed(lambda: ops.coarse_transformer(a, b, packed, tf.layer_names, ws), args.reps)
    for k in ("tf_stock_fp32", "tf_stock_bf16", "tf_cuda_bf16"):
        tflops = FLOP_PER_PAIR * N / (res[k + "_ms"] * 1e-3) / 1e12
        res[k + "_tflops"] = round(tflops, 1)
        res[k + "_share_of_sustained_bf16_peak"] = round(tflops / BF16_PEAK_TFLOPS["sustained"], 4)
    res["cuda_speedup_vs_stock_bf16"] = round(res["tf_stock_bf16_ms"] / res["tf_cuda_bf16_ms"], 3)

    gen = torch.Generator(device=dev).manual_seed(2)
    img = {"image0": torch.rand(N, 1, 480, 640, device=dev, generator=gen),
           "image1": torch.rand(N, 1, 480, 640, device=dev, generator=gen)}
    for name, flags in (("matcher_default", {}), ("matcher_fine_bf16", {"fine_cuda_bf16": True}),
                        ("matcher_fine_and_coarse_bf16", {"fine_cuda_bf16": True, "coarse_cuda_bf16": True})):
        mm = pope_b200.Matcher(cfg, **flags).eval().to(dev)
        mm.load_state_dict(m.state_dict())
        res[name + "_ms"] = timed(lambda: mm(dict(img)), max(2, args.reps // 2))
        del mm
        torch.cuda.empty_cache()

for k, v in res.items():
    print(f"{k:45s} {v}")
line = json.dumps(res)
print(line)
if args.json:
    os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
    with open(args.json, "w") as fh:
        fh.write(line + "\n")
