"""Times the fine level on M windows of 25 tokens (default: the bench workload's 162 812 matches per 64 pairs): the fine
transformer (2 layers: self, cross) alone and with FinePreprocess' two Linears in front of it, as the stock PyTorch
modules in fp32 (TF32 off) and cast to bf16, and as the CUDA fp32-accuracy and bf16 paths (csrc/fine_tf.cu).  CUDA events,
after a warm-up of every timed call; the windows (M x 25 x 128 per side) are larger than the 126 MB L2.  Prints the card's
name and power limit and one JSON line (also written to the path given with --json)."""
import argparse
import copy
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pope_b200
from pope_b200 import ops
from pope_b200.feature_net import LocalFeatureTransformer

ap = argparse.ArgumentParser()
ap.add_argument("--windows", type=int, default=162812)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--json", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("time_fine_tf.py needs a CUDA device")
M = args.windows
dev = torch.device("cuda:0")


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
torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False     # the stock fp32 arm is fp32
m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval().to(dev)
tf, pre = m.loftr_fine, m.fine_preprocess
names = tf.layer_names
g = torch.Generator(device=dev).manual_seed(1)
w0 = torch.randn(M, 25, 128, device=dev, generator=g)
w1 = torch.randn(M, 25, 128, device=dev, generator=g)
n, L = 64, 4800
fc0, fc1 = torch.randn(n, L, 256, device=dev, generator=g), torch.randn(n, L, 256, device=dev, generator=g)
ids = [torch.randint(0, hi, (M,), device=dev, generator=g) for hi in (n, L, L)]
res = {"card": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "windows": M, "tokens_per_window": 25}


def stock_merge(p, a, b, c0, c1):
    """fine_preprocess.py:50-57 with the stock Linears."""
    c = p.down_proj(torch.cat([c0[ids[0], ids[1]], c1[ids[0], ids[2]]], 0))
    merged = p.merge_feat(torch.cat([torch.cat([a, b], 0), c[:, None, :].expand(-1, 25, -1)], -1))
    return merged[:M], merged[M:]


with torch.no_grad():
    for dt, tag in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        st = LocalFeatureTransformer(copy.deepcopy(tf.config)).eval().to(dev)
        st.load_state_dict(tf.state_dict())
        sp = copy.deepcopy(pre).to(dt)
        st = st.to(dt)
        x0, x1, c0, c1 = w0.to(dt), w1.to(dt), fc0.to(dt), fc1.to(dt)
        res[f"tf_stock_{tag}_ms"] = timed(lambda: st(x0, x1), args.reps)
        res[f"level_stock_{tag}_ms"] = timed(lambda: st(*stock_merge(sp, x0, x1, c0, c1)), args.reps)
        del st, sp
        torch.cuda.empty_cache()
        packed, ppre = tf._packed_weights(dev, dt), pre._packed_weights(dev, dt)
        ws = ops.fine_level_workspace(M, 25, dev, dtype=dt)
        a, b = x0.clone(), x1.clone()
        res[f"tf_cuda_{tag}_ms"] = timed(lambda: ops.fine_transformer(a, b, packed, names, ws), args.reps)

        def cuda_level():
            ops.fine_merge_coarse(a, b, c0, c1, *ids, ppre, ws)
            ops.fine_transformer(a, b, packed, names, ws)
        res[f"level_cuda_{tag}_ms"] = timed(cuda_level, args.reps)
        del a, b, ws, x0, x1, c0, c1
        torch.cuda.empty_cache()
for stage in ("tf", "level"):
    res[f"{stage}_cuda_fp32_speedup_vs_stock_fp32"] = round(res[f"{stage}_stock_fp32_ms"] / res[f"{stage}_cuda_fp32_ms"], 3)
    res[f"{stage}_cuda_bf16_speedup_vs_stock_bf16"] = round(res[f"{stage}_stock_bf16_ms"] / res[f"{stage}_cuda_bf16_ms"], 3)

for k, v in res.items():
    print(f"{k:45s} {v}")
line = json.dumps(res)
print(line)
if args.json:
    os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
    with open(args.json, "w") as fh:
        fh.write(line + "\n")
