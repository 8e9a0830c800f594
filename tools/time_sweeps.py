"""Times the coarse stage with CUDA events.  Under the test hooks of csrc/coarse_tc.cu it times their reference sequences:
POPE_TC_DEBUG=16 (two-sweep online softmax, ungated) and POPE_TC_DEBUG=1024 (the single sweep as one launch).
    python tools/time_sweeps.py                 64 pairs at 480x640 (60x80 tokens), bf16
    python tools/time_sweeps.py highres [n]     n (default 4) pairs at 960x1280 (120x160 = 19 200 tokens, BASELINE configs[3])
    python tools/time_sweeps.py f32 [simt]      64 pairs, fp32 features: tensor-core split path (default) or the fp32-FMA kernels
    python tools/time_sweeps.py sigma <s>       64 pairs, bf16, features scaled by s (3.06 = token norm 49, |S| log2(e) ~ 135)
    python tools/time_sweeps.py hard            64 pairs, bf16, the hard set (x50 rows: every pair goes to the gated robust launch)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from pope_b200 import _lib, ops, synth
hi = len(sys.argv) > 1 and sys.argv[1] == "highres"
f32 = len(sys.argv) > 1 and sys.argv[1] == "f32"
impl = _lib.COARSE_SIMT if (f32 and len(sys.argv) > 2 and sys.argv[2] == "simt") else _lib.COARSE_AUTO
sig = float(sys.argv[2]) if len(sys.argv) > 2 and sys.argv[1] == "sigma" else 1.0
hard = len(sys.argv) > 1 and sys.argv[1] == "hard"
n = (int(sys.argv[2]) if len(sys.argv) > 2 else 4) if hi else 64
hc, wc = (120, 160) if hi else (60, 80)
L = hc * wc
dev = torch.device("cuda:0")
if hard:
    f0, f1 = synth.hard_coarse_features(1234, n, L, L, 256, dtype=torch.bfloat16)
else:
    f0, f1 = synth.coarse_features(1234, n, L, L, 256, sigma=sig, dtype=torch.float32 if f32 else torch.bfloat16)
d0, d1 = f0.to(dev), f1.to(dev)
ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, L, L, 256, _lib.dtype_code(d0)), dtype=torch.uint8, device=dev)
for _ in range(3):
    r = ops.coarse_match(d0, d1, (hc, wc), (hc, wc), 8.0, workspace=ws, impl=impl)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10):
    r = ops.coarse_match(d0, d1, (hc, wc), (hc, wc), 8.0, workspace=ws, impl=impl)
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 10
print(("fp32 " + ("fp32-FMA kernels" if impl == _lib.COARSE_SIMT else "tcgen05 split path") + "  ") if f32 else "", end="")
print(("sigma %.2f  " % sig) if sig != 1.0 else ("hard set  " if hard else ""), end="")
print("POPE_TC_DEBUG=%s coarse %.3f ms/step  n=%d L=S=%d  M=%d flags=%d  %.0f TFLOP/s algorithmic (2 L S C per pair)" % (
    os.environ.get("POPE_TC_DEBUG", "0"), ms, n, L, r.total(), r.flags(), n * 2.0 * L * L * 256 / (ms * 1e-3) / 1e12))
