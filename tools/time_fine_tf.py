"""Times the CUDA fine transformer (2 layers: self, cross) + FinePreprocess Linears on M windows of 25 tokens
(default: the bench workload's 162 812 matches per 64 pairs), and the torch reference modules in fp32 / bf16 beside it."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import pope_b200
from pope_b200 import ops

M = int(sys.argv[1]) if len(sys.argv) > 1 else 162812
dev = torch.device("cuda:0")
torch.manual_seed(0)
m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval().to(dev)
g = torch.Generator(device=dev).manual_seed(1)
w0 = torch.randn(M, 25, 128, device=dev, generator=g).to(torch.bfloat16)
w1 = torch.randn(M, 25, 128, device=dev, generator=g).to(torch.bfloat16)
packed = torch.cat([ops.pack_fine_layer({k: v for k, v in l.state_dict().items()}, dev) for l in m.loftr_fine.layers])
ws = ops.fine_level_workspace(M, 25, dev, merge=False)
names = m.loftr_fine.layer_names

def timed(fn, reps=3):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps

a, b = w0.clone(), w1.clone()
t_cuda = timed(lambda: ops.fine_transformer(a, b, packed, names, ws))
print(f"CUDA bf16 fine transformer: {t_cuda:.3f} ms for M={M} windows ({M * 25 * 2 / t_cuda / 1e3:.1f} M tokens/s, "
      f"{33.0e6 * M / t_cuda / 1e9:.1f} TFLOP/s at 33 MFLOP/match)")
Ms = min(M, 20000)
with torch.no_grad():
    x0, x1 = w0[:Ms].float(), w1[:Ms].float()
    from pope_b200.feature_net import LocalFeatureTransformer
    t32 = timed(lambda: m.loftr_fine(x0, x1), 2)
    mb = pope_b200.Matcher(pope_b200.make_default_cfg()).eval().to(dev).to(torch.bfloat16)
    y0, y1 = w0[:Ms], w1[:Ms]
    t16 = timed(lambda: LocalFeatureTransformer.forward(mb.loftr_fine, y0, y1), 2)      # the stock PyTorch layers
print(f"torch fp32 modules: {t32 * M / Ms:.1f} ms (scaled from {Ms} windows), torch bf16 modules: {t16 * M / Ms:.1f} ms")
