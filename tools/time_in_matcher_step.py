"""Steps 3-5 of Matcher.forward (coarse match -> window gather -> FinePreprocess Linears -> fine transformer -> fine match)
in bf16 (or, with `float32`, at fp32 accuracy) on 64 pairs at 480x640, with the synthetic inputs of bench.py's
`in_matcher_figure`, four ways (CUDA events after warm-up, one line of JSON with each arm's peak
torch.cuda.max_memory_allocated):
  (a) module      the Matcher(config, fine_cuda_bf16=True) modules (fine_cuda_fp32=True for float32): one host sync per step
                  (the match count)
  (b) device      ops.match_pairs_device(fine_level=Matcher.fine_level(dev, dtype)) on one stream, no host sync
  (c) runner      driver.DeviceBatchRunner with two streams over the timed steps
  (d) graph       a CUDA graph of (b), replayed
(b) is checked against (a) on the live rows, bit for bit.  All four run the same kernels, (b)-(d) in their forms bounded by
the device match count on capacity-sized launches; (a) has the host sync instead.
    python tools/time_in_matcher_step.py [pairs] [steps] [bfloat16|float32]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pope_b200
from pope_b200 import _lib, driver, ops, synth

n = int(sys.argv[1]) if len(sys.argv) > 1 else 64
K = int(sys.argv[2]) if len(sys.argv) > 2 else 20
DT = getattr(torch, sys.argv[3]) if len(sys.argv) > 3 else torch.bfloat16
assert DT in (torch.bfloat16, torch.float32), DT
F32 = DT == torch.float32
dev = torch.device("cuda:0")
H, W_IMG, HC, WC = 480, 640, 60, 80
L = HC * WC
hf, wf = HC * 4, WC * 4
shapes = {"hw0_i": torch.Size([H, W_IMG]), "hw1_i": torch.Size([H, W_IMG]), "hw0_c": torch.Size([HC, WC]),
          "hw1_c": torch.Size([HC, WC]), "hw0_f": torch.Size([hf, wf]), "hw1_f": torch.Size([hf, wf]), "bs": n}

torch.manual_seed(0)
m = pope_b200.Matcher(pope_b200.make_default_cfg(), fine_cuda_bf16=not F32, fine_cuda_fp32=F32).eval().to(dev)
f0, f1 = synth.coarse_features(99, n, L, L, 256, dtype=DT)
g = torch.Generator(device=dev).manual_seed(98)
ff0 = torch.randn(n, hf, wf, 128, device=dev, generator=g).to(DT).permute(0, 3, 1, 2)
ff1 = torch.randn(n, hf, wf, 128, device=dev, generator=g).to(DT).permute(0, 3, 1, 2)
f0, f1 = f0.to(dev), f1.to(dev)
fl = m.fine_level(dev, dtype=DT)
args = (f0, f1, ff0, ff1, (H, W_IMG), (HC, WC), (HC, WC))


def module_step():
    data = dict(shapes)
    with torch.no_grad():
        m.coarse_matching(f0, f1, data)
        w0, w1 = m.fine_preprocess(ff0, ff1, f0, f1, data)
        if w0.size(0):
            w0, w1 = m.loftr_fine(w0, w1)
        m.fine_matching(w0, w1, data)
    return data


ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, L, L, 256, _lib.dtype_code(f0)), dtype=torch.uint8,
                 device=dev)
fws = ops.fine_level_workspace(n * L, 25, dev, dtype=DT)


def device_step():
    return ops.match_pairs_device(*args, workspace=ws, fine_level=fl, fine_workspace=fws)


def timed(fn, warm=3):
    torch.cuda.reset_peak_memory_stats(dev)
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K


# correctness first: (b) against (a) on the live rows
data = module_step()
res = device_step()
k = res.total()
same = k == data["b_ids"].numel() and all(torch.equal(res[key][:k], data[key]) for key in ("b_ids", "i_ids", "j_ids", "mconf"))
same = same and all(torch.equal(res[key][:k].view(torch.int32), data[key].view(torch.int32)) for key in ("expec_f", "mkpts1_f"))
del res, data

out, peak = {}, {}
for key, fn in (("module", module_step), ("device", device_step)):
    out[key + "_ms"] = timed(fn)
    peak[key] = torch.cuda.max_memory_allocated(dev)

runner = driver.DeviceBatchRunner(dev, 2)


def runner_steps():
    runner.fork()
    for _ in range(K):
        runner.submit(*args, fine_level=fl)
    runner.join()


torch.cuda.reset_peak_memory_stats(dev)
runner_steps()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
runner_steps()
e1.record()
torch.cuda.synchronize()
out["runner_ms"] = e0.elapsed_time(e1) / K
peak["runner"] = torch.cuda.max_memory_allocated(dev)
del runner
torch.cuda.empty_cache()

side = torch.cuda.Stream(dev)
side.wait_stream(torch.cuda.current_stream(dev))
with torch.cuda.stream(side):
    device_step()
torch.cuda.current_stream(dev).wait_stream(side)
torch.cuda.synchronize()
graph = torch.cuda.CUDAGraph()
with torch.cuda.graph(graph, stream=side):
    gres = device_step()
out["graph_ms"] = timed(graph.replay)
peak["graph"] = torch.cuda.max_memory_allocated(dev)
graph_same = gres.total() == k

try:
    name, power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                 capture_output=True, text=True, check=True).stdout.strip().split(", ")
except Exception:
    name, power = torch.cuda.get_device_name(dev), "unknown"
prec = "fp32 accuracy" if F32 else "bf16"
line = {"workload": f"{n} pairs at 480x640, {prec}, steps 3-5 of Matcher.forward incl. the fine level", "pairs": n,
        "matches": k, "steps_timed": K, "card": name, "power_limit": power, "device_equals_module": bool(same),
        "graph_count_equal": bool(graph_same)}
for key in ("module", "device", "runner", "graph"):
    line[key] = {"ms_per_step": round(out[key + "_ms"], 4), "pairs_per_s": round(n / out[key + "_ms"] * 1e3),
                 "peak_gb": round(peak[key] / 1e9, 2)}
print(json.dumps(line))
sys.exit(0 if same and graph_same else 1)
