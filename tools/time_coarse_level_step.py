"""Everything in Matcher.forward after the backbone -- position encoding, coarse transformer, coarse match, window gather,
FinePreprocess Linears, fine transformer, fine match -- on 64 pairs at 480x640, in bf16 and at fp32 accuracy, from the
same fp32 backbone maps (synthetic, with planted correspondences), timed five ways (CUDA events after warm-up; peak
torch.cuda.max_memory_allocated per arm):
  (a) module   pos_encoding -> loftr_coarse -> steps 3-5 of Matcher(config, coarse_cuda_X=True, fine_cuda_X=True), as
               Matcher.forward runs them: one host sync per step (the match count)
  (b) device   ops.match_pairs_device(coarse_level=Matcher.coarse_level(dev, X), fine_level=Matcher.fine_level(dev, X)) on
               one stream, no host sync
  (c) runner   driver.DeviceBatchRunner with two streams over the timed steps
  (d) graph    a CUDA graph of (b), replayed
  (e) host     driver.match_pairs_host with both levels on page-locked host inputs (16-pair chunks; host clock around the
               call, which returns after the last copy; pipeline creation included) and Pipeline.run on a pipeline created
               beforehand
(b) is checked against (a) bit for bit (ids, mconf, keypoints, and the transformed features), (e) against (b).  The fine
maps are given in the level's dtype to every arm.  Writes one line of JSON per dtype, and the list to the path given.
    python tools/time_coarse_level_step.py [pairs] [steps] [out.json]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pope_b200
from pope_b200 import _lib, driver, ops, synth

n = int(sys.argv[1]) if len(sys.argv) > 1 else 64
K = int(sys.argv[2]) if len(sys.argv) > 2 else 10
OUT = sys.argv[3] if len(sys.argv) > 3 else None
dev = torch.device("cuda:0")
H, W_IMG, HC, WC = 480, 640, 60, 80
L = HC * WC
hf, wf = HC * 4, WC * 4
HW = ((H, W_IMG), (HC, WC), (HC, WC))
shapes = {"hw0_i": torch.Size([H, W_IMG]), "hw1_i": torch.Size([H, W_IMG]), "hw0_c": torch.Size([HC, WC]),
          "hw1_c": torch.Size([HC, WC]), "hw0_f": torch.Size([hf, wf]), "hw1_f": torch.Size([hf, wf]), "bs": n}

# the backbone's outputs, shared by both dtypes: fp32 coarse maps [n, 256, 60, 80] and fine maps [n, 128, 240, 320]
f0, f1 = synth.coarse_features(99, n, L, L, 256)
c0_host = f0.transpose(1, 2).reshape(n, 256, HC, WC).contiguous()
c1_host = f1.transpose(1, 2).reshape(n, 256, HC, WC).contiguous()
del f0, f1
c0, c1 = c0_host.to(dev), c1_host.to(dev)
g = torch.Generator(device=dev).manual_seed(98)
ff0_32 = torch.randn(n, hf, wf, 128, device=dev, generator=g).permute(0, 3, 1, 2)
ff1_32 = torch.randn(n, hf, wf, 128, device=dev, generator=g).permute(0, 3, 1, 2)


def timed(fn, warm=2):
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
    return e0.elapsed_time(e1) / K, torch.cuda.max_memory_allocated(dev)


def card():
    try:
        name, power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                     capture_output=True, text=True, check=True).stdout.strip().split(", ")
    except Exception:
        name, power = torch.cuda.get_device_name(dev), "unknown"
    return name, power


def run(DT):
    F32 = DT == torch.float32
    torch.manual_seed(0)
    m = pope_b200.Matcher(pope_b200.make_default_cfg(), coarse_cuda_bf16=not F32, fine_cuda_bf16=not F32,
                          coarse_cuda_fp32=F32, fine_cuda_fp32=F32).eval().to(dev)
    ff0, ff1 = ff0_32.to(DT), ff1_32.to(DT)
    cl, fl = m.coarse_level(dev, DT), m.fine_level(dev, DT)
    args = (c0, c1, ff0, ff1) + HW

    def module_step():
        data = dict(shapes)
        with torch.no_grad():
            if F32:                 # Matcher.forward, matcher.py: the stock encoding for fp32, the kernel for bf16
                a, b = m.pos_encoding(c0).flatten(2).transpose(1, 2), m.pos_encoding(c1).flatten(2).transpose(1, 2)
            else:
                a, b = ops.coarse_pos_encode(c0, m.pos_encoding.pe), ops.coarse_pos_encode(c1, m.pos_encoding.pe)
            a, b = m.loftr_coarse(a, b)
            m.coarse_matching(a, b, data)
            w0, w1 = m.fine_preprocess(ff0, ff1, a, b, data)
            if w0.size(0):
                w0, w1 = m.loftr_fine(w0, w1)
            m.fine_matching(w0, w1, data)
        return data, a, b

    ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, L, L, 256, _lib.dtype_code(ff0)), dtype=torch.uint8,
                     device=dev)
    fws = ops.fine_level_workspace(n * L, 25, dev, dtype=DT)
    cws = ops.coarse_tf_workspace(n, L, L, dev, dtype=DT)

    def device_step():
        return ops.match_pairs_device(*args, workspace=ws, fine_level=fl, fine_workspace=fws, coarse_level=cl,
                                      coarse_workspace=cws)

    # correctness first: (b) against (a), bit for bit
    data, a, b = module_step()
    res = device_step()
    k = res.total()
    same = k == data["b_ids"].numel() and res.flags() == 0
    same = same and all(torch.equal(res[key][:k], data[key]) for key in ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f"))
    same = same and all(torch.equal(res[key][:k].view(torch.int32), data[key].view(torch.int32))
                        for key in ("expec_f", "mkpts1_f"))
    same = same and torch.equal(res["feat_c0"], a) and torch.equal(res["feat_c1"], b)
    want = {key: res[key][:k].cpu() for key in ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f")}
    del res, data, a, b

    out, peak = {}, {}
    for key, fn in (("module", module_step), ("device", device_step)):
        out[key], peak[key] = timed(fn)

    runner = driver.DeviceBatchRunner(dev, 2)

    def runner_steps():
        runner.fork()
        for _ in range(K):
            runner.submit(*args, fine_level=fl, coarse_level=cl)
        runner.join()

    torch.cuda.reset_peak_memory_stats(dev)
    runner_steps()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    runner_steps()
    e1.record()
    torch.cuda.synchronize()
    out["runner"], peak["runner"] = e0.elapsed_time(e1) / K, torch.cuda.max_memory_allocated(dev)
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
    out["graph"], peak["graph"] = timed(graph.replay)
    graph_same = gres.total() == k
    del graph, gres, ws, fws, cws
    torch.cuda.empty_cache()

    # (e) the host pipeline from page-locked host inputs
    host = [c0_host.pin_memory(), c1_host.pin_memory(), ff0.cpu().pin_memory(), ff1.cpu().pin_memory()]
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    t0 = time.perf_counter()
    got = driver.match_pairs_host(*host, *HW, chunk_pairs=16, fine_level=fl, coarse_level=cl)
    host_ms = (time.perf_counter() - t0) * 1e3
    flat = driver.flatten_slots(got)
    host_same = all(torch.equal(flat[key], want[key]) for key in want)
    pl = driver.Pipeline(DT, 16, HW[0], HW[1], HW[2], fine_level=fl, coarse_level=cl)
    nhwc = [t.permute(0, 2, 3, 1).contiguous() for t in host[2:]]
    outb = pl.alloc_outputs(n)
    pl.run(host[0], host[1], *nhwc, out=outb)
    t0 = time.perf_counter()
    for _ in range(3):
        pl.run(host[0], host[1], *nhwc, out=outb)
    run_ms = (time.perf_counter() - t0) * 1e3 / 3
    h2d = pl.last_h2d_bytes
    pl.close()
    peak["host"] = torch.cuda.max_memory_allocated(dev)   # (the pipeline's own cudaMalloc buffers are not in torch's count)
    del m, cl, fl, host, nhwc, outb
    torch.cuda.empty_cache()

    name, power = card()
    prec = "fp32 accuracy" if F32 else "bf16"
    line = {"workload": f"{n} pairs at 480x640, {prec}, Matcher.forward after the backbone (coarse level + steps 3-5 "
                        "incl. the fine level) from fp32 backbone maps", "dtype": str(DT), "pairs": n, "matches": k,
            "steps_timed": K, "card": name, "power_limit": power, "device_equals_module": bool(same),
            "graph_count_equal": bool(graph_same), "host_equals_device": bool(host_same)}
    for key in ("module", "device", "runner", "graph"):
        line[key] = {"ms_per_step": round(out[key], 3), "pairs_per_s": round(n / out[key] * 1e3),
                     "peak_gb": round(peak[key] / 1e9, 2)}
    line["host"] = {"match_pairs_host_ms": round(host_ms, 1), "pipeline_run_ms": round(run_ms, 1),
                    "pairs_per_s": round(n / run_ms * 1e3), "h2d_bytes_per_pair": h2d // n,
                    "coarse_map_bytes_per_pair": 2 * L * 256 * 4, "torch_peak_gb": round(peak["host"] / 1e9, 2)}
    print(json.dumps(line), flush=True)
    return line, same and graph_same and host_same


lines, ok = [], True
for DT in (torch.bfloat16, torch.float32):
    line, good = run(DT)
    lines.append(line)
    ok = ok and good
if OUT:
    os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
    with open(OUT, "w") as fh:
        json.dump(lines, fh, indent=1)
sys.exit(0 if ok else 1)
