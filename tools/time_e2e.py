"""End-to-end host pipeline (pope_pipeline_run: pinned host buffers in, pinned host buffers out) on bench.py's workload,
over chunk sizes and the POPE_PIPELINE_F1 modes.  Wall clock around the call (it returns
after every copy has landed).  usage: python tools/time_e2e.py [pairs] [--chunks 8,16,32] [--modes union,windows]

--fine-level: the same pipeline with and without the bf16 fine level of a random-init Matcher(fine_cuda_bf16=True)
attached (pope_pipeline_set_fine_level), the two forms alternated run by run on the same handle and pinned buffers; also
prints the GPU's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pope_b200 import driver, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("pairs", nargs="?", type=int, default=64)
    ap.add_argument("--chunks", default="8,16,32")
    ap.add_argument("--modes", default="union")
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--fine-level", action="store_true",
                    help="time each chunk / mode with and without the bf16 fine level, alternating")
    a = ap.parse_args()
    n, hc, wc = a.pairs, 60, 80
    L = hc * wc
    f0, f1 = synth.coarse_features(1234, n, L, L, 256, dtype=torch.bfloat16)
    g = torch.Generator().manual_seed(4321)
    driver.bind_host_to_gpu(0)
    h_f0, h_f1 = f0.pin_memory(), f1.pin_memory()
    h_ff0 = torch.randn(n, hc * 4, wc * 4, 128, generator=g).to(torch.bfloat16).pin_memory()
    h_ff1 = torch.randn(n, hc * 4, wc * 4, 128, generator=g).to(torch.bfloat16).pin_memory()
    if a.fine_level:
        return fine_level_rows(a, n, hc, wc, (h_f0, h_f1, h_ff0, h_ff1))
    rows = []
    for chunk in [int(c) for c in a.chunks.split(",")]:
        pl = driver.Pipeline(torch.bfloat16, chunk, (480, 640), (hc, wc), (hc, wc), device=0)
        out = pl.alloc_outputs(n)
        for mode in a.modes.split(","):
            os.environ["POPE_PIPELINE_F1"] = mode
            pl.run(h_f0, h_f1, h_ff0, h_ff1, out)
            t0 = time.perf_counter()
            for _ in range(a.reps):
                pl.run(h_f0, h_f1, h_ff0, h_ff1, out)
            dt = (time.perf_counter() - t0) / a.reps
            rows.append({"chunk": chunk, "mode": pl.last_f1_mode, "ms": round(1e3 * dt, 3),
                         "pairs_per_s": round(n / dt, 1), "h2d_gb": round(pl.last_h2d_bytes / 1e9, 4),
                         "h2d_gbs": round(pl.last_h2d_bytes / dt / 1e9, 2), "matches": int(out["counts"].sum())})
            print(json.dumps(rows[-1]), flush=True)
        pl.close()


def fine_level_rows(a, n, hc, wc, host):
    import pope_b200
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print(json.dumps({"gpu": q.stdout.strip() or q.stderr.strip()}), flush=True)
    torch.manual_seed(0)
    matcher = pope_b200.Matcher(pope_b200.make_default_cfg(), fine_cuda_bf16=True).eval().to("cuda:0")
    fl = matcher.fine_level(torch.device("cuda", 0))
    for chunk in [int(c) for c in a.chunks.split(",")]:
        pl = driver.Pipeline(torch.bfloat16, chunk, (480, 640), (hc, wc), (hc, wc), device=0)
        out = pl.alloc_outputs(n)
        for mode in a.modes.split(","):
            os.environ["POPE_PIPELINE_F1"] = mode
            times, h2d, matches = {False: [], True: []}, {}, {}
            for rep in range(a.reps + 1):                  # rep 0 warms both forms up
                for fine in (False, True):
                    pl.set_fine_level(fl if fine else None)
                    t0 = time.perf_counter()
                    pl.run(*host, out)
                    if rep:
                        times[fine].append(time.perf_counter() - t0)
                    h2d[fine], matches[fine] = pl.last_h2d_bytes, int(out["counts"].sum())
            for fine in (False, True):
                dt = sum(times[fine]) / len(times[fine])
                print(json.dumps({"chunk": chunk, "mode": pl.last_f1_mode, "fine_level": fine, "ms": round(1e3 * dt, 3),
                                  "ms_min_max": [round(1e3 * min(times[fine]), 3), round(1e3 * max(times[fine]), 3)],
                                  "pairs_per_s": round(n / dt, 1), "h2d_gb": round(h2d[fine] / 1e9, 4),
                                  "h2d_gbs": round(h2d[fine] / dt / 1e9, 2), "matches": matches[fine]}), flush=True)
        pl.close()


if __name__ == "__main__":
    main()
