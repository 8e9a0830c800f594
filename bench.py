#!/usr/bin/env python
"""bench.py -- matched image pairs / second of the Matcher hot path (coarse match -> window gather -> fine match).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path (one JSON line)
    python bench.py [...] --dump-outputs DIR                      # also DIR/<name>.npy: the match lists of the last timed step
    python bench.py --impl reference [...]                        # the reference's CPU path (oracle port), rank 0 only

Workload (BASELINE.json configs[1]): a batch of 64 synthetic 480x640 pairs per GPU per step -- coarse features
[64, 4800, 256] x2 and fine maps [64, 128, 240, 320] x2 (channels-last), bf16, planted correspondences
(pope_b200/synth.py).  A "step" is one pass of the hot path over that batch.

  value : pairs/s with the inputs already resident in HBM (CUDA events, max over ranks).  The batch's inputs
          (2.8 GB) are far larger than the 126 MB L2, so every step streams them from HBM.  Consecutive steps go through
          pope_b200.driver.DeviceBatchRunner: they alternate between two CUDA streams (own scratch each), so the small
          latency-bound kernels that end a step overlap the next step's sweep; stage_ms / roofline come from a separate
          pass on ONE stream, where events bracket the kernels and not the queue (`one_stream` is that pass as pairs/s:
          what a single Matcher.forward-style caller gets).
          N > 1: every step appends its packed 20-byte match records to a device buffer and the job's ONE cross-GPU
          step -- a gather of the live records to rank 0 -- runs after the K steps, inside the timed region; after the
          timed region rank 0 checks the sizes and a per-rank checksum of what it received (`gather_verified`).
  e2e   : the same metric through the C-ABI host entry (pope_pipeline_run): pinned host buffers in, pinned host
          buffers out, host<->device copies inside the timed region; with the achieved H2D rate per rank and the box's
          ceiling (plain pinned cudaMemcpyAsync from all ranks at once).
  roofline : the coarse stage (dominant) against the measured bf16 tensor peak (burst: the timed region is ~20 ms;
             the sustained figure beside it); algorithmic work 2*L*S*C per pair; `traffic` = DRAM bytes per launch from the
             committed ncu capture profiles/r2_ncu_step.csv.
             roofline_fine: the fused window-gather + fine-match kernel against the measured HBM copy bandwidth, both
             as algorithmic bytes (window overlap is served by L2) and as DRAM bytes (`dram_frac`).
  robust   : the same workload with features of token norm 49 (sigma 3.06: what the coarse transformer emits, SURVEY
             section 7; similarities reach +-135 in log2 units) -- the lazily shifted single sweep must keep it on the fast
             path (`flags` 0).
  in_matcher / highres / single_pair / retrieval / job_4096 : the other configurations of BASELINE.json (steps 3-5 of Matcher.forward
             with the fine transformer in between; configs[3] 960x1280; configs[2] 1 query vs 256 crops; configs[4] a
             4096-pair job sharded over the ranks with a single gather).
  cpu_baseline : the oracle port (same op sequence as the reference, torch CPU) on a bounded sample, rank 0: the hot path
             on synthetic features (`value`) and the full Matcher from images on one pair (`full_matcher`).
"""
from __future__ import annotations

import argparse
import csv
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "matched_pairs_per_sec_480x640"
UNIT = "pairs/s"
H, W_IMG = 480, 640
HC, WC = H // 8, W_IMG // 8          # 60 x 80 coarse cells
L = HC * WC
C_COARSE, C_FINE, FINE_STRIDE, WIN = 256, 128, 4, 5
NORM49_SIGMA = 49.0 / 16.0           # |f| = sigma * sqrt(256)
TRAFFIC_CSV = os.path.join(ROOT, "profiles", "r2_ncu_step.csv")


def workload_config(n):
    """The workload both arms are run on (the reference arm times a bounded sample of it per step): identical in both lines."""
    return {"workload": ("batch of 64 pairs at 480x640, coarse+fine matching (BASELINE configs[1])" if n == 64 else
                         f"batch of {n} pairs at 480x640, coarse+fine matching"),
            "pairs_per_gpu_per_step": n, "coarse_tokens": [HC, WC], "d_coarse": C_COARSE, "d_fine": C_FINE, "window": WIN,
            "l2_policy": "inputs_exceed_l2 (2.8 GB of features per step vs 126 MB L2)"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=64, help="pairs per GPU per step")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--coarse-impl", default="auto", choices=["auto", "simt", "tcgen05"])
    ap.add_argument("--cpu-sample-pairs", type=int, default=2)
    ap.add_argument("--in-matcher", type=int, default=64, metavar="PAIRS",
                    help="pairs for the in-Matcher figure (steps 3-5 of Matcher.forward with the FinePreprocess Linears and "
                         "the fine transformer between the CUDA stages, SURVEY 8(d)); 0 = skip")
    ap.add_argument("--highres-pairs", type=int, default=16, help="pairs of the 960x1280 block (configs[3]); 0 = skip")
    ap.add_argument("--job-pairs", type=int, default=4096, help="size of the sharded job block (configs[4]); 0 = skip")
    ap.add_argument("--streams", type=int, default=2,
                    help="device-resident steps alternate between this many CUDA streams (each with its own scratch), so "
                         "that the small latency-bound kernels at the end of a step overlap the next step's sweep")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the robust / in_matcher / highres / retrieval / job blocks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what rank 0's last timed step returned as DIR/<name>.npy, so that two "
                         "builds can be compared output for output on the same seeded inputs (bench_outputs/ is ignored by git)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d["hbm_gbs"], d["bf16_tflops"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def dram_traffic_from_profiles():
    """DRAM bytes per launch (read + write) of the coarse kernels and of the fused fine kernel, from the committed
    `ncu --set full` capture of one 64-pair step (tools/ncu_extract.py table).  None if the file is absent."""
    if not os.path.exists(TRAFFIC_CSV):
        return None, None, None
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        with open(TRAFFIC_CSV) as f:
            rows = list(csv.reader(f))
        hdr = rows[0]
        cols = {}
        for k, name in enumerate(hdr):
            for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                if name.startswith(key + " ["):
                    cols[key] = (k, mult.get(name[name.index("[") + 1:name.index("]")], 1.0))
        if len(cols) != 2 or hdr[0] != "kernel":
            return None, None, None           # not the tools/ncu_extract.py table (e.g. ncu's raw page): no traffic figure
        coarse = fine = 0.0
        for r in rows[1:]:
            if not r:
                continue
            byts = sum(float(r[k]) * m for k, m in cols.values())
            if "fine_match_maps" in r[0]:
                fine += byts
            elif any(t in r[0] for t in ("sweep_tc", "colsum_reduce", "cand_eval", "count_emit")):
                coarse += byts
    except (OSError, ValueError, IndexError):
        return None, None, None
    return (coarse or None), (fine or None), os.path.relpath(TRAFFIC_CSV, ROOT)


DUMP_KEYS = ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c", "expec_f", "mkpts0_f", "mkpts1_f")
DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir, res, max_bytes=DUMP_MAX_BYTES):
    """Writes the match lists of one hot-path step (a capacity-sized `CoarseResult`) as out_dir/<name>.npy: the rows up to the
    live match count, ids as float64 (exact), confidences and coordinates as float32, and `counts` (matches per pair, the
    total, the flag word) as float64.  Should the rows need more than `max_bytes` in all, a fixed seeded sample of them is
    written, in their order, with their indices in `rows.npy`."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    m = res.total()
    out = {k: res[k][:m].cpu().numpy() for k in DUMP_KEYS}
    out = {k: v.astype(np.float64 if v.dtype.kind in "iu" else np.float32) for k, v in out.items()}
    counts = res["counts"].cpu().numpy().astype(np.float64)
    row_bytes = sum(v[:1].nbytes for v in out.values()) + 8                 # + the row's index in rows.npy
    budget = max_bytes - counts.nbytes - 128 * (len(out) + 2)              # (an .npy header takes 128 bytes)
    if m * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(m, size=budget // row_bytes, replace=False))
        out = {k: v[rows] for k, v in out.items()}
        out["rows"] = rows.astype(np.float64)
    out["counts"] = counts
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    return sorted(out)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled in the background from before the warm-up until the end of the
    run; `summary(t0, t1)` reports the samples that fall inside the timed region (wall-clock window)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, period_ms: int = 20):
        import threading
        self.samples, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.samples.append((time.time(), ln))

    def wait_first(self, timeout=5.0):
        t0 = time.time()
        while self.proc is not None and not self.samples and time.time() - t0 < timeout:
            time.sleep(0.01)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, t0: float, t1: float):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for ts, ln in list(self.samples):
            f = [x.strip() for x in ln.split(",")]
            try:
                rows.append((ts, float(f[0]), float(f[1]), float(f[2]), [nm for nm, v in zip(names, f[3:7]) if v.lower().startswith("active")]))
            except (ValueError, IndexError):
                continue
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        inside = [r for r in rows if t0 - 0.03 <= r[0] <= t1 + 0.03]
        scope = "timed region"
        if not inside:       # region shorter than one sampling period: fall back to the samples taken under load
            pmax = max(r[3] for r in rows)
            inside = [r for r in rows if r[3] >= 0.6 * pmax]
            scope = "samples under load (timed region shorter than the sampling period)"
        reasons = sorted({x for r in inside for x in r[4]})
        return {"sm_mhz": statistics.median(r[1] for r in inside), "sm_max_mhz": max(r[2] for r in rows),
                "power_w_max": max(r[3] for r in inside), "reasons": reasons, "samples": len(inside), "scope": scope}


# ---- CPU legs (the oracle port; checker code, timed here as the baseline only) -----------------------------------------

def cpu_reference_pairs_per_sec(n_sample: int, repeats: int = 1):
    """The reference's CPU path for the hot path (oracle port: einsum -> softmax x softmax -> ... -> unfold -> gather ->
    fine match), fp32, all host threads, on `n_sample` pairs of the bench workload."""
    from oracle import pope_oracle as O
    from pope_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    f0, f1 = synth.coarse_features(1234, n_sample, L, L, C_COARSE)
    ff0, ff1 = synth.fine_feature_maps(4321, n_sample, HC * FINE_STRIDE, WC * FINE_STRIDE, C_FINE, channels_last=False)
    best, m = float("inf"), 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        out = O.match_pairs(f0, f1, ff0, ff1, (H, W_IMG), (HC, WC), (HC, WC))
        best = min(best, time.perf_counter() - t0)
        m = out["b_ids"].numel()
    return n_sample / best, best, m, torch.get_num_threads()


def cpu_full_matcher_pairs_per_sec():
    """BASELINE.md 4.1 leg (i): the whole reference Matcher.forward (src/matcher/matcher.py:29-79) on ONE 480x640 image pair
    on the host cores: backbone -> position encoding -> coarse transformer (the same torch modules, on the CPU) -> the
    oracle port of coarse matching (-> fine level only if M > 0).  Random-init weights give M = 0 on any image pair (SURVEY
    section 7, "vacuous parity trap"), exactly as in the reference, so the fine level never runs here."""
    import pope_b200
    from oracle import pope_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    g = torch.Generator().manual_seed(7)
    img0, img1 = torch.rand(1, 1, H, W_IMG, generator=g), torch.rand(1, 1, H, W_IMG, generator=g)
    best, M = float("inf"), 0
    with torch.no_grad():
        for _ in range(2):
            t0 = time.perf_counter()
            feats_c, feats_f = m.backbone(torch.cat([img0, img1], 0))
            (fc0, fc1), (ff0, ff1) = feats_c.split(1), feats_f.split(1)
            hw_c = tuple(fc0.shape[2:])
            fc0 = m.pos_encoding(fc0).flatten(2).transpose(1, 2)
            fc1 = m.pos_encoding(fc1).flatten(2).transpose(1, 2)
            fc0, fc1 = m.loftr_coarse(fc0, fc1, None, None)
            out = O.coarse_match(fc0, fc1, (H, W_IMG), hw_c, hw_c)
            M = out["b_ids"].numel()
            if M:
                out = O.match_pairs(fc0, fc1, ff0, ff1, (H, W_IMG), hw_c, hw_c)
            best = min(best, time.perf_counter() - t0)
    return 1.0 / best, best, M


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, m = [], 0
    n = args.cpu_sample_pairs
    for it in range(args.warmup + args.steps):
        _, dt, m, cores = cpu_reference_pairs_per_sec(n)
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    v = n / (ms / 1e3)
    sample = f"{n} pairs/step of the 480x640 workload (fp32, torch CPU ops of the reference path, M={m} matches)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.pairs),
        "details": {"pairs_per_step_timed": n, "note": "every step times a bounded sample of the workload's batch on the host cores"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---- blocks for the other configurations of BASELINE.json (device-timed, not part of `value`) ---------------------------

def _timed(fn, reps, dev, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps, out


def stage_pass(d_f0, d_f1, ff0, ff1, hw_c, hw_i, n, impl, ws, dev, k_stage=6):
    """k_stage steps on the current stream with events around the two stages -> (coarse_ms, fine_ms, last result)."""
    from pope_b200 import ops
    hc, wc = hw_c
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(k_stage)]
    res = None
    for k in range(k_stage):
        evs[k][0].record()
        res = ops.coarse_match(d_f0, d_f1, hw_c, hw_c, hw_i[0] / hc, impl=impl, workspace=ws)
        evs[k][1].record()
        m_dev = res["counts"][n:n + 1]
        expec, mk1f = ops.fine_match_maps(ff0, ff1, res["b_ids"], res["i_ids"], res["j_ids"], res["mkpts1_c"], wc, wc,
                                          FINE_STRIDE, (WIN // 2) * (hw_i[0] / ff0.shape[2]), WIN, m_dev)
        evs[k][2].record()
        res.update(mkpts1_f=mk1f, mkpts0_f=res["mkpts0_c"], expec_f=expec)
    torch.cuda.synchronize(dev)
    # the first step of the pass starts on an idle stream: its first event also times the host's launch latency
    coarse_ms = statistics.median(e[0].elapsed_time(e[1]) for e in evs[1:])
    fine_ms = statistics.median(e[1].elapsed_time(e[2]) for e in evs[1:])
    return coarse_ms, fine_ms, res


def robust_block(n, ff0, ff1, impl, dev):
    """configs[1] with realistic dynamic range: token norm 49 -> similarities up to +-135 log2 units."""
    from pope_b200 import _lib, synth
    f0, f1 = synth.coarse_features(4242, n, L, L, C_COARSE, sigma=NORM49_SIGMA, dtype=torch.bfloat16)
    d0, d1 = f0.to(dev), f1.to(dev)
    ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, L, L, C_COARSE, _lib.POPE_BF16), dtype=torch.uint8, device=dev)
    cms, fms, res = stage_pass(d0, d1, ff0, ff1, (HC, WC), (H, W_IMG), n, impl, ws, dev)
    flags = res.flags()
    return {"workload": f"{n} pairs at 480x640, bf16 features of token norm 49 (sigma {NORM49_SIGMA:.2f}), one stream",
            "stage_ms": {"coarse": cms, "fine_gather_match_fused": fms}, "value": n / ((cms + fms) / 1e3), "unit": UNIT,
            "matches": res.total(), "flags": flags, "on_fast_path": not (flags & _lib.FLAG_ROBUST_PATH)}


def in_matcher_figure(n_pairs: int, dev):
    """Steps 3-5 of Matcher.forward (src/matcher/matcher.py:71-79) with the drop-in modules, i.e. WITH the FinePreprocess
    Linears and the fine transformer between coarse and fine matching (SURVEY 8(d) 'in-Matcher' figure), two ways:
      fp32      : CUDA coarse (fp32 features) -> CUDA gather -> torch Linears -> torch fine transformer -> CUDA fine match
      bf16_cuda : Matcher(config, fine_cuda_bf16=True) on bf16 features: tcgen05 coarse -> bf16 gather -> CUDA Linears ->
                  CUDA fine transformer (csrc/fine_tf.cu) -> CUDA fine match"""
    import pope_b200
    from pope_b200 import synth
    hf, wf = HC * FINE_STRIDE, WC * FINE_STRIDE
    shapes = {"hw0_i": torch.Size([H, W_IMG]), "hw1_i": torch.Size([H, W_IMG]), "hw0_c": torch.Size([HC, WC]),
              "hw1_c": torch.Size([HC, WC]), "hw0_f": torch.Size([hf, wf]), "hw1_f": torch.Size([hf, wf]), "bs": n_pairs}
    out = {}
    for name, dtype, reps in (("fp32", torch.float32, 1), ("bf16_cuda", torch.bfloat16, 5)):
        torch.manual_seed(0)
        m = pope_b200.Matcher(pope_b200.make_default_cfg(), fine_cuda_bf16=(dtype == torch.bfloat16)).eval().to(dev)
        f0, f1 = synth.coarse_features(99, n_pairs, L, L, C_COARSE, dtype=dtype)
        g = torch.Generator(device=dev).manual_seed(98)
        ff0 = torch.randn(n_pairs, hf, wf, C_FINE, device=dev, generator=g).to(dtype).permute(0, 3, 1, 2)
        ff1 = torch.randn(n_pairs, hf, wf, C_FINE, device=dev, generator=g).to(dtype).permute(0, 3, 1, 2)
        f0, f1 = f0.to(dev), f1.to(dev)

        def run():
            data = dict(shapes)
            with torch.no_grad():
                m.coarse_matching(f0, f1, data)
                w0, w1 = m.fine_preprocess(ff0, ff1, f0, f1, data)
                if w0.size(0):
                    w0, w1 = m.loftr_fine(w0, w1)
                m.fine_matching(w0, w1, data)
            return data

        ms, data = _timed(run, reps, dev, warm=2 if dtype == torch.bfloat16 else 1)
        out[name] = {"value": n_pairs / (ms / 1e3), "unit": UNIT, "pairs": n_pairs, "ms": ms,
                     "matches": int(data["mconf"].numel())}
        del m, f0, f1, ff0, ff1, data
        torch.cuda.empty_cache()
    out["note"] = ("steps 3-5 of Matcher.forward incl. FinePreprocess Linears + fine transformer; the module flow has one host "
                   "sync per call (the match count), like the reference's torch.where")
    return out


def single_pair_block(impl, dev):
    """BASELINE configs[0]'s shape on the GPU: ONE 480x640 pair per call, the way the reference's evaluation loop calls the
    Matcher.  Latency of the hot path for that call, eager (ctypes launches from Python) and replayed from a CUDA graph (the
    step has no host synchronisation, so it can be captured: tests/test_gpu_parity.py::test_hot_path_step_is_graph_capturable)."""
    from pope_b200 import _lib, ops, synth
    f0, f1 = synth.coarse_features(555, 1, L, L, C_COARSE, dtype=torch.bfloat16)
    d0, d1 = f0.to(dev), f1.to(dev)
    g = torch.Generator(device=dev).manual_seed(556)
    ff0 = torch.randn(1, HC * FINE_STRIDE, WC * FINE_STRIDE, C_FINE, device=dev, generator=g).to(torch.bfloat16).permute(0, 3, 1, 2)
    ff1 = torch.randn(1, HC * FINE_STRIDE, WC * FINE_STRIDE, C_FINE, device=dev, generator=g).to(torch.bfloat16).permute(0, 3, 1, 2)
    ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(1, L, L, C_COARSE, _lib.POPE_BF16), dtype=torch.uint8, device=dev)

    def step():
        return ops.match_pairs_device(d0, d1, ff0, ff1, (H, W_IMG), (HC, WC), (HC, WC), impl=impl, workspace=ws)

    ms, res = _timed(step, 50, dev, warm=3)
    out = {"workload": "1 pair at 480x640 per call (BASELINE configs[0]'s shape), bf16, inputs resident",
           "eager": {"us_per_pair": ms * 1e3, "value": 1e3 / ms, "unit": UNIT}, "matches": res.total(), "flags": res.flags()}
    try:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            gres = step()
        gms, _ = _timed(graph.replay, 50, dev, warm=3)
        out["graph"] = {"us_per_pair": gms * 1e3, "value": 1e3 / gms, "unit": UNIT, "matches": gres.total()}
    except Exception as e:
        out["graph"] = {"error": repr(e)[:200]}
    return out


def highres_block(n, impl, dev):
    """BASELINE configs[3]: 960x1280 pairs, 19 200 coarse tokens per image (the L x S matrix would be 1.47 GB per pair)."""
    from pope_b200 import _lib, synth
    hc, wc = 120, 160
    Lh = hc * wc
    f0, f1 = synth.coarse_features(777, n, Lh, Lh, C_COARSE, dtype=torch.bfloat16)
    d0, d1 = f0.to(dev), f1.to(dev)
    g = torch.Generator(device=dev).manual_seed(778)
    ff0 = torch.randn(n, hc * 4, wc * 4, C_FINE, device=dev, generator=g).to(torch.bfloat16).permute(0, 3, 1, 2)
    ff1 = torch.randn(n, hc * 4, wc * 4, C_FINE, device=dev, generator=g).to(torch.bfloat16).permute(0, 3, 1, 2)
    ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, Lh, Lh, C_COARSE, _lib.POPE_BF16), dtype=torch.uint8, device=dev)
    cms, fms, res = stage_pass(d0, d1, ff0, ff1, (hc, wc), (960, 1280), n, impl, ws, dev, k_stage=4)
    _, tf_burst, tf_sus, _ = measured_peaks()
    ach = n * 2.0 * Lh * Lh * C_COARSE / (cms / 1e3) / 1e12
    return {"workload": f"{n} pairs at 960x1280 (coarse 120x160 = 19200 tokens per image, BASELINE configs[3]), bf16, one stream",
            "stage_ms": {"coarse": cms, "fine_gather_match_fused": fms}, "value": n / ((cms + fms) / 1e3), "unit": UNIT,
            "coarse_tflops_algorithmic": ach, "coarse_frac_of_burst_peak": ach / tf_burst,
            "coarse_frac_of_sustained_peak": ach / tf_sus, "matches": res.total(), "flags": res.flags()}


def retrieval_block(dev):
    """BASELINE configs[2]: 1 query vs 256 reference crops at 224x224 (eval_linemod_json.py:72-101).  Kernel only (CLS
    tokens, D = 384, and the patch-token stress shape D = 256 * 384) and end to end with the batched ViT-S/14 forwards
    (random-init weights, bf16) instead of 257 batch-1 forwards with a host sync after each."""
    from pope_b200 import ops, retrieval, synth
    out = {"workload": "1 query vs 256 crops at 224x224, DINOv2 ViT-S/14 tokens (BASELINE configs[2])"}
    for name, D, dt in (("cls_d384_f32", 384, torch.float32), ("patch_d98304_bf16", 256 * 384, torch.bfloat16)):
        q, refs = synth.retrieval_tokens(5, 256, D, dtype=dt)
        q, refs = q.to(dev), refs.to(dev)
        ms, r = _timed(lambda: ops.cosine_topk(q, refs, 3), 20, dev, warm=3)
        byts = 257 * D * q.element_size()
        out[name] = {"us_per_query": ms * 1e3, "gbs": byts / (ms / 1e3) / 1e9, "top3": r[2].tolist()}
        try:        # the same call replayed from a CUDA graph: what the kernels take without the Python / launch overhead
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                ops.cosine_topk(q, refs, 3)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    keep = ops.cosine_topk(q, refs, 3)
            torch.cuda.current_stream(dev).wait_stream(side)
            gms, _ = _timed(graph.replay, 50, dev, warm=3)
            out[name].update(us_per_query_graph=gms * 1e3, gbs_graph=byts / (gms / 1e3) / 1e9, top3_graph=keep[2].tolist())
        except Exception as e:
            out[name]["graph_error"] = repr(e)[:200]
    try:
        from pope_b200.dino_vit import DinoViT
        torch.manual_seed(3)
        vit = DinoViT(init_values=1.0).eval().to(dev).to(torch.bfloat16)
        g = torch.Generator(device=dev).manual_seed(11)
        ref = torch.randn(1, 3, 224, 224, device=dev, generator=g).to(torch.bfloat16)
        crops = torch.randn(256, 3, 224, 224, device=dev, generator=g).to(torch.bfloat16)
        with torch.no_grad():
            ms, r = _timed(lambda: retrieval.retrieve_topk_images(vit, ref, crops, 3), 3, dev, warm=2)
        out["with_vit_bf16"] = {"ms_per_query": ms, "queries_per_s": 1e3 / ms, "top3": list(r[2]),
                                "note": "3 batched forwards (128 + 128 + 1 images) + cosine/top-k kernel; stock PyTorch ViT"}
    except Exception as e:      # the block is informative; the headline does not depend on it
        out["with_vit_bf16"] = {"error": repr(e)[:200]}
    return out


def h2d_ceiling(dev, world, dist):
    """Plain pinned cudaMemcpyAsync host->device from every rank at the same time: the box's ceiling for the e2e path."""
    nbytes = 1 << 30
    src = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        dst.copy_(src, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(dev)
    gbs = 3 * nbytes / (e0.elapsed_time(e1) / 1e3) / 1e9
    t = torch.tensor([gbs], device=dev)
    if world > 1:
        lo = t.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return {"per_rank_min_gbs": float(lo.item()), "aggregate_gbs": float(t.item())}
    return {"per_rank_min_gbs": gbs, "aggregate_gbs": gbs}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from pope_b200 import _lib, driver, ops, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path to fall back to)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    impl = {"auto": _lib.COARSE_AUTO, "simt": _lib.COARSE_SIMT, "tcgen05": _lib.COARSE_TCGEN05}[args.coarse_impl]
    n = args.pairs
    esize = 2 if dtype == torch.bfloat16 else 4
    std_workload = n == 64 and dtype == torch.bfloat16

    # ---- synthetic inputs (seeded per rank: every rank owns different pairs) --------------------------------------
    f0, f1 = synth.coarse_features(1234 + rank, n, L, L, C_COARSE, dtype=dtype)
    g = torch.Generator(device=dev).manual_seed(4321 + rank)
    hf, wf = HC * FINE_STRIDE, WC * FINE_STRIDE
    ff0 = torch.randn(n, hf, wf, C_FINE, device=dev, generator=g).to(dtype).permute(0, 3, 1, 2)   # channels-last
    ff1 = torch.randn(n, hf, wf, C_FINE, device=dev, generator=g).to(dtype).permute(0, 3, 1, 2)
    d_f0, d_f1 = f0.to(dev), f1.to(dev)
    # the job's record buffer (and, on rank 0, the receive buffer of the gather) exists before anything is timed: sized
    # for the longest job of this run
    job_steps = -(-args.job_pairs // (n * world)) if (args.job_pairs > 0 and not args.no_extra) else 0
    max_steps = max(args.steps, args.warmup, 3, job_steps)
    job = driver.JobGather(max_steps, n * L, dev, rank=rank, world=world, compact=True)
    n_streams = max(1, args.streams)
    runner = driver.DeviceBatchRunner(dev, n_streams)      # the public form of "consecutive batches on alternating streams"
    ws_stage = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, L, L, C_COARSE, _lib.dtype_code(d_f0)), dtype=torch.uint8,
                           device=dev)

    def add_to_job(res):                   # JobGather.add orders appends from different streams by itself
        job.add(res, rank * n)

    def step_device():
        res, _ = runner.submit(d_f0, d_f1, ff0, ff1, (H, W_IMG), (HC, WC), (HC, WC), impl=impl,
                               after=add_to_job if world > 1 else None)
        return res

    def finish_job():
        runner.join()
        return job.finish() if world > 1 else (None, None)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def run_job(steps):
        """`steps` device-resident steps + the job's single gather, device-timed -> (ms max over ranks, records, sizes, my
        checksum, the last step's result)"""
        barrier()
        t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_beg.record()
        runner.fork()
        for _ in range(steps):
            last = step_device()
        runner.join()
        my_sum = None
        if world > 1:
            my_total = job.total.clone()                # device copies: read after the timed region
            recs, sizes = job.finish()
        else:
            recs, sizes, my_total = None, None, None
        t_end.record()
        barrier()
        ms = t_beg.elapsed_time(t_end)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            my_sum = job.checksum(totals=int(my_total.item()))
        return float(t.item()), recs, sizes, my_sum, last

    def verify_gather(recs, sizes, my_sum, steps, m_step):
        """rank 0 holds every rank's live records: sizes = steps x matches per step of each rank (every rank runs the same
        seeded batch `steps` times), and the word checksum of what arrived equals the one each rank took of its own buffer"""
        sums = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(sums, my_sum)
        m_all = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(m_all, torch.tensor([m_step], dtype=torch.int64, device=dev))
        if rank != 0:
            return None
        ok = [int(s) for s in sizes] == [steps * int(m) for m in m_all.tolist()]
        ok = ok and torch.equal(job.checksum(recs, sizes), sums)
        first = driver.unpack_records(recs[world - 1, :8], WC, 8.0)         # spot check: decodable, belongs to the last rank
        ok = ok and bool((first["b_ids"] >= (world - 1) * n).all()) and bool((first["mconf"] > 0.2).all())
        return bool(ok)

    clk = ClockSampler(local)
    clk.wait_first()
    run_job(max(args.warmup, 3))                         # warm-up: same code path as the timed region, gather included
    wall0 = time.time()
    total_ms, recs, sizes, my_sum, last = run_job(args.steps)
    wall1 = time.time()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    ms_per_step = total_ms / args.steps
    value = world * n * args.steps / (total_ms / 1e3)

    # per-stage durations for the rooflines: a few extra steps on ONE stream (with several streams the stages of
    # consecutive steps overlap, so events around them would time the queue, not the kernels); not part of `value`
    coarse_ms, fine_ms, res = stage_pass(d_f0, d_f1, ff0, ff1, (HC, WC), (H, W_IMG), n, impl, ws_stage, dev,
                                         k_stage=max(4, min(args.steps, 6)))
    M = res.total()
    flags = res.flags()
    gather_verified = verify_gather(recs, sizes, my_sum, args.steps, M) if world > 1 else None
    gather_bytes = (sum(sizes) - sizes[0]) * 4 * job.words if (world > 1 and rank == 0) else 0

    # ---- the 4096-pair job of configs[4]: sharded over the ranks, one gather at the end ------------------------------
    job_block = None
    if job_steps > 0:
        jms, jrecs, jsizes, jsum, _ = run_job(job_steps)
        jver = verify_gather(jrecs, jsizes, jsum, job_steps, M) if world > 1 else None
        job_block = {"workload": f"{job_steps * n * world} synthetic pairs at 480x640 sharded over {world} GPU(s) in steps of {n} "
                                 f"pairs, one gather of the match lists at the end (BASELINE configs[4])",
                     "steps_per_gpu": job_steps, "ms": jms, "value": job_steps * n * world / (jms / 1e3), "unit": UNIT,
                     "gather_verified": jver}

    # ---- end to end through the C-ABI host entry (pinned host buffers, copies inside the timed region) -------------
    e2e = None
    if not args.no_e2e:
        chunk = min(16, n)
        pl = driver.Pipeline(dtype, chunk, (H, W_IMG), (HC, WC), (HC, WC), C_COARSE, C_FINE, FINE_STRIDE, WIN, impl=impl,
                             device=local)
        prev_aff = driver.bind_host_to_gpu(local)        # page-locked staging buffers on the GPU's NUMA node
        h_f0, h_f1 = f0.pin_memory(), f1.pin_memory()
        h_ff0 = ff0.permute(0, 2, 3, 1).contiguous().cpu().pin_memory()
        h_ff1 = ff1.permute(0, 2, 3, 1).contiguous().cpu().pin_memory()
        out = pl.alloc_outputs(n)
        if prev_aff is not None:
            os.sched_setaffinity(0, prev_aff)
        def time_e2e(k, warm):
            for _ in range(warm):
                pl.run(h_f0, h_f1, h_ff0, h_ff1, out)
            barrier()
            t0 = time.perf_counter()
            for _ in range(k):
                pl.run(h_f0, h_f1, h_ff0, h_ff1, out)       # returns after the results are in host memory
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        k_e2e = max(3, min(args.steps, 5))
        dt = time_e2e(k_e2e, 2)
        h2d = pl.last_h2d_bytes      # bulk copies + what crosses the link from pinned memory on demand (image 0's centre
                                     # pixels, image 1's windows: in place or as their union, see `f1_mode`)
        d2h = sum(out[k].numel() * out[k].element_size() for k in ("i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f", "counts")) + 4 * ((n + chunk - 1) // chunk)
        e2e = {"value": world * n * k_e2e / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": k_e2e, "ms_per_step": 1e3 * dt / k_e2e, "matches": int(out["counts"].sum()),
               "h2d_gbs_per_rank": h2d * k_e2e / dt / 1e9, "f1_mode": pl.last_f1_mode,
               "api": "pope_pipeline_run (C ABI, pinned host buffers, chunk=%d pairs)" % chunk,
               "note": "coarse features are copied; of the fine maps only the matched cells' pixels cross the link (image 0: "
                       "centre pixels read in place by the fine kernel; image 1: `f1_mode`), which is why the achieved rate "
                       "sits below the bulk-copy ceiling"}
        # the three ways image 1's fine map can reach the device, same buffers, same box (POPE_PIPELINE_F1)
        by_mode = {}
        for mode in ("windows", "union", "bulk"):
            os.environ["POPE_PIPELINE_F1"] = mode
            try:
                dtm = time_e2e(3, 1)
                by_mode[mode] = {"value": world * n * 3 / dtm, "h2d_bytes_per_step": pl.last_h2d_bytes,
                                 "h2d_gbs_per_rank": pl.last_h2d_bytes * 3 / dtm / 1e9}
                assert pl.last_f1_mode == mode and int(out["counts"].sum()) == M
            finally:
                del os.environ["POPE_PIPELINE_F1"]
        e2e["by_f1_mode"] = by_mode
        assert int(out["counts"].sum()) == M, (int(out["counts"].sum()), M)
        pl.close()
        del h_f0, h_f1, h_ff0, h_ff1
        e2e["h2d_ceiling"] = dict(h2d_ceiling(dev, world, dist), how="pinned cudaMemcpyAsync of 1 GiB x 3 from every rank at once")
        e2e["frac_of_h2d_ceiling"] = e2e["h2d_gbs_per_rank"] / e2e["h2d_ceiling"]["per_rank_min_gbs"]

    clk.stop()
    clocks = clk.summary(wall0, wall1)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm, tf_burst, tf_sus, peak_src = measured_peaks()
    coarse_traffic, fine_traffic, traffic_src = dram_traffic_from_profiles() if std_workload else (None, None, None)
    flops = n * 2.0 * L * L * C_COARSE
    ach = flops / (coarse_ms / 1e3) / 1e12
    fine_bytes = M * ((1 + 25) * C_FINE * esize + 3 * 8 + 8 + 12 + 8)     # 26 feature rows + ids + coords in/out
    tc = impl == _lib.COARSE_TCGEN05 or (impl == _lib.COARSE_AUTO and _lib.tcgen05_available())   # fp32: split path
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": workload_config(n),
        "details": {"coarse_impl": ("tcgen05" if dtype == torch.bfloat16 else "tcgen05 on a three-way bf16 split of the fp32 features") if tc else "simt-fp32fma",
                    "fine_map_layout": "channels_last", "streams": n_streams, "matches_per_step": M, "flags": flags,
                    "gather": ("one NCCL gather of the job's live 20-byte match records to rank 0 after the K steps (inside the "
                               "timed region; receive buffer preallocated)") if world > 1 else "none"},
        "clocks": clocks,
        "stage_ms": {"coarse": coarse_ms, "fine_gather_match_fused": fine_ms},
        "one_stream": {"value": n / ((coarse_ms + fine_ms) / 1e3), "unit": UNIT, "ms_per_step": coarse_ms + fine_ms,
                       "note": "coarse + fine on a single stream (a single Matcher.forward-style caller)"},
        "roofline": {"kernel": "coarse stage (tcgen05 single sweep with lazily shifted exponentials: row sums + shuffle-reduced column sums + candidate lists; column log-sum-exp merge, list evaluation, compaction)" if tc else
                               "coarse stage (fp32-FMA sweeps + compaction)", "bound": "tensor",
                     "achieved": ach, "peak": tf_burst, "unit": "TFLOP/s", "frac": ach / tf_burst,
                     "peak_sustained": tf_sus, "frac_of_sustained": ach / tf_sus, "traffic": coarse_traffic,
                     "traffic_source": traffic_src,
                     "peak_source": f"{peak_src} bf16_tflops (burst: the timed region lasts ~{total_ms:.0f} ms at full clocks)",
                     "algorithmic_flops_per_launch": flops},
        "roofline_fine": {"kernel": "fine_match_maps_kernel (fused 5x5 window gather + correlation + softmax expectation)",
                          "bound": "hbm", "achieved": fine_bytes / (fine_ms / 1e3) / 1e9, "peak": hbm, "unit": "GB/s",
                          "frac": fine_bytes / (fine_ms / 1e3) / 1e9 / hbm, "traffic": fine_traffic,
                          "dram_gbs": (fine_traffic / (fine_ms / 1e3) / 1e9) if fine_traffic else None,
                          "dram_frac": (fine_traffic / (fine_ms / 1e3) / 1e9 / hbm) if fine_traffic else None,
                          "traffic_source": traffic_src,
                          "note": "frac counts algorithmic bytes (5x5 windows at stride 4 overlap; the overlap is served by L2), "
                                  "dram_frac the DRAM bytes of the ncu capture",
                          "algorithmic_bytes_per_launch": fine_bytes},
        "gpu_launches": args.steps * (_lib.KERNELS_PER_STEP[("tcgen05" if dtype == torch.bfloat16 else "tcgen05_f32") if tc else "simt"]
                                      + (1 if (tc and dtype == torch.bfloat16 and _lib.single_sweep_is_split(n, L)) else 0)
                                      + (1 if world > 1 else 0)),
    }
    if world > 1:
        line["gather_verified"] = gather_verified
        line["gather_bytes_received_rank0"] = gather_bytes
    if job_block:
        line["job_4096"] = job_block
    if not args.no_extra:
        for name, fn in (("robust", lambda: robust_block(n, ff0, ff1, impl, dev)),
                         ("in_matcher", (lambda: in_matcher_figure(args.in_matcher, dev)) if args.in_matcher > 0 else None),
                         ("highres", (lambda: highres_block(args.highres_pairs, impl, dev)) if args.highres_pairs > 0 else None),
                         ("single_pair", lambda: single_pair_block(impl, dev)),
                         ("retrieval", lambda: retrieval_block(dev))):
            if fn is None:
                continue
            try:
                line[name] = fn()
            except Exception as e:                   # an extra block must not take the headline down with it
                line[name] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
    if e2e:
        line["e2e"] = e2e
    if not args.no_cpu:
        v, dt, m_cpu, cores = cpu_reference_pairs_per_sec(args.cpu_sample_pairs)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{args.cpu_sample_pairs} pairs of the same 480x640 workload, fp32 torch CPU "
                                          f"(oracle port of the reference op sequence), {dt:.2f} s, M={m_cpu}"}
        try:
            vf, dtf, mf = cpu_full_matcher_pairs_per_sec()
            line["cpu_baseline"]["full_matcher"] = {
                "value": vf, "unit": UNIT, "cores": cores,
                "sample": f"1 image pair [1,1,480,640] through backbone + coarse transformer (torch modules on the CPU) + the "
                          f"oracle port of coarse matching, random-init weights, best of 2: {dtf:.2f} s, M={mf} "
                          f"(BASELINE.md 4.1 leg (i); M = 0 with random weights, so the fine level does not run)"}
        except Exception as e:
            line["cpu_baseline"]["full_matcher"] = {"error": repr(e)[:300]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
