"""Host-side logic that needs no GPU: drop-in surface, state-dict layout, C-ABI loading and argument checking."""
import ctypes as C
import json
import os
import re

import pytest
import torch

import pope_b200
from pope_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def layout(golden_dir):
    with open(os.path.join(golden_dir, "matcher_layout.json")) as f:
        return json.load(f)


def test_default_cfg_equals_reference(layout):
    assert json.loads(json.dumps(pope_b200.default_cfg)) == layout["default_cfg"]


def test_state_dict_layout_equals_reference(layout):
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    sd = m.state_dict()
    assert list(sd.keys()) == list(layout["state_dict"].keys())
    assert {k: list(v.shape) for k, v in sd.items()} == layout["state_dict"]
    assert sum(p.numel() for p in m.parameters()) == layout["n_params"]
    for name in ("backbone", "pos_encoding", "loftr_coarse", "coarse_matching", "fine_preprocess", "loftr_fine",
                 "fine_matching"):
        assert hasattr(m, name)


def test_load_state_dict_strips_matcher_prefix():
    a = pope_b200.Matcher(pope_b200.make_default_cfg())
    b = pope_b200.Matcher(pope_b200.make_default_cfg())
    sd = {"matcher." + k: v for k, v in a.state_dict().items()}
    res = b.load_state_dict(sd, strict=False)
    assert not res.missing_keys and not res.unexpected_keys
    assert all(torch.equal(v, b.state_dict()[k]) for k, v in a.state_dict().items())


def test_matcher_constructor_does_not_mutate_config():
    cfg = pope_b200.make_default_cfg()
    before = json.dumps(cfg, sort_keys=True)
    pope_b200.Matcher(cfg)
    assert json.dumps(cfg, sort_keys=True) == before


def test_hot_path_has_no_cpu_fallback():
    cm = pope_b200.CoarseMatching(pope_b200.default_cfg["match_coarse"]).eval()
    data = {"hw0_i": (64, 64), "hw0_c": (8, 8), "hw1_c": (8, 8)}
    with pytest.raises(_lib.PopeError):
        cm(torch.randn(1, 64, 256), torch.randn(1, 64, 256), data)           # CPU tensors are rejected
    with pytest.raises(_lib.PopeError):
        pope_b200.FineMatching().eval()(torch.randn(4, 25, 128), torch.randn(4, 25, 128),
                                        {"hw0_i": (64, 64), "hw0_f": (32, 32), "mconf": torch.ones(4),
                                         "mkpts0_c": torch.zeros(4, 2), "mkpts1_c": torch.zeros(4, 2)})
    with pytest.raises(_lib.PopeError):                                       # the padded-batch route is CUDA-only as well
        cm(torch.randn(1, 64, 256), torch.randn(1, 64, 256), data, mask_c0=torch.ones(1, 64), mask_c1=torch.ones(1, 64))
    with pytest.raises(NotImplementedError):                                  # the training-time sampling branch is not built
        cm.train()(torch.randn(1, 64, 256), torch.randn(1, 64, 256), data)


def test_product_package_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "pope_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "ref_shim" not in src, f


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "pope_b200.h")).read()
    declared = set(re.findall(r"\b(pope_[a-z_0-9]+)\s*\(", header))
    declared -= {"pope_pipeline"}        # the opaque struct tag
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    h = _lib.lib()                        # raises if the .so is missing or lacks a symbol
    for name in declared:
        assert getattr(h, name) is not None
    assert h.pope_abi_version() == 1
    assert h.pope_status_string(0) == b"ok"


def test_argument_errors_are_reported_before_touching_the_gpu():
    h = _lib.lib()
    assert h.pope_coarse_workspace_bytes(0, 10, 10) == 0
    need = h.pope_coarse_workspace_bytes(2, 4800, 4800)
    assert need >= 2 * 4800 * (8 + 8 + 4 + 4 + 4 + 8 * 8 + 4)
    # null pointers / bad sizes / bad dtype: negative status, no CUDA call is made
    args_ok = [1, 1, 0, 1, 64, 64, 256, 8, 8, 8, 8, 8.0, 0.1, 0.2, 2, 0, 1, need, 1, 1, 1, 1, 1, 1, 1, 64, None]
    bad = list(args_ok); bad[0] = None
    assert h.pope_coarse_match(*bad) == -1
    bad = list(args_ok); bad[2] = 7
    assert h.pope_coarse_match(*bad) == -2
    bad = list(args_ok); bad[6] = 250
    assert h.pope_coarse_match(*bad) == -4
    bad = list(args_ok); bad[7] = 9           # h0c*w0c != L
    assert h.pope_coarse_match(*bad) == -1
    assert h.pope_fine_match(None, None, 0, 4, None, 25, 64, None, 4.0, None, None, None) == -4
    assert h.pope_fine_match(None, None, 0, 0, None, 25, 128, None, 4.0, None, None, None) == 0     # M == 0 is a no-op
    assert h.pope_cosine_topk(None, None, 0, 4, 4, 3, 1e-8, None, None, None, None) == -1
    assert b"workspace" in h.pope_status_string(-3)


def test_header_is_plain_c_and_a_c_program_links(tmp_path):
    """The boundary is a C ABI: include/pope_b200.h must compile as C99 (no C++ in the declarations) and a C program must
    link against the library and call it without any Python or torch in the process."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    src = tmp_path / "c_abi.c"
    src.write_text('#include <stdio.h>\n#include "pope_b200.h"\n'
                   'int main(void) {\n'
                   '  if (pope_abi_version() != 1) return 1;\n'
                   '  if (pope_coarse_workspace_bytes(0, 1, 1) != 0) return 2;\n'
                   '  if (pope_coarse_match(0, 0, 0, 1, 64, 64, 256, 8, 8, 8, 8, 8.0f, 0.1f, 0.2f, 2, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 64, 0) >= 0) return 3;\n'
                   '  puts(pope_status_string(-3));\n  return 0;\n}\n')
    exe = tmp_path / "c_abi"
    libdir = os.path.join(ROOT, "pope_b200")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-lpope_b200", "-Wl,-rpath," + libdir, "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    assert "workspace" in out


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the reference's CPU path = the oracle port, rank 0 only): one JSON line with the contract's
    keys, and the SAME `config` the CUDA arm prints for the same workload (the arm-specific facts sit in `details`)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample-pairs", "1"], capture_output=True, text=True, timeout=600, check=True).stdout
    line = json.loads(out.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sys.path.insert(0, root)
    import bench
    assert line["config"] == bench.workload_config(64) and line["metric"] == bench.METRIC and line["unit"] == bench.UNIT


def test_single_sweep_split_rule():
    """The Python mirror of coarse_tc_run's head / tail rule (used for bench.py's launch count): 64 pairs at 480x640 are 1 216
    units = 16 rounds of 74 CTA pairs + 32, so 62 + 2 pairs; 16 pairs at 960x1280 (1 200 units) would need a round more when cut
    at a pair boundary; one pair, or a unit count that fills its rounds, is never cut."""
    assert _lib.single_sweep_is_split(64, 4800) and _lib.single_sweep_is_split(32, 4800)
    assert not _lib.single_sweep_is_split(16, 19200)
    assert not _lib.single_sweep_is_split(1, 4800)
    assert not _lib.single_sweep_is_split(74, 256)          # 74 units: exactly one round
    assert not _lib.single_sweep_is_split(3, 4800)          # 57 units: fewer than one round


def test_bench_reads_the_committed_ncu_table(tmp_path, monkeypatch):
    """bench.py takes `roofline.traffic` from the committed ncu table (tools/ncu_extract.py format): the committed file must
    parse to plausible per-launch DRAM bytes, and a file in another format (ncu's raw page) must give None, not an exception
    that takes the headline line down."""
    import bench
    coarse, fine, src = bench.dram_traffic_from_profiles()
    assert src == "profiles/r2_ncu_step.csv"
    assert 3e8 < coarse < 2e9 and 5e8 < fine < 2e9
    raw = tmp_path / "raw.csv"
    raw.write_text('"ID","Process ID","Kernel Name","dram__bytes_read.sum","dram__bytes_write.sum"\n'
                   '"","","","Mbyte","Mbyte"\n"0","1","sweep_tc_kernel","310.9","168.7"\n')
    monkeypatch.setattr(bench, "TRAFFIC_CSV", str(raw))
    assert bench.dram_traffic_from_profiles() == (None, None, None)
    monkeypatch.setattr(bench, "TRAFFIC_CSV", str(tmp_path / "absent.csv"))
    assert bench.dram_traffic_from_profiles() == (None, None, None)


def test_bench_dump_outputs_writes_the_live_rows(tmp_path):
    """`bench.py --dump-outputs`: the rows up to the live count of a capacity-sized result, ids exact in float64, the rest
    float32; over the byte budget, the same seeded sample of rows on every call, within the budget."""
    import numpy as np
    import bench
    from pope_b200 import ops
    cap, n, m = 1000, 3, 700
    g = torch.Generator().manual_seed(0)
    res = ops.CoarseResult(n_pairs=n, counts=torch.tensor([300, 0, 400, m, 0], dtype=torch.int32))
    for k in ("b_ids", "i_ids", "j_ids"):
        res[k] = torch.randint(0, 4800, (cap,), generator=g) + (1 << 40)
    for k, w in (("mconf", 0), ("mkpts0_c", 2), ("mkpts1_c", 2), ("expec_f", 3), ("mkpts1_f", 2)):
        res[k] = torch.randn((cap, w) if w else (cap,), generator=g)
    res["mkpts0_f"] = res["mkpts0_c"]
    names = bench.dump_outputs(str(tmp_path / "all"), res)
    assert names == sorted(bench.DUMP_KEYS + ("counts",))
    for k in bench.DUMP_KEYS:
        a = np.load(tmp_path / "all" / f"{k}.npy")
        assert a.dtype == (np.float64 if k.endswith("_ids") else np.float32) and a.shape[0] == m, k
        assert np.array_equal(a, res[k][:m].numpy().astype(a.dtype)), k
    assert np.load(tmp_path / "all" / "counts.npy").tolist() == [300, 0, 400, m, 0]
    budget = 20_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res, max_bytes=budget)
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert 0 < rows.size < m and np.all(np.diff(rows) > 0) and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "i_ids.npy"), res["i_ids"][rows.astype(np.int64)].numpy().astype(np.float64))
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= budget


def test_union_fetch_cover_rule():
    """The host pipeline's union fetch (csrc/pipeline.cu::fetch_union_kernel) copies a fine-map pixel iff it lies in the WxW
    window (stride `stride`, zero padding W//2: fine_preprocess.py:40-43) of at least one matched coarse cell.  The kernel
    finds the covering cells of pixel (y, x) as cy in [ceil((y - half) / stride), floor((y + half) / stride)] clipped to the
    grid (same for x); this is that rule's Python mirror against windows painted cell by cell."""
    import numpy as np
    rng = np.random.default_rng(3)
    for stride in (1, 2, 3, 4, 5, 8):
        half, hc, wc = 2, 7, 9
        hf, wf = hc * stride, wc * stride
        marked = rng.random((hc, wc)) < 0.4
        want = np.zeros((hf, wf), dtype=bool)
        for cy, cx in zip(*np.nonzero(marked)):
            want[max(0, cy * stride - half):cy * stride + half + 1, max(0, cx * stride - half):cx * stride + half + 1] = True
        got = np.zeros_like(want)
        for y in range(hf):
            for x in range(wf):
                cy_lo = (y - half + stride - 1) // stride if y > half else 0
                cx_lo = (x - half + stride - 1) // stride if x > half else 0
                cy_hi, cx_hi = min((y + half) // stride, hc - 1), min((x + half) // stride, wc - 1)
                got[y, x] = marked[cy_lo:cy_hi + 1, cx_lo:cx_hi + 1].any()
        assert np.array_equal(got, want), stride
