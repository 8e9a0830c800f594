"""Every coarse sweep path held to a float64 reference with an error bound derived from the inputs.

The paths: the tcgen05 single sweep (bf16, thr > 0.15), its two-sweep online-softmax form (POPE_TC_DEBUG=16, ungated), the
three sweeps (thr <= 0.15), the fp32 features' single sweep through the three-way bf16 split, and the SIMT fp32-FMA kernels;
at every width the tensor cores take (C = 64 ... 256, one to four 64-wide k-chunks) and at widths they do not.

For every case the reference is built on the CPU in float64 from exactly the values the kernel reads, and every row's and
column's log-sum-exp (read from the scratch through `ops.scratch_views`), every confidence and every match list is checked
against it.  The bound (see `_bounds`) is not a tuned tolerance: at the benchmark shape it is below log2(1.001) = 1.44e-3
log2 units (`test_bound_catches_a_tenth_of_a_percent_at_the_benchmark_shape`), so a kernel that loses 0.1 % of any row or
column sum fails.  Set POPE_BOUND_REPORT=<file.json> to write the largest error / bound ratio of every case."""
from __future__ import annotations

import collections
import json
import math
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import pope_oracle as O
from oracle.gen_golden import COARSE_CASES, coarse_inputs
from pope_b200 import _lib, ops, synth
from tests.parity_utils import assert_sorted_by_pair_and_row, compare_match_lists

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda:0")
LN2 = math.log(2.0)
U = 2.0 ** -24                  # fp32 unit roundoff
ACC_C = 2.0                     # tensor-core fp32 accumulation may truncate instead of rounding: twice the rounding bound
SPLIT_RESIDUAL = 4.1 * U        # fp32 split path: a b minus its six kept bf16 products is below 4.1 u |a| |b| (a3 b2, a2 b3,
                                # a3 b3 and the residuals of a and b after three bf16 terms, each about u |a| |b|)
SINGLE, TWO, THREE, SIMT, SPLIT = "single", "two_sweeps", "three_sweeps", "simt", "split"
GRID_SHAPES = [(1, 1), (1, 300), (300, 1), (31, 33), (127, 129), (255, 257), (256, 256), (4800, 37), (37, 4800)]
RATIOS = collections.OrderedDict()      # test id -> largest error / bound of the log-sum-exps and of mconf


@pytest.fixture(scope="module", autouse=True)
def _bound_report():
    yield
    path = os.environ.get("POPE_BOUND_REPORT")
    if path and RATIOS:
        with open(path, "w") as f:
            json.dump(RATIOS, f, indent=1)


# ---- float64 reference -------------------------------------------------------------------------------------------------
def reference(f0: torch.Tensor, f1: torch.Tensor, temperature: float = 0.1, with_bound: bool = True) -> dict:
    """x = f0 f1^T log2(e) / (C T) and its base-2 row / column log-sum-exps in float64 from the values the kernel reads
    (bf16-rounded for bf16 runs), plus |f0| |f1|^T, from which `_bounds` derives the error bound."""
    a, b = f0.double(), f1.double()
    Cc = a.shape[2]
    scale = 1.0 / (LN2 * Cc * temperature)
    x = torch.einsum("nlc,nsc->nls", a, b) * scale
    ref = dict(x=x, scale=scale, C=Cc, lse_r=torch.logsumexp(x * LN2, 2) / LN2, lse_c=torch.logsumexp(x * LN2, 1) / LN2)
    if with_bound:
        ref["absab"] = torch.einsum("nlc,nsc->nls", a.abs(), b.abs())
    return ref


def conf_of(ref: dict) -> torch.Tensor:
    return torch.exp2(2.0 * ref["x"] - ref["lse_r"][:, :, None] - ref["lse_c"][:, None, :])


def _bounds(ref: dict, split: bool):
    """Per cell: dx = scale (c C u + split residual) sum_k |a_ik b_jk|.  Per row: dlse_r = max_j dx + (S u + 2^-21) / ln 2
    (the S-term fp32 sum, and ex2 / lg2.approx); the mirror bound per column."""
    n, L, S = ref["x"].shape
    dx = ref["absab"] * (ref["scale"] * (ACC_C * ref["C"] * U + (SPLIT_RESIDUAL if split else 0.0)))
    dlr = dx.amax(2) + (S * U + 2.0 ** -21) / LN2
    dlc = dx.amax(1) + (L * U + 2.0 ** -21) / LN2
    return dx, dlr, dlc


def margins(conf: torch.Tensor) -> dict:
    """Top-2 of every row and column of conf (a single entry's runner-up is 0)."""
    def top2(dim):
        if conf.shape[dim] == 1:
            first = conf.squeeze(dim)
            return first.numpy(), np.zeros_like(first.numpy())
        t = conf.topk(2, dim=dim)[0]
        return t.select(dim, 0).numpy(), t.select(dim, 1).numpy()
    rm, r2 = top2(2)
    cm, c2 = top2(1)
    return dict(conf_rowmax=rm, conf_row2nd=r2, conf_colmax=cm, conf_col2nd=c2)


_REF_CACHE = collections.OrderedDict()


def cached_case(kind: str, seed: int, n: int, L: int, S: int, Cc: int, dtype, temperature: float = 0.1, sigma: float = 1.0):
    """(f0, f1, reference) for seeded inputs; the paths of one case share the reference."""
    key = (kind, seed, n, L, S, Cc, str(dtype), temperature, sigma)
    if key not in _REF_CACHE:
        if kind == "plain":
            f0, f1 = synth.coarse_features(seed, n, L, S, Cc, sigma=sigma, dtype=dtype)
        elif kind == "hard":
            f0, f1 = synth.hard_coarse_features(seed, n, L, S, Cc, sigma=sigma, dtype=dtype)
        else:
            raise KeyError(kind)
        _REF_CACHE[key] = (f0, f1, reference(f0, f1, temperature))
        while len(_REF_CACHE) > 3:
            _REF_CACHE.popitem(last=False)
    return _REF_CACHE[key]


# ---- one GPU run, checked against the reference ------------------------------------------------------------------------
def poisoned_workspace(n: int, L: int, S: int, Cc: int, dtype) -> torch.Tensor:
    """A coarse workspace filled with 0xFF bytes: every float the launch sequence fails to write reads back as nan, so no
    log-sum-exp can pass on a value an earlier run left behind (the paths of one case run on the same inputs one after
    another, and the caching allocator would hand each the block the previous one freed)."""
    need = _lib.lib().pope_coarse_workspace_bytes_ex(n, L, S, Cc, _lib.dtype_code(torch.empty(0, dtype=dtype)))
    return torch.full((need,), 0xFF, dtype=torch.uint8, device=DEV)


def run_coarse(f0, f1, hw0, hw1, impl, thr=0.2, border_rm=2, temperature=0.1, pixel_scale=8.0, knob=None) -> dict:
    n, L, S = f0.shape[0], f0.shape[1], f1.shape[1]
    ws = poisoned_workspace(n, L, S, f0.shape[2], f0.dtype)
    if knob is not None:
        os.environ["POPE_TC_DEBUG"] = knob
    try:
        res = ops.coarse_match(f0.to(DEV), f1.to(DEV), hw0, hw1, pixel_scale, thr, border_rm, temperature, impl, ws)
    finally:
        os.environ.pop("POPE_TC_DEBUG", None)
    assert res["workspace"] is ws
    v = ops.scratch_views(res["workspace"], n, L, S)
    flags = res.flags()
    out = {k: t.cpu() for k, t in res.sliced().items()} if not flags & ~_lib.FLAG_ROBUST_PATH else None
    return dict(out=out, flags=flags, counts=res["counts"][:n].cpu(), lse_r=v["lse_r"].cpu().double(),
                lse_c=v["lse_c"].cpu().double())


def check(request, ref, got, hw0, hw1, thr=0.2, border_rm=2, pixel_scale=8.0, split=False, flags=0):
    """Flags exactly `flags`; every log-sum-exp and every mconf within the bound; no index difference outside the near-tie /
    near-threshold classes; mkpts exact; counts = bincount; sorted by (b, i).  Returns the list."""
    assert got["flags"] == flags, f"flags {got['flags']}, expected {flags}"
    out = got["out"]
    n, L, S = ref["x"].shape
    dx, dlr, dlc = _bounds(ref, split)
    er = (got["lse_r"] - ref["lse_r"]).abs() / dlr
    ec = (got["lse_c"] - ref["lse_c"]).abs() / dlc
    assert bool(torch.isfinite(got["lse_r"]).all() and torch.isfinite(got["lse_c"]).all())
    worst_r, worst_c = divmod(int(er.argmax()), L), divmod(int(ec.argmax()), S)
    assert float(er.max()) <= 1.0, f"lse_r (pair, row) {worst_r}: error {float(er.max()):.3f} x the bound"
    assert float(ec.max()) <= 1.0, f"lse_c (pair, column) {worst_c}: error {float(ec.max()):.3f} x the bound"

    conf = conf_of(ref)
    thr32 = float(np.float32(thr))                       # the kernels compare against log2(float(thr))
    want = O.coarse_match_from_conf(conf, (hw0[0] * pixel_scale, hw0[1] * pixel_scale), hw0, hw1, thr32, border_rm)
    mg = margins(conf)
    same, near, bad = compare_match_lists(out, want, mg, thr32)
    assert not bad, f"index differences that are not near-ties: {bad[:5]}"
    assert len(near) <= max(2, want["b_ids"].numel() // 200), near

    b, i, j = out["b_ids"], out["i_ids"], out["j_ids"]
    for k in ("b_ids", "i_ids", "j_ids"):
        assert out[k].dtype == torch.int64
    assert out["mconf"].dtype == torch.float32 and not out["gt_mask"].any()
    em = torch.zeros(0, dtype=torch.float64)
    if b.numel():
        em = (torch.log2(out["mconf"].double()) - torch.log2(conf[b, i, j])).abs() / (
            2 * dx[b, i, j] + dlr[b, i] + dlc[b, j] + 2.0 ** -20)
        assert float(em.max()) <= 1.0, f"mconf of match {int(em.argmax())}: error {float(em.max()):.3f} x the bound"
        assert_sorted_by_pair_and_row(b, i, L)
    ps = torch.tensor(pixel_scale, dtype=torch.float32)
    for ids, w, key in ((i, hw0[1], "mkpts0_c"), (j, hw1[1], "mkpts1_c")):
        assert torch.equal(out[key], torch.stack([ids % w, ids // w], 1).float() * ps), key
    assert torch.equal(torch.bincount(b, minlength=n).to(torch.int32), got["counts"])
    RATIOS[request.node.name] = dict(lse=round(max(float(er.max()), float(ec.max())), 4),
                                     mconf=round(float(em.max()) if em.numel() else 0.0, 4), matches=int(b.numel()))
    return out


PATHS_BF16 = {SINGLE: dict(impl=_lib.COARSE_TCGEN05, thr=0.2), TWO: dict(impl=_lib.COARSE_TCGEN05, thr=0.2, knob="16"),
              THREE: dict(impl=_lib.COARSE_TCGEN05, thr=0.1), "simt_0.2": dict(impl=_lib.COARSE_SIMT, thr=0.2),
              "simt_0.1": dict(impl=_lib.COARSE_SIMT, thr=0.1)}
PATHS_F32 = {SPLIT: dict(impl=_lib.COARSE_TCGEN05, thr=0.2), "simt_0.2": dict(impl=_lib.COARSE_SIMT, thr=0.2),
             "simt_0.1": dict(impl=_lib.COARSE_SIMT, thr=0.1)}
HW0, HW1 = (30, 40), (27, 37)           # S = 999: odd, S % 32 = 7 (colsum_reduce_kernel<1>), L % 256 != 0


# ---- CPU: scratch layout, dispatch, reference -------------------------------------------------------------------------
_CARVE_SRC = r"""
#include <stdio.h>
#include <stdlib.h>
#include "common.cuh"
int main(int argc, char** argv) {
  for (int a = 1; a + 2 < argc; a += 3) {
    const int n = atoi(argv[a]), L = atoi(argv[a + 1]), S = atoi(argv[a + 2]);
    const pope::CoarseScratch w = pope::carve_coarse_scratch(nullptr, n, L, S);
    const void* r[] = {w.rowbest, w.colbest, w.cand_cnt, w.ready, w.lse_r, w.lse_c, w.cand, w.cbound, w.cminb, w.colpart,
                       w.cshift, w.pairflag};
    for (const void* q : r) printf("%zu ", size_t(q));
    printf("%zu\n", w.bytes);
  }
  return 0;
}
"""


def test_scratch_views_place_every_region_where_the_library_carves_it(tmp_path):
    """ops.scratch_views against carve_coarse_scratch itself (csrc/common.cuh, compiled for the host): every region at the
    library's offset, and the regions add up to pope_coarse_workspace_bytes.  n = 64 and 128 are the batches where a
    one-int error in the size of `ready` (it holds n + 1 ints) moves every later region by 256 bytes."""
    src = tmp_path / "carve.cu"
    src.write_text(_CARVE_SRC)
    exe = tmp_path / "carve"
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc) and shutil.which(nvcc) is None:
        pytest.skip("nvcc not found: the scratch layout is compiled from csrc/common.cuh")
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(ROOT, "pope_b200", "csrc"), str(src), "-o", str(exe)], check=True)
    shapes = [(n, L, S) for n in (1, 63, 64, 65, 128) for L, S in ((1, 1), (37, 999), (1200, 4801))]
    lines = subprocess.run([str(exe)] + [str(v) for s in shapes for v in s], check=True, capture_output=True,
                           text=True).stdout.split("\n")
    names = ("rowbest", "colbest", "cand_cnt", "ready", "lse_r", "lse_c", "cand", "cbound", "cminb", "colpart", "cshift",
             "pairflag")
    h = _lib.lib()
    for (n, L, S), line in zip(shapes, lines):
        offs = [int(t) for t in line.split()]
        total = h.pope_coarse_workspace_bytes(n, L, S)
        assert offs[-1] == total
        ws = torch.empty(total, dtype=torch.uint8)
        base = ws.data_ptr()
        v = ops.scratch_views(ws, n, L, S)
        assert list(v) == list(names)
        for name, off in zip(names, offs):
            assert v[name].data_ptr() - base == off, (n, L, S, name)
        assert v["pairflag"].data_ptr() - base + v["pairflag"].numel() * 4 <= total


def test_dispatch_table():
    """AUTO takes the tensor cores exactly for C in {64, 128, 192, 256}, for bf16 and fp32 features alike; the extended
    workspace adds the six split planes exactly for fp32 with C % 64 == 0 and C <= 256."""
    h = _lib.lib()
    for dtype in (_lib.POPE_BF16, _lib.POPE_F32):
        for Cc in range(16, 513, 16):
            want = _lib.COARSE_TCGEN05 if Cc in (64, 128, 192, 256) else _lib.COARSE_SIMT
            assert h.pope_coarse_auto_impl(dtype, 1200, 999, Cc) == want, (dtype, Cc)
            for n, L, S in ((1, 1, 1), (3, 1200, 999)):
                std = -(-h.pope_coarse_workspace_bytes(n, L, S) // 256) * 256
                planes = 3 * 2 * (n * L * Cc + n * S * Cc) + 6 * 256
                split = dtype == _lib.POPE_F32 and Cc % 64 == 0 and Cc <= 256
                assert h.pope_coarse_workspace_bytes_ex(n, L, S, Cc, dtype) == std + (planes if split else 0), (dtype, Cc)


@pytest.mark.parametrize("name", list(COARSE_CASES))
def test_reference_agrees_with_the_golden_fixtures(golden_dir, name):
    """The float64 reference gives the reference implementation's own match lists (tests/golden/coarse_*.npz) outside
    the near-tie / near-threshold classes."""
    case = COARSE_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    f0, f1 = coarse_inputs(case)
    ref = reference(f0, f1, with_bound=False)
    hw0, hw1 = case["hw0_c"], case["hw1_c"]
    want = O.coarse_match_from_conf(conf_of(ref), (hw0[0] * 8, hw0[1] * 8), hw0, hw1)
    gold = {k: torch.from_numpy(g[k]) for k in ("b_ids", "i_ids", "j_ids")}
    same, near, bad = compare_match_lists(want, gold, g)
    assert not bad, bad[:5]
    assert len(near) <= max(2, gold["b_ids"].numel() // 200)
    if not near:
        np.testing.assert_allclose(want["mconf"].numpy(), g["mconf"], rtol=1e-4 if case["kind"] != "hard" else 5e-4)


def test_bound_catches_a_tenth_of_a_percent_at_the_benchmark_shape():
    """At the benchmark shape (480x640 -> 60 x 80 cells, C = 256, bf16) the bound of every row and column log-sum-exp is
    below log2(1.001): a kernel that loses 0.1 % of one sum cannot pass."""
    f0, f1 = synth.coarse_features(1234, 1, 4800, 4800, 256, dtype=torch.bfloat16)
    _, dlr, dlc = _bounds(reference(f0, f1), split=False)
    assert max(float(dlr.max()), float(dlc.max())) < 1.4e-3


def _planted_candidates(seed, rows, L, S, Cc, dtype):
    """Background of small similarities plus, for each planted row, graded cells (log2 offsets) in columns that all fall
    into ONE six-slot sub-list of the single sweep, weakest first in sweep order.  The sweep's epilogue thread
    (column group cg, lane p % 4) of a row sees the columns with (j % 256) // 64 == cg and (j % 8) // 2 == p; tiles of 256
    columns are swept in order, and each thread's 64 columns in two chunks of 32.  Returns (f0, f1, [(row, strongest col)])."""
    g = torch.Generator().manual_seed(seed)
    f0, f1 = 0.3 * torch.randn(1, L, Cc, generator=g), 0.3 * torch.randn(1, S, Cc, generator=g)
    scale = 1.0 / (LN2 * Cc * 0.1)
    planted = []
    for t, (row, offsets) in enumerate(rows):
        base = 64 * (t % 4) + 2 * ((t // 4) % 4) + (t // 16) % 2
        steps = {5: (0, 8, 32, 512, 768), 6: (0, 8, 32, 256, 512, 768), 8: (0, 32, 256, 288, 512, 544, 768, 800)}[len(offsets)]
        u = torch.randn(Cc, generator=g)
        f0[0, row] = u
        for s, off in zip(steps, offsets):
            f1[0, base + s] = u * ((24.0 + off) / (scale * float(u @ u)))
        planted.append((row, base + steps[-1]))
    return f0.to(dtype), f1.to(dtype), planted


# ---- GPU: widths x paths ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS_BF16))
@pytest.mark.parametrize("Cc", [64, 128, 192, 256])
def test_width_path_bf16(request, Cc, path):
    f0, f1, ref = cached_case("plain", 300 + Cc, 2, 1200, 999, Cc, torch.bfloat16)
    p = dict(PATHS_BF16[path])
    got = run_coarse(f0, f1, HW0, HW1, **p)
    out = check(request, ref, got, HW0, HW1, thr=p["thr"])
    assert out["b_ids"].numel() > 300


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS_F32))
@pytest.mark.parametrize("Cc", [64, 128, 192, 256])
def test_width_path_fp32(request, Cc, path):
    f0, f1, ref = cached_case("plain", 400 + Cc, 2, 1200, 999, Cc, torch.float32)
    p = dict(PATHS_F32[path])
    got = run_coarse(f0, f1, HW0, HW1, **p)
    out = check(request, ref, got, HW0, HW1, thr=p["thr"], split=path == SPLIT)
    assert out["b_ids"].numel() > 300


@pytest.mark.gpu
@pytest.mark.parametrize("Cc", [64, 128, 192, 256])
def test_fp32_split_equals_simt(Cc):
    """fp32 features: the tensor-core split path and the fp32-FMA kernels give identical index lists; the split path does not
    take thr <= 0.15 (its single sweep needs the candidate lists) and says so."""
    f0, f1 = synth.coarse_features(400 + Cc, 2, 1200, 999, Cc)
    a = run_coarse(f0, f1, HW0, HW1, _lib.COARSE_TCGEN05)["out"]
    b = run_coarse(f0, f1, HW0, HW1, _lib.COARSE_SIMT)["out"]
    for k in ("b_ids", "i_ids", "j_ids"):
        assert torch.equal(a[k], b[k]), k
    with pytest.raises(_lib.PopeError):
        ops.coarse_match(f0.to(DEV), f1.to(DEV), HW0, HW1, 8.0, thr=0.1, impl=_lib.COARSE_TCGEN05)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("Cc", [16, 48, 80, 320])
def test_width_the_tensor_cores_cannot_take(request, Cc, dtype):
    """AUTO runs the SIMT kernels and matches the reference; an explicit tcgen05 request is refused."""
    assert _lib.lib().pope_coarse_auto_impl(_lib.dtype_code(torch.empty(0, dtype=dtype)), 1200, 999, Cc) == _lib.COARSE_SIMT
    f0, f1, ref = cached_case("plain", 500 + Cc, 2, 1200, 999, Cc, dtype)
    check(request, ref, run_coarse(f0, f1, HW0, HW1, _lib.COARSE_AUTO), HW0, HW1)
    with pytest.raises(_lib.PopeError):
        ops.coarse_match(f0.to(DEV), f1.to(DEV), HW0, HW1, 8.0, impl=_lib.COARSE_TCGEN05)


# ---- GPU: grids -------------------------------------------------------------------------------------------------------
GRID_VARIANTS = {"bf16_c256": (torch.bfloat16, 256, _lib.COARSE_TCGEN05), "fp32_c64_split": (torch.float32, 64, _lib.COARSE_TCGEN05),
                 "bf16_c256_simt": (torch.bfloat16, 256, _lib.COARSE_SIMT)}
GRID_CASES = [(shape, var) for shape in GRID_SHAPES for var in GRID_VARIANTS
              if var != "bf16_c256_simt" or shape in ((1, 1), (31, 33), (255, 257), (4800, 37))]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,variant", GRID_CASES, ids=[f"{L}x{S}-{v}" for (L, S), v in GRID_CASES])
def test_grid(request, shape, variant):
    """(h, 1) column grids with no border, as CoarseMatching._forward_masked runs a padded pair's valid cells: single rows
    and columns, ragged row groups and tiles, exactly one tile, and long thin grids in both orientations."""
    L, S = shape
    dtype, Cc, impl = GRID_VARIANTS[variant]
    f0, f1, ref = cached_case("plain", 600 + L + 7 * S, 2, L, S, Cc, dtype)
    got = run_coarse(f0, f1, (L, 1), (S, 1), impl, border_rm=0)
    check(request, ref, got, (L, 1), (S, 1), border_rm=0, split=variant == "fp32_c64_split")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(GRID_VARIANTS))
def test_border_without_interior_returns_empty_lists(variant):
    dtype, Cc, impl = GRID_VARIANTS[variant]
    f0, f1 = synth.coarse_features(7, 2, 12, 12, Cc, dtype=dtype)
    res = ops.coarse_match(f0.to(DEV), f1.to(DEV), (3, 4), (4, 3), 8.0, border_rm=2, impl=impl,
                           workspace=poisoned_workspace(2, 12, 12, Cc, dtype))
    assert res.flags() == 0
    out = res.sliced()
    for k, dt in (("b_ids", torch.int64), ("i_ids", torch.int64), ("j_ids", torch.int64), ("mconf", torch.float32),
                  ("mkpts0_c", torch.float32), ("mkpts1_c", torch.float32), ("gt_mask", torch.bool)):
        assert out[k].dtype == dt and out[k].shape[0] == 0, k
    assert out["mkpts0_c"].shape == (0, 2) and out["mkpts1_c"].shape == (0, 2)


# ---- GPU: batches -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_batch_with_split_single_sweep(request, dtype):
    """80 pairs of 255 cells: 80 units = one full round of 74 CTA pairs + 6, so the single sweep runs as head + tail with
    the head's column merge beside the tail."""
    n, hw0, hw1 = 80, (15, 17), (13, 11)
    assert _lib.single_sweep_is_split(n, hw0[0] * hw0[1])
    f0, f1, ref = cached_case("plain", 700, n, 255, 143, 128, dtype)
    check(request, ref, run_coarse(f0, f1, hw0, hw1, _lib.COARSE_TCGEN05), hw0, hw1, split=dtype == torch.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("path", [SINGLE, THREE, "simt_0.2"])
def test_batch_of_64_pairs(request, path):
    """n = 64, where the scratch's `ready` region (n + 1 ints) ends exactly on a 256-byte boundary plus one int."""
    n, hw0, hw1 = 64, (12, 16), (11, 13)
    f0, f1, ref = cached_case("plain", 701, n, 192, 143, 256, torch.bfloat16)
    p = dict(PATHS_BF16[path])
    check(request, ref, run_coarse(f0, f1, hw0, hw1, **p), hw0, hw1, thr=p["thr"])


# ---- GPU: match parameters -------------------------------------------------------------------------------------------
PARAMS = {"temperature_0.05": dict(temperature=0.05), "temperature_0.2": dict(temperature=0.2), "border_1": dict(border_rm=1),
          "border_3": dict(border_rm=3), "thr_0.149": dict(thr=0.149), "thr_0.151": dict(thr=0.151), "thr_0.16": dict(thr=0.16),
          "thr_0.5": dict(thr=0.5), "thr_0.9": dict(thr=0.9), "pixel_scale_4": dict(pixel_scale=4.0),
          "pixel_scale_2.5": dict(pixel_scale=2.5)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PARAMS))
def test_match_parameters(request, name):
    """C = 256 bf16 on the tcgen05 path.  The temperature moves scale_log2 and with it the shift ranges; thr 0.149 / 0.151
    sit on either side of the three-sweep / single-sweep boundary (thr * 8 > 1.2), 0.151 - 0.16 leave the single sweep's
    six-slot lane lists the least room."""
    kw = dict(PARAMS[name])
    temperature = kw.pop("temperature", 0.1)
    f0, f1, ref = cached_case("plain", 800, 2, 1200, 999, 256, torch.bfloat16, temperature=temperature)
    got = run_coarse(f0, f1, HW0, HW1, _lib.COARSE_TCGEN05, temperature=temperature, **kw)
    check(request, ref, got, HW0, HW1, **kw)


# ---- GPU: dynamic range ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("Cc", [128, 192])
def test_large_token_norm_stays_on_the_single_sweep(request, Cc):
    """Token norm ~ 49 (sigma 49/16): |x| reaches ~135 log2 units, so every epilogue warp raises its lazy shift; at two and
    three k-chunks the pair must stay on the fast path."""
    f0, f1, ref = cached_case("plain", 900 + Cc, 2, 1200, 999, Cc, torch.bfloat16, sigma=49.0 / 16.0)
    check(request, ref, run_coarse(f0, f1, HW0, HW1, _lib.COARSE_TCGEN05), HW0, HW1)


@pytest.mark.gpu
def test_hard_features_take_the_gated_two_sweep_launch(request):
    """x50 rows are out of one shift's range: the single sweep flags the pairs and the gated MODE 2 launch redoes them at
    kchunks = 2 (C = 128)."""
    f0, f1, ref = cached_case("hard", 950, 2, 1200, 999, 128, torch.bfloat16, sigma=0.9)
    got = run_coarse(f0, f1, HW0, HW1, _lib.COARSE_TCGEN05)
    check(request, ref, got, HW0, HW1, flags=_lib.FLAG_ROBUST_PATH)


# ---- GPU: candidate lists --------------------------------------------------------------------------------------------
CAND_ROWS = (0, 9, 31, 32, 45, 100, 127, 128, 200, 255, 256, 300, 511, 640, 1000, 1199)
GRADED5, GRADED6 = (0.0, 0.1, 0.2, 0.3, 0.5), (0.0, 0.1, 0.2, 0.3, 0.4, 0.6)
GEOMETRIC8 = tuple(0.45 * k for k in range(8))      # each cell above 0.2 x the sum so far: the full list is re-filtered


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.151, 0.2])
def test_candidate_lists_fill_before_the_strongest_cell(request, thr):
    """Planted rows whose candidates all land in one lane's six-slot sub-list, weakest first: five graded cells, or eight
    growing geometrically (thr 0.2: the list is full when the seventh arrives and must be re-filtered against the running
    row sum), or six graded cells at thr 0.151 (every slot used).  The strongest cell must win, with no flag at all."""
    rows = [(r, (GRADED6 if thr < 0.2 else (GRADED5 if t % 2 == 0 else GEOMETRIC8))) for t, r in enumerate(CAND_ROWS)]
    f0, f1, planted = _planted_candidates(1000 + int(thr * 1000), rows, 1200, 999, 256, torch.bfloat16)
    ref = reference(f0, f1)
    got = run_coarse(f0, f1, HW0, HW1, _lib.COARSE_TCGEN05, thr=thr, border_rm=0)
    out = check(request, ref, got, HW0, HW1, thr=thr, border_rm=0)
    assert sorted(zip(out["i_ids"].tolist(), out["j_ids"].tolist())) == sorted(planted)
