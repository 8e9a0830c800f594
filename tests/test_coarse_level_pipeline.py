"""The coarse level inside the host pipeline, so that it starts from the backbone's coarse maps:
`pope_pipeline_set_coarse_level`, `driver.Pipeline(coarse_level=)`, `driver.match_pairs_host(coarse_level=)`.

The reference is the device step with both levels, `ops.match_pairs_device(..., coarse_level=, fine_level=)`, which
tests/test_coarse_level_device.py holds bit for bit to `Matcher(config, coarse_cuda_X=True, fine_cuda_X=True)`.  The maps
cross the link in fp32 whatever the pipeline's dtype; `last_h2d_bytes` is checked to the byte."""
import ctypes as C

import numpy as np
import pytest
import torch

import pope_b200
from pope_b200 import _lib, driver, ops, synth

DEV = torch.device("cuda:0")
DTYPES = {"bf16": torch.bfloat16, "fp32": torch.float32}


def _matcher(seed=0):
    torch.manual_seed(seed)
    return pope_b200.Matcher(pope_b200.make_default_cfg()).eval().to(DEV)


def _inputs(seed, n, hw0, hw1, dt):
    """CPU inputs: fp32 coarse maps [n, 256, h, w] and channels-last fine maps (logical [n, 128, 4h, 4w]) in `dt`"""
    (h0, w0), (h1, w1) = hw0, hw1
    f0, f1 = synth.coarse_features(seed, n, h0 * w0, h1 * w1, 256, sigma=0.9)
    c0 = f0.transpose(1, 2).reshape(n, 256, h0, w0).contiguous()
    c1 = f1.transpose(1, 2).reshape(n, 256, h1, w1).contiguous()
    ff0, ff1 = synth.fine_feature_maps(seed + 1, n, 4 * max(h0, h1), 4 * max(w0, w1), 128, dtype=dt)
    ff0 = ff0[:, :, :4 * h0, :4 * w0].contiguous(memory_format=torch.channels_last)
    ff1 = ff1[:, :, :4 * h1, :4 * w1].contiguous(memory_format=torch.channels_last)
    return c0, c1, ff0, ff1


def _device_step(inputs, hw0, hw1, **levels):
    res = ops.match_pairs_device(*(t.to(DEV) for t in inputs), (8 * hw0[0], 8 * hw0[1]), hw0, hw1, **levels)
    k = res.total()
    assert res.flags() == 0
    out = {key: res[key][:k].cpu() for key in ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f")}
    out["feat_c0"], out["feat_c1"] = res["feat_c0"].cpu(), res["feat_c1"].cpu()
    return out


def _union_pixels(b_ids, cell_ids, n, hw_c):
    """pixels of a [n, 4h, 4w] fine map inside the 5 x 5 window of at least one of the listed cells"""
    h, w = hw_c
    need = np.zeros((n, 4 * h, 4 * w), dtype=bool)
    for b, c in zip(b_ids.tolist(), cell_ids.tolist()):
        cy, cx = divmod(c, w)
        need[b, max(0, 4 * cy - 2):4 * cy + 3, max(0, 4 * cx - 2):4 * cx + 3] = True
    return int(need.sum())


def _expected_h2d(form, inputs, want, hw0, hw1):
    c0, c1, ff0, ff1 = inputs
    n = c0.shape[0]
    maps = n * (hw0[0] * hw0[1] + hw1[0] * hw1[1]) * 256 * 4          # the coarse maps, fp32
    assert maps == (c0.numel() + c1.numel()) * 4
    if form == "pageable":
        return maps + (ff0.numel() + ff1.numel()) * ff0.element_size()
    pixel = 128 * ff0.element_size()
    return maps + (_union_pixels(want["b_ids"], want["i_ids"], n, hw0) + _union_pixels(want["b_ids"], want["j_ids"], n, hw1)) * pixel


def _run(pl, inputs, form):
    c0, c1, ff0, ff1 = inputs
    host = [c0, c1] + [t.permute(0, 2, 3, 1).contiguous() for t in (ff0, ff1)]
    if form != "pageable":
        host = [t.pin_memory() for t in host]
    return pl.run(*host)


def _bits(t):
    return t.contiguous().view(torch.int32)


def _assert_equal(out, want, what=""):
    got = driver.flatten_slots(out)
    assert int(out["counts"].sum()) == want["b_ids"].numel(), what
    for key in ("b_ids", "i_ids", "j_ids", "mconf"):
        assert torch.equal(got[key], want[key]), (what, key)
    for key in ("mkpts0_f", "mkpts1_f"):
        assert torch.equal(_bits(got[key]), _bits(want[key])), (what, key)


@pytest.fixture
def f1_form(monkeypatch):
    """union for page-locked buffers (the default form); pageable buffers are always copied whole"""
    monkeypatch.delenv("POPE_PIPELINE_WINDOWS_IN_PLACE", raising=False)
    monkeypatch.delenv("POPE_PIPELINE_F1", raising=False)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["pageable", "union"])
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
def test_pipeline_with_both_levels_equals_the_device_step(dt, form, f1_form):
    """5 pairs in chunks of 2 (a ragged last chunk)"""
    dt = DTYPES[dt]
    n, hw = 5, (20, 24)
    m = _matcher()
    cl, fl = m.coarse_level(DEV, dt), m.fine_level(DEV, dt)
    inputs = _inputs(11, n, hw, hw, dt)
    want = _device_step(inputs, hw, hw, coarse_level=cl, fine_level=fl)
    assert want["b_ids"].numel() > 100
    pl = driver.Pipeline(dt, 2, (8 * hw[0], 8 * hw[1]), hw, hw, device=0, fine_level=fl, coarse_level=cl)
    out = _run(pl, inputs, form)
    _assert_equal(out, want, form)
    assert pl.last_f1_mode == ("bulk" if form == "pageable" else form)
    assert pl.last_h2d_bytes == _expected_h2d(form, inputs, want, hw, hw), form
    pl.close()
    if form == "pageable":              # the one-shot entry point takes the same route
        _assert_equal(driver.match_pairs_host(*inputs, (8 * hw[0], 8 * hw[1]), hw, hw, chunk_pairs=2, fine_level=fl,
                                              coarse_level=cl), want)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
def test_pipeline_with_both_levels_on_different_grids(dt, f1_form):
    """a 60 x 80 grid against 32 x 32 (a prompt image against a 256 x 256 crop), 3 pairs in chunks of 2"""
    dt = DTYPES[dt]
    n, hw0, hw1 = 3, (60, 80), (32, 32)
    m = _matcher(1)
    cl, fl = m.coarse_level(DEV, dt), m.fine_level(DEV, dt)
    inputs = _inputs(21, n, hw0, hw1, dt)
    want = _device_step(inputs, hw0, hw1, coarse_level=cl, fine_level=fl)
    assert want["b_ids"].numel() > 300
    pl = driver.Pipeline(dt, 2, (8 * hw0[0], 8 * hw0[1]), hw0, hw1, device=0, fine_level=fl, coarse_level=cl)
    _assert_equal(_run(pl, inputs, "union"), want)
    assert pl.last_h2d_bytes == _expected_h2d("union", inputs, want, hw0, hw1)
    pl.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
def test_pipeline_coarse_level_detaches_and_reattaches(dt, f1_form):
    """detached, the pipeline takes token-major features again and returns what a pipeline that never had a coarse level
    returns; on the transformed features that is the two-level result again.  Re-attached, the staging buffers and the
    scratch of the first attach are reused."""
    dt = DTYPES[dt]
    n, hw = 5, (20, 24)
    hw_i = (8 * hw[0], 8 * hw[1])
    m = _matcher(2)
    cl, fl = m.coarse_level(DEV, dt), m.fine_level(DEV, dt)
    inputs = _inputs(31, n, hw, hw, dt)
    want = _device_step(inputs, hw, hw, coarse_level=cl, fine_level=fl)
    pl = driver.Pipeline(dt, 2, hw_i, hw, hw, device=0, fine_level=fl, coarse_level=cl)
    assert pl.coarse_level is cl
    _assert_equal(_run(pl, inputs, "union"), want)
    pl.set_coarse_level(None)
    assert pl.coarse_level is None
    transformed = (want["feat_c0"], want["feat_c1"]) + tuple(inputs[2:])
    detached = driver.flatten_slots(_run(pl, transformed, "union"))
    plain_pl = driver.Pipeline(dt, 2, hw_i, hw, hw, device=0, fine_level=fl)
    plain = driver.flatten_slots(_run(plain_pl, transformed, "union"))
    plain_pl.close()
    for key in detached:
        assert torch.equal(detached[key], plain[key]), key
    _assert_equal(_run(pl, transformed, "union"), want, "detached, on the transformed features")
    pl.set_coarse_level(cl)
    _assert_equal(_run(pl, inputs, "union"), want, "re-attached")
    pl.close()


@pytest.mark.gpu
def test_set_coarse_level_status_codes():
    """the packing's dtype must be the pipeline's; the grids must fit the encoding; pointers aligned"""
    m = _matcher(3)
    h = _lib.lib()
    args = ((160, 192), (20, 24), (20, 24))
    cl32, cl16 = m.coarse_level(DEV, torch.float32), m.coarse_level(DEV)
    kinds = (C.c_int * len(cl32["layer_names"]))(*[0 if nm == "self" else 1 for nm in cl32["layer_names"]])
    fp32 = driver.Pipeline(torch.float32, 2, *args, device=0)
    bf16 = driver.Pipeline(torch.bfloat16, 2, *args, device=0)
    pe = cl32["pe"].data_ptr()
    for pl, cl, wrong in ((fp32, cl32, _lib.POPE_BF16), (bf16, cl16, _lib.POPE_F32)):
        layers = cl["layers"].data_ptr()
        assert h.pope_pipeline_set_coarse_level(pl._h, wrong, pe, 256, 256, layers, len(kinds), kinds) == -2
        assert h.pope_pipeline_set_coarse_level(pl._h, 7, pe, 256, 256, layers, len(kinds), kinds) == -2
    layers = cl32["layers"].data_ptr()
    code = _lib.POPE_F32
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, pe, 20, 23, layers, len(kinds), kinds) == -4   # grid > pe
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, pe + 2, 256, 256, layers, len(kinds), kinds) == -5
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, pe, 256, 256, layers + 8, len(kinds), kinds) == -5
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, pe, 256, 256, layers, 0, kinds) == -1
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, None, 256, 256, layers, len(kinds), kinds) == -1
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, pe, 0, 256, layers, len(kinds), kinds) == -1
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, pe, 256, 256, layers, len(kinds), kinds) == 0
    assert h.pope_pipeline_set_coarse_level(fp32._h, code, None, 0, 0, None, 0, None) == 0             # detach
    c128 = driver.Pipeline(torch.float32, 2, *args, C_coarse=128, device=0)
    assert h.pope_pipeline_set_coarse_level(c128._h, code, pe, 256, 256, layers, len(kinds), kinds) == -4
    for pl in (fp32, bf16, c128):
        pl.close()
