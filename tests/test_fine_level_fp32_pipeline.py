"""The fp32-accuracy fine level inside the host pipeline: `pope_pipeline_set_fine_level_ex(..., POPE_F32, ...)`,
`driver.Pipeline(torch.float32, fine_level=<fp32 bundle>)`, `driver.match_pairs_host(fine_level=)`.

The reference is the fp32 device step `ops.match_pairs_device(..., fine_level=<fp32 bundle>)` on the same inputs, which
tests/test_fine_level_fp32_device.py holds bit for bit to the Matcher's steps 3-5 with `fine_cuda_fp32=True`: ids and
confidences must be equal and the fine keypoints equal bit for bit, whichever way the fp32 fine maps (512-byte pixels)
reach the device.  `last_h2d_bytes` is checked to the byte."""
import ctypes as C

import numpy as np
import pytest
import torch

import pope_b200
from pope_b200 import _lib, driver, ops, synth

PIXEL = 128 * 4          # one fp32 fine-map pixel (Cf = 128)
DEV = torch.device("cuda:0")


def _matcher(seed=0, **cfg_changes):
    torch.manual_seed(seed)
    cfg = pope_b200.make_default_cfg()
    cfg.update(cfg_changes)
    return pope_b200.Matcher(cfg, fine_cuda_fp32=True).eval().to(DEV)


def _inputs(seed, n, hw0, hw1):
    """CPU fp32 inputs: coarse features [n, L|S, 256] and channels-last fine maps (logical [n, 128, 4h, 4w])."""
    (h0, w0), (h1, w1) = hw0, hw1
    f0, f1 = synth.coarse_features(seed, n, h0 * w0, h1 * w1, 256, sigma=0.9)
    ff0, ff1 = synth.fine_feature_maps(seed + 1, n, 4 * max(h0, h1), 4 * max(w0, w1), 128)
    ff0 = ff0[:, :, :4 * h0, :4 * w0].contiguous(memory_format=torch.channels_last)
    ff1 = ff1[:, :, :4 * h1, :4 * w1].contiguous(memory_format=torch.channels_last)
    return f0, f1, ff0, ff1


def _device_step(inputs, hw0, hw1, fine_level):
    f0, f1, ff0, ff1 = (t.to(DEV) for t in inputs)
    res = ops.match_pairs_device(f0, f1, ff0, ff1, (8 * hw0[0], 8 * hw0[1]), hw0, hw1, fine_level=fine_level)
    k = res.total()
    assert res.flags() == 0
    return {key: res[key][:k].cpu() for key in ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f")}


def _union_pixels(b_ids, cell_ids, n, hw_c):
    """pixels of a [n, 4h, 4w] fine map inside the 5 x 5 window of at least one of the listed cells"""
    h, w = hw_c
    need = np.zeros((n, 4 * h, 4 * w), dtype=bool)
    for b, c in zip(b_ids.tolist(), cell_ids.tolist()):
        cy, cx = divmod(c, w)
        need[b, max(0, 4 * cy - 2):4 * cy + 3, max(0, 4 * cx - 2):4 * cx + 3] = True
    return int(need.sum())


def _expected_h2d(form, inputs, want, hw0, hw1):
    f0, f1, ff0, ff1 = inputs
    n, m = f0.shape[0], want["b_ids"].numel()
    coarse = (f0.numel() + f1.numel()) * 4
    if form in ("pageable", "bulk"):
        return coarse + (ff0.numel() + ff1.numel()) * 4
    if form == "windows":
        return coarse + 2 * m * 25 * PIXEL
    u0, u1 = _union_pixels(want["b_ids"], want["i_ids"], n, hw0), _union_pixels(want["b_ids"], want["j_ids"], n, hw1)
    assert 0 < u0 < m * 25 and 0 < u1 < m * 25
    return coarse + (u0 + u1) * PIXEL


def _run(pl, inputs, form):
    f0, f1, ff0, ff1 = inputs
    nhwc = [t.permute(0, 2, 3, 1).contiguous() for t in (ff0, ff1)]
    host = [f0, f1] + nhwc
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
    """sets POPE_PIPELINE_F1 for the form under test (pageable buffers: unset, they are always copied whole)"""
    monkeypatch.delenv("POPE_PIPELINE_WINDOWS_IN_PLACE", raising=False)

    def set_form(form):
        if form == "pageable":
            monkeypatch.delenv("POPE_PIPELINE_F1", raising=False)
        else:
            monkeypatch.setenv("POPE_PIPELINE_F1", form)
    return set_form


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["pageable", "union", "windows", "bulk"])
def test_fp32_pipeline_with_fine_level_equals_the_device_step(form, f1_form):
    """5 pairs in chunks of 2 (a ragged last chunk), in each form the fine maps can reach the device."""
    n, hw = 5, (20, 24)
    m = _matcher()
    fl = m.fine_level(DEV, dtype=torch.float32)
    inputs = _inputs(11, n, hw, hw)
    want = _device_step(inputs, hw, hw, fl)
    assert want["b_ids"].numel() > 100
    f1_form(form)
    pl = driver.Pipeline(torch.float32, 2, (8 * hw[0], 8 * hw[1]), hw, hw, device=0, fine_level=fl)
    out = _run(pl, inputs, form)
    _assert_equal(out, want, form)
    assert pl.last_f1_mode == ("bulk" if form == "pageable" else form)
    assert pl.last_h2d_bytes == _expected_h2d(form, inputs, want, hw, hw), form
    pl.close()
    if form == "pageable":              # the one-shot entry point takes the same route
        _assert_equal(driver.match_pairs_host(*inputs, (8 * hw[0], 8 * hw[1]), hw, hw, chunk_pairs=2, fine_level=fl), want)


@pytest.mark.gpu
@pytest.mark.parametrize("n,hw0,hw1", [(4, (20, 24), (16, 20)), (3, (16, 20), (20, 24))])
def test_fp32_pipeline_with_fine_level_other_geometries(n, hw0, hw1, f1_form):
    """L != S both ways: image 0 larger than image 1 (its own grid in the image-0 union fetch), and smaller"""
    m = _matcher(1)
    fl = m.fine_level(DEV, dtype=torch.float32)
    inputs = _inputs(21 + n, n, hw0, hw1)
    want = _device_step(inputs, hw0, hw1, fl)
    assert want["b_ids"].numel() > 100
    f1_form("union")
    pl = driver.Pipeline(torch.float32, 2, (8 * hw0[0], 8 * hw0[1]), hw0, hw1, device=0, fine_level=fl)
    out = _run(pl, inputs, "union")
    _assert_equal(out, want, (hw0, hw1))
    assert pl.last_f1_mode == "union"
    assert pl.last_h2d_bytes == _expected_h2d("union", inputs, want, hw0, hw1)
    pl.close()


@pytest.mark.gpu
def test_fp32_pipeline_with_fine_level_without_coarse_concat(f1_form):
    """fine_concat_coarse_feat off: no FinePreprocess Linears (pre = NULL), the transformer alone"""
    n, hw = 3, (20, 24)
    m = _matcher(2, fine_concat_coarse_feat=False)
    fl = m.fine_level(DEV, dtype=torch.float32)
    assert fl["pre"] is None
    inputs = _inputs(31, n, hw, hw)
    want = _device_step(inputs, hw, hw, fl)
    f1_form("union")
    pl = driver.Pipeline(torch.float32, 2, (8 * hw[0], 8 * hw[1]), hw, hw, device=0, fine_level=fl)
    _assert_equal(_run(pl, inputs, "union"), want)
    pl.close()


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["union", "windows"])
def test_fp32_pipeline_with_fine_level_chunk_without_matches(form, f1_form):
    """the first chunk's pairs have no match (every count 0 bounds every fine-level launch), the second chunk has"""
    n, hw = 4, (20, 24)
    m = _matcher(3)
    fl = m.fine_level(DEV, dtype=torch.float32)
    f0, f1, ff0, ff1 = _inputs(41, n, hw, hw)
    f1[:2] = 0                           # every similarity 0: uniform softmaxes, confidence 1 / (L S), no match
    inputs = (f0, f1, ff0, ff1)
    want = _device_step(inputs, hw, hw, fl)
    assert int((want["b_ids"] < 2).sum()) == 0 and want["b_ids"].numel() > 50
    f1_form(form)
    pl = driver.Pipeline(torch.float32, 2, (8 * hw[0], 8 * hw[1]), hw, hw, device=0, fine_level=fl)
    out = _run(pl, inputs, form)
    assert out["counts"][:2].tolist() == [0, 0]
    _assert_equal(out, want)
    assert pl.last_h2d_bytes == _expected_h2d(form, inputs, want, hw, hw)
    pl.close()


@pytest.mark.gpu
def test_fp32_pipeline_fine_level_detaches_and_reattaches(f1_form):
    """detached, the pipeline returns what an fp32 pipeline that never had a fine level returns (the level really ran:
    that differs); attached again, the windows and scratch of the first attach are reused and the results return"""
    n, hw = 5, (20, 24)
    hw_i = (8 * hw[0], 8 * hw[1])
    m = _matcher(4)
    fl = m.fine_level(DEV, dtype=torch.float32)
    inputs = _inputs(51, n, hw, hw)
    want = _device_step(inputs, hw, hw, fl)
    f1_form("union")
    pl = driver.Pipeline(torch.float32, 2, hw_i, hw, hw, device=0, fine_level=fl)
    assert pl.fine_level is fl
    _assert_equal(_run(pl, inputs, "union"), want)
    pl.set_fine_level(None)
    detached = driver.flatten_slots(_run(pl, inputs, "union"))
    plain_pl = driver.Pipeline(torch.float32, 2, hw_i, hw, hw, device=0)
    plain = driver.flatten_slots(_run(plain_pl, inputs, "union"))
    plain_pl.close()
    for key in detached:
        assert torch.equal(detached[key], plain[key]), key
    assert torch.equal(detached["i_ids"], want["i_ids"]) and not torch.equal(detached["mkpts1_f"], want["mkpts1_f"])
    pl.set_fine_level(fl)
    _assert_equal(_run(pl, inputs, "union"), want, "re-attached")
    pl.close()


@pytest.mark.gpu
def test_set_fine_level_ex_status_codes():
    """the packing's dtype must be the pipeline's, in both directions; the bf16 entry point keeps rejecting fp32 pipelines"""
    m = _matcher(5)
    h = _lib.lib()
    args = ((160, 192), (20, 24), (20, 24))
    f32_fl, bf_fl = m.fine_level(DEV, dtype=torch.float32), m.fine_level(DEV)
    kinds = (C.c_int * len(f32_fl["layer_names"]))(*[0 if nm == "self" else 1 for nm in f32_fl["layer_names"]])
    fp32 = driver.Pipeline(torch.float32, 2, *args, device=0)
    bf16 = driver.Pipeline(torch.bfloat16, 2, *args, device=0)
    for pl, fl, wrong in ((fp32, f32_fl, _lib.POPE_BF16), (bf16, bf_fl, _lib.POPE_F32)):
        pre, layers = fl["pre"].data_ptr(), fl["layers"].data_ptr()
        assert h.pope_pipeline_set_fine_level_ex(pl._h, wrong, pre, layers, len(kinds), kinds) == -2     # POPE_ERR_DTYPE
        assert h.pope_pipeline_set_fine_level_ex(pl._h, 7, pre, layers, len(kinds), kinds) == -2
    assert h.pope_pipeline_set_fine_level(fp32._h, f32_fl["pre"].data_ptr(), f32_fl["layers"].data_ptr(), len(kinds),
                                          kinds) == -2
    pre, layers = f32_fl["pre"].data_ptr(), f32_fl["layers"].data_ptr()
    assert h.pope_pipeline_set_fine_level_ex(fp32._h, _lib.POPE_F32, pre + 8, layers, len(kinds), kinds) == -5
    assert h.pope_pipeline_set_fine_level_ex(fp32._h, _lib.POPE_F32, pre, layers, 0, kinds) == -1
    assert h.pope_pipeline_set_fine_level_ex(fp32._h, _lib.POPE_F32, pre, layers, len(kinds), kinds) == 0
    assert h.pope_pipeline_set_fine_level_ex(fp32._h, _lib.POPE_F32, None, None, 0, None) == 0             # detach
    fp32.close()
    bf16.close()
