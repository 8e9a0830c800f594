"""The bf16 fine level (FinePreprocess Linears + fine transformer) inside the host pipeline: `pope_pipeline_set_fine_level`,
`driver.Pipeline(fine_level=)`, `driver.match_pairs_host(fine_level=)`.

The reference is the sync-free device step `ops.match_pairs_device(..., fine_level=)` on the same inputs, which
tests/test_fine_level_device.py holds bit for bit to the Matcher's steps 3-5: ids and confidences must be equal and the
fine keypoints equal bit for bit, whichever way the fine maps reach the device.  `last_h2d_bytes` is checked to the byte:
with a fine level image 0's map crosses the host link in the same form as image 1's."""
import ctypes as C

import numpy as np
import pytest
import torch

import pope_b200
from pope_b200 import _lib, driver, ops, synth

PIXEL = 128 * 2          # one bf16 fine-map pixel (Cf = 128)


def _fine_level_cpu(**cfg_changes):
    cfg = pope_b200.make_default_cfg()
    cfg.update(cfg_changes)
    return pope_b200.Matcher(cfg, fine_cuda_bf16=True).eval().fine_level("cpu")


# ---- CPU: argument checking -----------------------------------------------------------------------------------------

def test_set_fine_level_rejects_a_null_handle():
    kinds = (C.c_int * 2)(0, 1)
    assert _lib.lib().pope_pipeline_set_fine_level(None, 16, 16, 2, kinds) == -1          # POPE_ERR_INVALID_ARG
    assert _lib.lib().pope_pipeline_set_fine_level(None, None, None, 0, None) == -1


def test_set_fine_level_is_declared_and_bound():
    import os
    import re
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "pope_b200.h")).read()
    assert "pope_pipeline_set_fine_level" in re.findall(r"\b(pope_[a-z_0-9]+)\s*\(", header)
    restype, args = _lib.SIGNATURES["pope_pipeline_set_fine_level"]
    assert restype is C.c_int and len(args) == 5
    assert _lib.lib().pope_abi_version() == 1


def test_pipeline_rejects_a_fine_level_it_cannot_run_before_touching_the_gpu():
    fl = _fine_level_cpu()
    args = (2, (160, 192), (20, 24), (20, 24))
    with pytest.raises(_lib.PopeError, match="bfloat16"):                      # an fp32 pipeline
        driver.Pipeline(torch.float32, *args, fine_level=fl)
    with pytest.raises(_lib.PopeError, match="C_coarse"):                      # coarse features other than 256 wide
        driver.Pipeline(torch.bfloat16, *args, C_coarse=128, fine_level=fl)
    with pytest.raises(_lib.PopeError, match="cuda"):                          # packed weights on the CPU
        driver.Pipeline(torch.bfloat16, *args, fine_level=fl)
    with pytest.raises(_lib.PopeError, match="layer names"):                   # one layer name too few
        driver.Pipeline(torch.bfloat16, *args, fine_level=dict(fl, layer_names=fl["layer_names"][:-1]))
    with pytest.raises(_lib.PopeError, match="layer names"):                   # a layer kind the kernels do not have
        driver.Pipeline(torch.bfloat16, *args, fine_level=dict(fl, layer_names=["self", "full"]))
    with pytest.raises(_lib.PopeError, match="FinePreprocess"):
        driver.Pipeline(torch.bfloat16, *args, fine_level=dict(fl, pre=fl["pre"][:-16]))
    with pytest.raises(_lib.PopeError, match="cuda"):                          # the one-shot entry passes it through
        driver.match_pairs_host(*synth.coarse_features(1, 1, 480, 480, 256, dtype=torch.bfloat16),
                                *synth.fine_feature_maps(2, 1, 80, 96, 128, dtype=torch.bfloat16),
                                (160, 192), (20, 24), (20, 24), fine_level=fl)


# ---- GPU ------------------------------------------------------------------------------------------------------------

DEV = torch.device("cuda:0")


def _matcher(seed=0, **cfg_changes):
    torch.manual_seed(seed)
    cfg = pope_b200.make_default_cfg()
    cfg.update(cfg_changes)
    return pope_b200.Matcher(cfg, fine_cuda_bf16=True).eval().to(DEV)


def _inputs(seed, n, hw0, hw1):
    """CPU bf16 inputs: coarse features [n, L|S, 256] and channels-last fine maps (logical [n, 128, 4h, 4w])."""
    (h0, w0), (h1, w1) = hw0, hw1
    f0, f1 = synth.coarse_features(seed, n, h0 * w0, h1 * w1, 256, sigma=0.9, dtype=torch.bfloat16)
    ff0, ff1 = synth.fine_feature_maps(seed + 1, n, 4 * max(h0, h1), 4 * max(w0, w1), 128, dtype=torch.bfloat16)
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
    coarse = (f0.numel() + f1.numel()) * 2
    if form in ("pageable", "bulk"):
        return coarse + (ff0.numel() + ff1.numel()) * 2
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
def test_pipeline_with_fine_level_equals_the_device_step(form, f1_form):
    """5 pairs in chunks of 2 (a ragged last chunk), in each form the fine maps can reach the device."""
    n, hw = 5, (20, 24)
    m = _matcher()
    fl = m.fine_level(DEV)
    inputs = _inputs(11, n, hw, hw)
    want = _device_step(inputs, hw, hw, fl)
    assert want["b_ids"].numel() > 100
    f1_form(form)
    pl = driver.Pipeline(torch.bfloat16, 2, (8 * hw[0], 8 * hw[1]), hw, hw, device=0, fine_level=fl)
    out = _run(pl, inputs, form)
    _assert_equal(out, want, form)
    assert pl.last_f1_mode == ("bulk" if form == "pageable" else form)
    assert pl.last_h2d_bytes == _expected_h2d(form, inputs, want, hw, hw), form
    pl.close()
    if form == "pageable":              # the one-shot entry point takes the same route
        _assert_equal(driver.match_pairs_host(*inputs, (8 * hw[0], 8 * hw[1]), hw, hw, chunk_pairs=2, fine_level=fl), want)


@pytest.mark.gpu
@pytest.mark.parametrize("n,hw0,hw1", [(4, (20, 24), (16, 20)), (3, (60, 80), (60, 80))])
def test_pipeline_with_fine_level_other_geometries(n, hw0, hw1, f1_form):
    """image 0 larger than image 1 (its own grid in the image-0 union fetch), and the full 480x640 geometry"""
    m = _matcher(1)
    fl = m.fine_level(DEV)
    inputs = _inputs(21 + n, n, hw0, hw1)
    want = _device_step(inputs, hw0, hw1, fl)
    assert want["b_ids"].numel() > 100
    f1_form("union")
    pl = driver.Pipeline(torch.bfloat16, 2, (8 * hw0[0], 8 * hw0[1]), hw0, hw1, device=0, fine_level=fl)
    out = _run(pl, inputs, "union")
    _assert_equal(out, want, (hw0, hw1))
    assert pl.last_f1_mode == "union"
    assert pl.last_h2d_bytes == _expected_h2d("union", inputs, want, hw0, hw1)
    pl.close()


@pytest.mark.gpu
def test_pipeline_with_fine_level_without_coarse_concat(f1_form):
    """fine_concat_coarse_feat off: no FinePreprocess Linears (pre = NULL), the transformer alone"""
    n, hw = 3, (20, 24)
    m = _matcher(2, fine_concat_coarse_feat=False)
    fl = m.fine_level(DEV)
    assert fl["pre"] is None
    inputs = _inputs(31, n, hw, hw)
    want = _device_step(inputs, hw, hw, fl)
    f1_form("union")
    pl = driver.Pipeline(torch.bfloat16, 2, (8 * hw[0], 8 * hw[1]), hw, hw, device=0, fine_level=fl)
    _assert_equal(_run(pl, inputs, "union"), want)
    pl.close()


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["union", "windows"])
def test_pipeline_with_fine_level_chunk_without_matches(form, f1_form):
    """the first chunk's pairs have no match (every count 0 bounds every fine-level launch), the second chunk has"""
    n, hw = 4, (20, 24)
    m = _matcher(3)
    fl = m.fine_level(DEV)
    f0, f1, ff0, ff1 = _inputs(41, n, hw, hw)
    f1[:2] = 0                           # every similarity 0: uniform softmaxes, confidence 1 / (L S), no match
    inputs = (f0, f1, ff0, ff1)
    want = _device_step(inputs, hw, hw, fl)
    assert int((want["b_ids"] < 2).sum()) == 0 and want["b_ids"].numel() > 50
    f1_form(form)
    pl = driver.Pipeline(torch.bfloat16, 2, (8 * hw[0], 8 * hw[1]), hw, hw, device=0, fine_level=fl)
    out = _run(pl, inputs, form)
    assert out["counts"][:2].tolist() == [0, 0]
    _assert_equal(out, want)
    assert pl.last_h2d_bytes == _expected_h2d(form, inputs, want, hw, hw)
    pl.close()


@pytest.mark.gpu
def test_pipeline_fine_level_reruns_and_detaches(f1_form):
    """one handle run twice gives the same results; detached, it returns exactly what a pipeline that never had a fine
    level returns, and that differs from the refined keypoints (the level really ran)"""
    n, hw = 5, (20, 24)
    hw_i = (8 * hw[0], 8 * hw[1])
    m = _matcher(4)
    fl = m.fine_level(DEV)
    inputs = _inputs(51, n, hw, hw)
    want = _device_step(inputs, hw, hw, fl)
    f1_form("union")
    pl = driver.Pipeline(torch.bfloat16, 2, hw_i, hw, hw, device=0, fine_level=fl)
    assert pl.fine_level is fl
    for rep in range(2):
        _assert_equal(_run(pl, inputs, "union"), want, rep)
    pl.set_fine_level(None)
    assert pl.fine_level is None
    detached = _run(pl, inputs, "union")
    h2d_detached = pl.last_h2d_bytes
    plain_pl = driver.Pipeline(torch.bfloat16, 2, hw_i, hw, hw, device=0)
    plain = _run(plain_pl, inputs, "union")
    assert plain_pl.last_h2d_bytes == h2d_detached
    plain_pl.close()
    assert torch.equal(detached["flags"], plain["flags"])
    a, b = driver.flatten_slots(detached), driver.flatten_slots(plain)       # (slot rows past the counts are not written)
    for key in a:
        assert torch.equal(a[key], b[key]), key
    assert torch.equal(a["i_ids"], want["i_ids"]) and not torch.equal(a["mkpts1_f"], want["mkpts1_f"])
    pl.set_fine_level(fl)                # attached again: the windows and scratch of the first attach are reused
    _assert_equal(_run(pl, inputs, "union"), want, "re-attached")
    pl.close()


@pytest.mark.gpu
def test_set_fine_level_status_codes():
    m = _matcher(5)
    fl = m.fine_level(DEV)
    h = _lib.lib()
    layers, pre = fl["layers"].data_ptr(), fl["pre"].data_ptr()
    kinds = (C.c_int * len(fl["layer_names"]))(*[0 if nm == "self" else 1 for nm in fl["layer_names"]])
    args = ((160, 192), (20, 24), (20, 24))
    fp32 = driver.Pipeline(torch.float32, 2, *args, device=0)
    assert h.pope_pipeline_set_fine_level(fp32._h, pre, layers, len(kinds), kinds) == -2        # POPE_ERR_DTYPE
    fp32.close()
    narrow = driver.Pipeline(torch.bfloat16, 2, *args, C_coarse=128, device=0)
    assert h.pope_pipeline_set_fine_level(narrow._h, pre, layers, len(kinds), kinds) == -4      # POPE_ERR_SHAPE
    narrow.close()
    pl = driver.Pipeline(torch.bfloat16, 2, *args, device=0)
    assert h.pope_pipeline_set_fine_level(pl._h, pre, layers, 0, kinds) == -1                   # no layer
    assert h.pope_pipeline_set_fine_level(pl._h, pre, layers, 2, (C.c_int * 2)(0, 2)) == -1     # unknown kind
    assert h.pope_pipeline_set_fine_level(pl._h, pre, layers, 2, None) == -1
    assert h.pope_pipeline_set_fine_level(pl._h, pre + 8, layers, len(kinds), kinds) == -5      # POPE_ERR_ALIGNMENT
    assert h.pope_pipeline_set_fine_level(pl._h, None, layers, len(kinds), kinds) == 0          # pre is optional
    assert h.pope_pipeline_set_fine_level(pl._h, None, None, 0, None) == 0                      # detach
    pl.close()
    with pytest.raises(_lib.PopeError, match="cuda"):                # weights on another device than the pipeline's
        driver.Pipeline(torch.bfloat16, 2, *args, device=0, fine_level=m.fine_level("cpu"))
