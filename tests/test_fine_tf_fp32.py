"""Fine level at fp32 accuracy (csrc/fine_tf.cu, fine_gemm_split_kernel): pope_fine_transformer_f32 /
pope_fine_merge_coarse_f32, `ops.pack_fine_layer / pack_fine_pre(..., dtype=torch.float32)`, `ops.fine_transformer` and
`ops.fine_merge_coarse` on fp32 windows, `FineTransformerB200.cuda_fp32`, `FinePreprocess.cuda_fp32` and
`Matcher(config, fine_cuda_fp32=True)`.

Every GEMM operand is split into three bf16 terms and the six significant products are accumulated in fp32, so the path
is held to the fp32 modules, not to bf16: against the stock modules run in float64 (with the same full fp32 weights), its
error (rms and max, relative to the output RMS) must stay within STOCK_FACTOR x that of the stock fp32 modules (TF32 off)
and BF16_FACTOR x below that of the bf16 CUDA fine level on the same case.  Both factors are chosen bars, not
measurements; the measured ratios are printed.
"""
import copy
import json
import os
import re

import numpy as np
import pytest
import torch
import torch.nn as nn

import pope_b200
from pope_b200 import _lib, ops, synth
from pope_b200.feature_net import FineTransformerB200, LocalFeatureTransformer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
# measured on a B200: 0.43-1.26x the stock fp32 error (rms and max), 8 800-120 000x below the bf16 path's (DESIGN 4.6)
STOCK_FACTOR = 6.0
BF16_FACTOR = 100.0
LAYER_MATS = (("qkv", (384, 128), 0), ("merge.weight", (128, 128), 294912), ("mlp.0.weight", (256, 256), 393216),
              ("mlp.2.weight", (128, 256), 786432))
PRE_MATS = (("down_proj.weight", (128, 256), 0), ("merge_feat.weight", (128, 256), 196608))


def _fine_cfg(names=None):
    cfg = copy.deepcopy(pope_b200.make_default_cfg()["fine"])
    if names is not None:
        cfg["layer_names"] = list(names)
    return cfg


def _model(names, seed=0):
    """A stock fine transformer with its own fp32 (xavier) weights and perturbed LayerNorm parameters."""
    torch.manual_seed(seed)
    m = LocalFeatureTransformer(_fine_cfg(names)).eval()
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if p.dim() == 1:
                p.copy_((1 if name.endswith("weight") else 0) + (0.2 if name.endswith("weight") else 0.1) *
                        torch.randn(p.shape, generator=gen))
    return m


def _pre(seed=0):
    """down_proj / merge_feat with fp32 weights as FinePreprocess initialises them, and random biases."""
    torch.manual_seed(seed)
    pre = nn.Module()
    pre.down_proj, pre.merge_feat = nn.Linear(256, 128), nn.Linear(256, 128)
    for lin in (pre.down_proj, pre.merge_feat):
        nn.init.kaiming_normal_(lin.weight, mode="fan_out", nonlinearity="relu")
        nn.init.normal_(lin.bias, std=0.1)
    return pre.eval()


def _matrix(sd, key):
    if key == "qkv":
        return torch.cat([sd["q_proj.weight"], sd["k_proj.weight"], sd["v_proj.weight"]])
    return sd[key]


def _rel_err(got, want):
    rms = want.double().pow(2).mean().sqrt()
    d = (got.double() - want.double()).abs()
    return float(d.pow(2).mean().sqrt() / rms), float(d.max() / rms)


def _windows(seed, m, ww=25, sigma=1.0):
    gen = torch.Generator().manual_seed(seed)
    return sigma * torch.randn(m, ww, 128, generator=gen), sigma * torch.randn(m, ww, 128, generator=gen)


# ---- CPU ------------------------------------------------------------------------------------------------------------

def _check_planes(packed, sd, mats, end):
    for key, shp, off in mats:
        w = _matrix(sd, key)
        n = shp[0] * shp[1] * 2
        planes = [packed[off + p * n:off + (p + 1) * n].view(torch.bfloat16).view(shp) for p in range(3)]
        assert torch.equal(planes[0], w.to(torch.bfloat16)), key
        assert torch.equal((planes[0].float() + planes[1].float()) + planes[2].float(), w), key
        assert off + 3 * n <= end
    return end


def test_fp32_packings_put_every_plane_at_the_header_offsets():
    header = open(os.path.join(ROOT, "include", "pope_b200.h")).read()
    for name, val in (("POPE_FINE_TF_F32_LAYER_BYTES", _lib.FINE_TF_F32_LAYER_BYTES),
                      ("POPE_FINE_PRE_F32_BYTES", _lib.FINE_PRE_F32_BYTES)):
        assert int(re.search(rf"#define {name} (\d+)", header).group(1)) == val
    for off in (294912, 393216, 786432, 983040, 196608, 393216, 393728):
        assert f"+{off} " in header
    sd = _model(["self"]).layers[0].state_dict()
    packed = ops.pack_fine_layer(sd, "cpu", dtype=torch.float32)
    assert packed.dtype == torch.uint8 and packed.numel() == _lib.FINE_TF_F32_LAYER_BYTES
    off = _check_planes(packed, sd, LAYER_MATS, 983040)
    for key in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"):
        assert torch.equal(packed[off:off + 512].view(torch.float32), sd[key]), key
        off += 512
    assert off == _lib.FINE_TF_F32_LAYER_BYTES
    psd = _pre().state_dict()
    pp = ops.pack_fine_pre(psd, "cpu", dtype=torch.float32)
    assert pp.numel() == _lib.FINE_PRE_F32_BYTES
    off = _check_planes(pp, psd, PRE_MATS, 393216)
    assert torch.equal(pp[off:off + 512].view(torch.float32), psd["down_proj.bias"])
    assert torch.equal(pp[off + 512:off + 1024].view(torch.float32), psd["merge_feat.bias"])
    # the bf16 layouts (the default) are unchanged
    mats = ("q_proj.weight", "k_proj.weight", "v_proj.weight", "merge.weight", "mlp.0.weight", "mlp.2.weight")
    old = torch.cat([torch.cat([sd[k].to(torch.bfloat16).reshape(-1) for k in mats]).view(torch.uint8),
                     torch.cat([sd[k].reshape(-1) for k in ("norm1.weight", "norm1.bias", "norm2.weight",
                                                            "norm2.bias")]).view(torch.uint8)])
    assert torch.equal(ops.pack_fine_layer(sd, "cpu"), old)
    assert torch.equal(ops.pack_fine_layer(sd, "cpu", dtype=torch.bfloat16), old)
    old_pre = torch.cat([torch.cat([psd[k].to(torch.bfloat16).reshape(-1) for k in ("down_proj.weight",
                                                                                   "merge_feat.weight")]).view(torch.uint8),
                         torch.cat([psd["down_proj.bias"], psd["merge_feat.bias"]]).view(torch.uint8)])
    assert torch.equal(ops.pack_fine_pre(psd, "cpu"), old_pre)
    for fn, arg in ((ops.pack_fine_layer, sd), (ops.pack_fine_pre, psd)):
        with pytest.raises(_lib.PopeError):
            fn(arg, "cpu", dtype=torch.float16)


def test_f32_transformer_entry_point_rejects_bad_arguments_before_touching_the_gpu():
    h = _lib.lib()
    kinds = (_lib.C.c_int * 2)(0, 1)
    ws = h.pope_fine_tf_f32_workspace_bytes(3, 25)
    assert ws > h.pope_fine_tf_workspace_bytes(3, 25) > 0
    assert h.pope_fine_tf_f32_workspace_bytes(0, 25) == 0 and h.pope_fine_tf_f32_workspace_bytes(3, 0) == 0
    assert h.pope_fine_tf_f32_workspace_bytes(-1, 25) == 0
    # feat0, feat1, m_windows, window_tokens, weights, n_layers, layer_kinds, workspace, workspace_bytes, stream
    ok = [16, 16, 3, 25, 16, 2, kinds, 16, ws, None]
    f = h.pope_fine_transformer_f32
    for i in (0, 1, 4, 6, 7):                                      # null windows, weights, kinds and workspace
        bad = list(ok); bad[i] = None
        assert f(*bad) == -1, i
    for i, v in ((2, -1), (3, 0), (5, -1)):                        # negative / empty sizes
        bad = list(ok); bad[i] = v
        assert f(*bad) == -1, i
    bad = list(ok); bad[6] = (_lib.C.c_int * 2)(0, 2)              # layer kind other than 'self' / 'cross'
    assert f(*bad) == -1
    for i in (0, 1, 4, 7):                                         # misaligned pointers
        bad = list(ok); bad[i] = 40
        assert f(*bad) == -5, i
    bad = list(ok); bad[8] = ws - 1                                # workspace too small (the bf16 size, too)
    assert f(*bad) == -3
    bad = list(ok); bad[8] = h.pope_fine_tf_workspace_bytes(3, 25)
    assert f(*bad) == -3
    bad = list(ok); bad[2] = 1 << 27                               # more rows than the kernels index
    assert f(*bad) == -4
    bad = list(ok); bad[2] = 0                                     # no windows: a no-op
    assert f(*bad) == 0


def test_f32_merge_entry_point_rejects_bad_arguments_before_touching_the_gpu():
    h = _lib.lib()
    ws = h.pope_fine_merge_f32_workspace_bytes(3)
    assert ws > h.pope_fine_merge_workspace_bytes(3) > 0
    assert h.pope_fine_merge_f32_workspace_bytes(0) == 0 and h.pope_fine_merge_f32_workspace_bytes(-2) == 0
    # win0, win1, m, tokens, feat_c0, feat_c1, L, S, C, b_ids, i_ids, j_ids, weights, workspace, workspace_bytes, stream
    ok = [16, 16, 3, 25, 16, 16, 64, 48, 256, 16, 16, 16, 16, 16, ws, None]
    f = h.pope_fine_merge_coarse_f32
    for i in (0, 1, 4, 5, 9, 10, 11, 12, 13):                      # null pointers
        bad = list(ok); bad[i] = None
        assert f(*bad) == -1, i
    for i, v in ((2, -1), (3, 0), (6, 0), (7, -3)):                # negative / empty sizes
        bad = list(ok); bad[i] = v
        assert f(*bad) == -1, i
    bad = list(ok); bad[8] = 128                                   # coarse width other than 256
    assert f(*bad) == -4
    for i in (0, 1, 4, 5, 12, 13):                                 # misaligned pointers
        bad = list(ok); bad[i] = 40
        assert f(*bad) == -5, i
    bad = list(ok); bad[14] = ws - 1
    assert f(*bad) == -3
    bad = list(ok); bad[14] = h.pope_fine_merge_workspace_bytes(3)
    assert f(*bad) == -3
    bad = list(ok); bad[2] = 0
    assert f(*bad) == 0


def test_matcher_fine_fp32_flag_wiring():
    cfg = pope_b200.make_default_cfg()
    stock = pope_b200.Matcher(cfg)
    m = pope_b200.Matcher(cfg, fine_cuda_fp32=True)
    assert list(m.state_dict()) == list(stock.state_dict()) and len(m.state_dict()) == 211
    assert m.fine_cuda_fp32 and m.loftr_fine.cuda_fp32 and m.fine_preprocess.cuda_fp32 and m.loftr_fine.inplace
    assert not m.fine_cuda_bf16 and not m.fine_preprocess.cuda_bf16
    assert not stock.fine_cuda_fp32 and not stock.loftr_fine.cuda_fp32 and not stock.fine_preprocess.cuda_fp32
    with pytest.raises(ValueError):
        pope_b200.Matcher(cfg, fine_cuda_bf16=True, fine_cuda_fp32=True)
    with pytest.raises(ValueError):
        m.set_fine_cuda_bf16(True)
    b = pope_b200.Matcher(cfg, fine_cuda_bf16=True)
    with pytest.raises(ValueError):
        b.set_fine_cuda_fp32(True)
    b.set_fine_cuda_bf16(False)
    b.set_fine_cuda_fp32(True)                                     # switching over is fine
    assert b.fine_cuda_fp32 and not b.fine_cuda_bf16 and b.loftr_fine.inplace
    b.set_fine_cuda_fp32(False)
    assert not b.loftr_fine.cuda_fp32 and not b.fine_preprocess.cuda_fp32 and not b.loftr_fine.inplace
    for coarse in ({"coarse_cuda_bf16": True}, {"coarse_cuda_fp32": True}):      # combines with either coarse flag
        c = pope_b200.Matcher(cfg, fine_cuda_fp32=True, **coarse)
        assert c.fine_cuda_fp32 and c.loftr_fine.cuda_fp32
    for key, val in (("d_model", 64), ("nhead", 4), ("attention", "full")):
        bad = copy.deepcopy(cfg)
        bad["fine"][key] = val
        with pytest.raises(NotImplementedError):
            pope_b200.Matcher(bad, fine_cuda_fp32=True)
        pope_b200.Matcher(bad).set_fine_cuda_fp32(False)


def test_cuda_fp32_mode_leaves_cpu_tensors_to_the_stock_layers():
    ref = _model(["self", "cross"], seed=2)
    m = FineTransformerB200(_fine_cfg(["self", "cross"])).eval()
    m.load_state_dict(ref.state_dict())
    m.cuda_fp32 = True
    m.inplace = True
    f0, f1 = _windows(1, 7)
    with torch.no_grad():
        got, want = m(f0, f1), ref(f0, f1)
    assert got[0].dtype == torch.float32 and torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


# ---- GPU ------------------------------------------------------------------------------------------------------------

DEV = torch.device("cuda:0")


def _stock_fp32(fn):
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            return fn()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


def _tf_errors(m, f0, f1):
    """(CUDA fp32, stock fp32 with TF32 off, CUDA bf16) errors against the stock module in float64, per side."""
    names = m.layer_names
    ref = copy.deepcopy(m).to(DEV).double()
    with torch.no_grad():
        want = ref(f0.to(DEV, torch.float64), f1.to(DEV, torch.float64))
    del ref
    sm = copy.deepcopy(m).to(DEV)
    stock = _stock_fp32(lambda: sm(f0.to(DEV), f1.to(DEV)))
    sd = [layer.state_dict() for layer in m.layers]
    p32 = torch.cat([ops.pack_fine_layer(l, DEV, dtype=torch.float32) for l in sd])
    got = ops.fine_transformer(f0.to(DEV).contiguous(), f1.to(DEV).contiguous(), p32, names)
    p16 = torch.cat([ops.pack_fine_layer(l, DEV) for l in sd])
    b16 = ops.fine_transformer(f0.to(DEV, torch.bfloat16), f1.to(DEV, torch.bfloat16), p16, names)
    assert got[0].dtype == torch.float32 and got[0].shape == f0.shape
    return [(_rel_err(got[s], want[s]), _rel_err(stock[s], want[s]), _rel_err(b16[s], want[s])) for s in range(2)]


def _assert_bars(tag, errs):
    for side, (e_cuda, e_stock, e_bf16) in enumerate(errs):
        print(f"{tag} side {side}: cuda fp32 rms {e_cuda[0]:.3e} max {e_cuda[1]:.3e} | "
              f"stock fp32 rms {e_stock[0]:.3e} max {e_stock[1]:.3e} | cuda bf16 rms {e_bf16[0]:.3e} max {e_bf16[1]:.3e} | "
              f"ratios vs stock {e_cuda[0] / e_stock[0]:.2f} / {e_cuda[1] / e_stock[1]:.2f}, "
              f"bf16 / cuda {e_bf16[0] / e_cuda[0]:.0f} / {e_bf16[1] / e_cuda[1]:.0f}")
        for k in range(2):
            assert e_cuda[k] <= STOCK_FACTOR * e_stock[k], (side, e_cuda, e_stock)
            assert BF16_FACTOR * e_cuda[k] <= e_bf16[k], (side, e_cuda, e_bf16)


CASES = [  # (windows, layer schedule, sigma, tokens): one window, a few, a ragged 128-row tile, >= 20 000, 7 x 7 windows
    (1, ["self"], 1.0, 25), (5, ["cross"], 1.0, 25), (1003, ["self", "cross"], 1.0, 25),
    (1003, ["cross", "self", "cross"], 0.1, 25), (20000, ["self", "cross"], 1.0, 25), (5, ["self", "cross"], 30.0, 25),
    (300, ["self", "cross"], 1.0, 49), (1003, ["self"], 30.0, 49),
]


@pytest.mark.gpu
@pytest.mark.parametrize("m,names,sigma,ww", CASES)
def test_cuda_fp32_fine_transformer_error_within_stock_fp32(m, names, sigma, ww):
    model = _model(names, seed=m + ww)
    f0, f1 = _windows(17 + m, m, ww, sigma)
    _assert_bars(f"{names} m={m} ww={ww} sigma={sigma}", _tf_errors(model, f0, f1))


def _merge_inputs(seed, m, ww=25, n=2, L=96, S=80, sigma=1.0):
    gen = torch.Generator().manual_seed(seed)
    w0, w1 = _windows(seed, m, ww, sigma)
    fc0, fc1 = sigma * torch.randn(n, L, 256, generator=gen), sigma * torch.randn(n, S, 256, generator=gen)
    ids = (torch.randint(0, n, (m,), generator=gen), torch.randint(0, L, (m,), generator=gen),
           torch.randint(0, S, (m,), generator=gen))
    return w0, w1, fc0, fc1, ids


def _stock_merge(pre, w0, w1, fc0, fc1, ids):
    """fine_preprocess.py:50-57 with the given modules (in the modules' dtype)."""
    b, i, j = ids
    m, ww = w0.shape[0], w0.shape[1]
    c = pre.down_proj(torch.cat([fc0[b, i], fc1[b, j]], 0))
    merged = pre.merge_feat(torch.cat([torch.cat([w0, w1], 0), c[:, None, :].expand(-1, ww, -1)], -1))
    return merged[:m], merged[m:]


@pytest.mark.gpu
@pytest.mark.parametrize("m,ww,sigma", [(1, 25, 1.0), (5, 25, 30.0), (1003, 25, 0.1), (20000, 25, 1.0), (300, 49, 1.0)])
def test_cuda_fp32_fine_merge_coarse_error_within_stock_fp32(m, ww, sigma):
    pre = _pre(seed=m)
    w0, w1, fc0, fc1, ids = _merge_inputs(5 + m, m, ww, sigma=sigma)
    dids = [t.to(DEV) for t in ids]
    with torch.no_grad():
        want = _stock_merge(copy.deepcopy(pre).to(DEV).double(), w0.to(DEV).double(), w1.to(DEV).double(),
                            fc0.to(DEV).double(), fc1.to(DEV).double(), dids)
    sp = copy.deepcopy(pre).to(DEV)
    stock = _stock_fp32(lambda: _stock_merge(sp, w0.to(DEV), w1.to(DEV), fc0.to(DEV), fc1.to(DEV), dids))
    sd = pre.state_dict()
    got = ops.fine_merge_coarse(w0.to(DEV), w1.to(DEV), fc0.to(DEV), fc1.to(DEV), *dids,
                                ops.pack_fine_pre(sd, DEV, dtype=torch.float32))
    bf = torch.bfloat16
    b16 = ops.fine_merge_coarse(w0.to(DEV, bf), w1.to(DEV, bf), fc0.to(DEV, bf), fc1.to(DEV, bf), *dids,
                                ops.pack_fine_pre(sd, DEV))
    _assert_bars(f"merge m={m} ww={ww} sigma={sigma}",
                 [(_rel_err(got[s], want[s]), _rel_err(stock[s], want[s]), _rel_err(b16[s], want[s])) for s in range(2)])


def _bf16_bits(bits):
    return torch.from_numpy(bits.view(np.int16).copy()).view(torch.bfloat16).float()


@pytest.mark.gpu
def test_cuda_fp32_fine_level_vs_reference_fixtures():
    """The fixtures of the unmodified reference (bf16-representable weights and inputs, fp32 arithmetic): the fp32 path
    meets a bar 1 000x tighter than the bf16 path's 1.5e-2."""
    g = {}
    for name in ("fine_transformer.npz", "fine_merge_coarse.npz"):
        g.update(np.load(os.path.join(GOLDEN, name)))
    meta = json.loads(str(g["meta"]))
    conv = lambda v: _bf16_bits(v) if v.dtype == np.uint16 else torch.from_numpy(v)
    layers = [{k[len(f"tf.layers.{l}."):]: conv(v) for k, v in g.items() if k.startswith(f"tf.layers.{l}.")}
              for l in range(len(meta["layer_names"]))]
    pre_sd = {k[4:]: conv(v) for k, v in g.items() if k.startswith("pre.") and ("weight" in k or "bias" in k)}
    gen = torch.Generator().manual_seed(meta["input_seed"])
    f0 = torch.randn(meta["m"], 25, 128, generator=gen).to(torch.bfloat16).float()
    f1 = torch.randn(meta["m"], 25, 128, generator=gen).to(torch.bfloat16).float()
    k = meta["kept"]
    d0, d1 = f0.to(DEV), f1.to(DEV)
    ops.fine_transformer(d0, d1, torch.cat([ops.pack_fine_layer(sd, DEV, dtype=torch.float32) for sd in layers]),
                         meta["layer_names"])
    for got, key in ((d0, "out0"), (d1, "out1")):
        rms, mx = _rel_err(got[:k].cpu(), torch.from_numpy(g[key]))
        print(f"fixture {key}: rms {rms:.3e} max {mx:.3e}")
        assert rms < 1.5e-5 and mx < 1e-4, (key, rms, mx)
    ids = [torch.from_numpy(g["pre." + n]).to(DEV) for n in ("b_ids", "i_ids", "j_ids")]
    d0, d1 = f0.to(DEV), f1.to(DEV)
    ops.fine_merge_coarse(d0, d1, _bf16_bits(g["pre.feat_c0"]).to(DEV), _bf16_bits(g["pre.feat_c1"]).to(DEV), *ids,
                          ops.pack_fine_pre(pre_sd, DEV, dtype=torch.float32))
    for got, key in ((d0, "pre.merged0"), (d1, "pre.merged1")):
        rms, mx = _rel_err(got[:k].cpu(), torch.from_numpy(g[key]))
        print(f"fixture {key}: rms {rms:.3e} max {mx:.3e}")
        assert rms < 1.5e-5 and mx < 1e-4, (key, rms, mx)


@pytest.mark.gpu
def test_cuda_fp32_fine_level_is_deterministic_and_window_independent():
    names = ["self", "cross"]
    p32 = torch.cat([ops.pack_fine_layer(l.state_dict(), DEV, dtype=torch.float32) for l in _model(names, 4).layers])
    pre = ops.pack_fine_pre(_pre(4).state_dict(), DEV, dtype=torch.float32)
    w0, w1, fc0, fc1, ids = _merge_inputs(8, 2000)
    w0, w1, fc0, fc1 = w0.to(DEV), w1.to(DEV), fc0.to(DEV), fc1.to(DEV)
    ids = [t.to(DEV) for t in ids]

    def run(sel):
        a, b = w0[sel].clone(), w1[sel].clone()
        ops.fine_merge_coarse(a, b, fc0, fc1, *[t[sel] for t in ids], pre)
        return ops.fine_transformer(a, b, p32, names)

    full = torch.arange(2000, device=DEV)
    r1, r2 = run(full), run(full)
    assert torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1])
    for sel in (torch.arange(37, 1181, device=DEV), torch.tensor([1999, 3, 500], device=DEV)):
        sub = run(sel)
        assert torch.equal(sub[0], r1[0][sel]) and torch.equal(sub[1], r1[1][sel])


@pytest.mark.gpu
def test_cuda_fp32_fine_level_empty_in_place_copy_and_errors():
    names = ["self", "cross"]
    model = _model(names, 6)
    p32 = torch.cat([ops.pack_fine_layer(l.state_dict(), DEV, dtype=torch.float32) for l in model.layers])
    p16 = torch.cat([ops.pack_fine_layer(l.state_dict(), DEV) for l in model.layers])
    e0 = torch.empty(0, 25, 128, device=DEV)
    r0, r1 = ops.fine_transformer(e0, e0.clone(), p32, names)
    assert r0.shape == (0, 25, 128) and r0.dtype == torch.float32
    fc = torch.randn(1, 16, 256, device=DEV)
    noid = torch.empty(0, dtype=torch.int64, device=DEV)
    pre32 = ops.pack_fine_pre(_pre().state_dict(), DEV, dtype=torch.float32)
    assert ops.fine_merge_coarse(e0, e0.clone(), fc, fc, noid, noid, noid, pre32)[0].shape == (0, 25, 128)
    f0, f1 = _windows(3, 40)
    a, b = f0.to(DEV), f1.to(DEV)
    r0, r1 = ops.fine_transformer(a, b, p32, names)                # in place
    assert r0.data_ptr() == a.data_ptr() and r1.data_ptr() == b.data_ptr()
    m = FineTransformerB200(_fine_cfg(names)).eval().to(DEV)       # the module works on copies unless `inplace`
    m.load_state_dict(model.state_dict())
    m.cuda_fp32 = True
    x0, x1 = f0.to(DEV), f1.to(DEV)
    with torch.no_grad():
        y0, y1 = m(x0, x1)
    assert torch.equal(x0.cpu(), f0) and torch.equal(x1.cpu(), f1)
    assert torch.equal(y0, a) and torch.equal(y1, b) and y0.dtype == torch.float32
    m.inplace = True
    with torch.no_grad():
        z0, _ = m(x0, x1)
    assert z0.data_ptr() == x0.data_ptr() and torch.equal(x0, a)
    z = torch.zeros(2, 25, 128, device=DEV)
    for bad in (lambda: ops.fine_transformer(z, z.clone(), p16, names),                    # fp32 windows, bf16 packing
                lambda: ops.fine_transformer(z.bfloat16(), z.bfloat16(), p32, names),      # bf16 windows, fp32 packing
                lambda: ops.fine_transformer(z, z.bfloat16(), p32, names),                 # mixed dtypes
                lambda: ops.fine_transformer(z, z.clone(), p32, names, m_dev=torch.ones(1, dtype=torch.int32, device=DEV)),
                lambda: ops.fine_merge_coarse(z, z.clone(), fc, fc, *[torch.zeros(2, dtype=torch.int64, device=DEV)] * 3,
                                              ops.pack_fine_pre(_pre().state_dict(), DEV)),
                lambda: ops.fine_merge_coarse(z, z.clone(), fc, fc, *[torch.zeros(2, dtype=torch.int64, device=DEV)] * 3,
                                              pre32, m_dev=torch.ones(1, dtype=torch.int32, device=DEV))):
        with pytest.raises(_lib.PopeError):
            bad()


def _steps_3_to_5(mm, f0, f1, ff0, ff1, hw, n):
    h, w = hw
    data = {"hw0_i": torch.Size([h * 8, w * 8]), "hw1_i": torch.Size([h * 8, w * 8]), "hw0_c": torch.Size([h, w]),
            "hw1_c": torch.Size([h, w]), "hw0_f": torch.Size([h * 4, w * 4]), "hw1_f": torch.Size([h * 4, w * 4]), "bs": n}
    with torch.no_grad():
        x0, x1 = mm.loftr_coarse(f0, f1)
        mm.coarse_matching(x0, x1, data)
        if x0.dtype != ff0.dtype:
            x0, x1 = x0.to(ff0.dtype), x1.to(ff0.dtype)
        w0, w1 = mm.fine_preprocess(ff0, ff1, x0, x1, data)
        if w0.size(0) != 0:
            w0, w1 = mm.loftr_fine(w0, w1)
        mm.fine_matching(w0, w1, data)
    return data


@pytest.mark.gpu
@pytest.mark.parametrize("coarse,concat", [({}, True), ({}, False), ({"coarse_cuda_fp32": True}, True)],
                         ids=["stock_coarse", "no_concat", "coarse_cuda_fp32"])
def test_matcher_fp32_fine_level_vs_stock_fp32_flow(coarse, concat):
    """Steps 3-5 of Matcher.forward with `fine_cuda_fp32=True` (CUDA FinePreprocess Linears and fine transformer at fp32
    accuracy) against the stock fp32 flow on the GPU with TF32 off, on synthetic features with planted correspondences
    (with coarse_cuda_fp32 they go through the coarse transformer first): the match ids are identical and the refined
    coordinates agree to 1e-3 px (the bf16 fine level's bar is 0.3 px)."""
    cfg = pope_b200.make_default_cfg()
    cfg["fine_concat_coarse_feat"] = concat
    torch.manual_seed(0)
    stock = pope_b200.Matcher(cfg).eval().to(DEV)
    fast = pope_b200.Matcher(cfg, fine_cuda_fp32=True, **coarse).eval().to(DEV)
    fast.load_state_dict(stock.state_dict())
    if not coarse:                                   # no coarse transformer: the planted features go to the matcher as is
        stock.loftr_coarse.layer_names = fast.loftr_coarse.layer_names = []
    h, w, n = 20, 24, 2
    ff0, ff1 = synth.fine_feature_maps(62, n, h * 4, w * 4, 128, channels_last=False)
    ff0, ff1 = ff0.to(DEV), ff1.to(DEV)
    for sigma in (0.85, 4.0, 16.0, 32.0):
        f0, f1 = synth.coarse_features(61, n, h * w, h * w, 256, sigma=sigma)
        want = _stock_fp32(lambda: _steps_3_to_5(stock, f0.to(DEV), f1.to(DEV), ff0, ff1, (h, w), n))
        if want["b_ids"].numel() > 200:
            break
    got = _steps_3_to_5(fast, f0.to(DEV), f1.to(DEV), ff0, ff1, (h, w), n)
    assert want["b_ids"].numel() > 200, sigma
    assert list(got) == list(want)
    for k in ("b_ids", "i_ids", "j_ids"):
        assert torch.equal(got[k], want[k]), k
    for k, v in want.items():
        if isinstance(v, torch.Tensor):
            assert got[k].dtype == v.dtype, k
    d = (got["mkpts1_f"] - want["mkpts1_f"]).abs()
    print(f"{coarse} concat={concat} sigma={sigma}: {want['b_ids'].numel()} matches, |d mkpts1_f| mean "
          f"{float(d.mean()):.2e} max {float(d.max()):.2e} px")
    assert float(d.max()) < 1e-3, float(d.max())
