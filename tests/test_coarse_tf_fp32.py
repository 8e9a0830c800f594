"""Coarse-level transformer at fp32 accuracy (csrc/coarse_tf.cu, coarse_gemm_kernel<true>): pope_coarse_transformer_f32,
`ops.pack_coarse_layer(..., dtype=torch.float32)`, `ops.coarse_transformer` on fp32 features,
`CoarseTransformerB200.cuda_fp32` and `Matcher(config, coarse_cuda_fp32=True)`.

Every GEMM operand is split into three bf16 terms a = a1 + a2 + a3 and the six significant products are accumulated in
fp32, so the path is held to the fp32 modules, not to bf16: against the stock module run in float64 (with the same full
fp32 weights), its error (rms and max, relative to the output RMS) must stay within STOCK_FACTOR x that of the stock
fp32 modules (TF32 off) and BF16_FACTOR x below that of the bf16 CUDA transformer on the same case.  Both factors are
chosen bars, not measurements; the measured ratios are printed.
"""
import copy
import os
import re

import pytest
import torch

import pope_b200
from pope_b200 import _lib, ops, synth
from pope_b200.feature_net import CoarseTransformerB200, LocalFeatureTransformer
from tests import parity_utils

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT = ["self", "cross"] * 4
# measured on a B200: 2.2-4.6x the stock fp32 error (rms and max), 1 700-65 000x below the bf16 path's (DESIGN 4.10)
STOCK_FACTOR = 6.0
BF16_FACTOR = 100.0
MATS = (("qkv", (768, 256)), ("merge.weight", (256, 256)), ("mlp.0.weight", (512, 512)), ("mlp.2.weight", (256, 512)))


def _coarse_cfg(names=None):
    cfg = copy.deepcopy(pope_b200.make_default_cfg()["coarse"])
    if names is not None:
        cfg["layer_names"] = list(names)
    return cfg


def _model(names, seed=0):
    """A stock coarse transformer with its own fp32 (xavier) weights and perturbed LayerNorm parameters."""
    torch.manual_seed(seed)
    m = LocalFeatureTransformer(_coarse_cfg(names)).eval()
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if p.dim() == 1:
                p.copy_((1 if name.endswith("weight") else 0) + (0.2 if name.endswith("weight") else 0.1) *
                        torch.randn(p.shape, generator=gen))
    return m


def _matrix(sd, key):
    if key == "qkv":
        return torch.cat([sd["q_proj.weight"], sd["k_proj.weight"], sd["v_proj.weight"]])
    return sd[key]


def _rel_err(got, want):
    rms = want.pow(2).mean().sqrt()
    d = (got.double() - want).abs()
    return float(d.pow(2).mean().sqrt() / rms), float(d.max() / rms)


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_pack_fp32_layer_puts_every_plane_at_the_header_offsets():
    header = open(os.path.join(ROOT, "include", "pope_b200.h")).read()
    assert int(re.search(r"#define POPE_COARSE_TF_F32_LAYER_BYTES (\d+)", header).group(1)) == _lib.COARSE_TF_F32_LAYER_BYTES
    sd = _model(["self"]).layers[0].state_dict()
    packed = ops.pack_coarse_layer(sd, "cpu", dtype=torch.float32)
    assert packed.dtype == torch.uint8 and packed.numel() == _lib.COARSE_TF_F32_LAYER_BYTES
    off = 0
    for (key, shp), doc in zip(MATS, (0, 1179648, 1572864, 3145728)):
        assert off == doc, key                                    # the offsets written in the header
        w = _matrix(sd, key)
        n = shp[0] * shp[1] * 2
        planes = [packed[off + p * n:off + (p + 1) * n].view(torch.bfloat16).view(shp) for p in range(3)]
        assert torch.equal(planes[0], w.to(torch.bfloat16)), key
        assert torch.equal((planes[0].float() + planes[1].float()) + planes[2].float(), w), key
        off += 3 * n
    assert off == 3932160
    for key in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"):
        assert torch.equal(packed[off:off + 1024].view(torch.float32), sd[key]), key
        off += 1024
    # the bf16 layout (the default) is unchanged
    old = torch.cat([torch.cat([sd[k].to(torch.bfloat16).reshape(-1) for k in
                                ("q_proj.weight", "k_proj.weight", "v_proj.weight", "merge.weight", "mlp.0.weight",
                                 "mlp.2.weight")]).view(torch.uint8),
                     torch.cat([sd[k].reshape(-1) for k in ("norm1.weight", "norm1.bias", "norm2.weight",
                                                            "norm2.bias")]).view(torch.uint8)])
    assert torch.equal(ops.pack_coarse_layer(sd, "cpu"), old)
    assert torch.equal(ops.pack_coarse_layer(sd, "cpu", dtype=torch.bfloat16), old)
    with pytest.raises(_lib.PopeError):
        ops.pack_coarse_layer(sd, "cpu", dtype=torch.float16)


@pytest.mark.parametrize("kind", ["random", "large", "tiny", "subnormal"])
def test_three_plane_split_holds_the_fp32_value(kind):
    gen = torch.Generator().manual_seed(4)
    n = 1 << 16
    if kind == "random":
        w = torch.randn(n, generator=gen)
    else:   # random signs and mantissas over a range of binary exponents
        lo, hi = {"large": (100, 127), "tiny": (-110, -100), "subnormal": (-149, -126)}[kind]
        e = torch.randint(lo, hi, (n,), generator=gen).double()
        m = 1 + torch.rand(n, generator=gen, dtype=torch.float64)
        s = torch.randint(0, 2, (n,), generator=gen).double() * 2 - 1
        w = (s * m * torch.exp2(e)).float()
    if kind == "subnormal":
        assert bool((w.abs() < 2.0 ** -126).all()) and bool((w != 0).any())
    w1, w2, w3 = ops.split3_bf16(w)
    total = (w1.float() + w2.float()) + w3.float()
    assert torch.equal(w1.double() + w2.double() + w3.double(), total.double())    # the fp32 sum is exact
    if kind == "subnormal":
        # below 2^-110 the third term reaches the bf16 subnormal range (spacing 2^-133): the split is w to half a spacing
        assert float((total.double() - w.double()).abs().max()) <= 2.0 ** -134
    else:
        assert torch.equal(total, w)


def test_six_products_stay_within_the_fp32_error_model():
    """Host restatement of the kernel's arithmetic: a1w1 + a2w1 + a3w1 + a1w2 + a2w2 + a1w3 against the float64
    product.  The dropped products a2w3, a3w2, a3w3 are at most 2^-24 |a||w| each (|a2| <= 2^-8 |a|, |a3| <= 2^-16 |a|),
    so with float64 accumulation |error| <= 2.01 * 2^-24 * sum |a||w|; with fp32 accumulation (as in TMEM) add the
    summation's own K * 2^-24."""
    gen = torch.Generator().manual_seed(9)
    for K, scale in ((256, 1.0), (512, 30.0), (512, 1e-3)):
        a = scale * torch.randn(96, K, generator=gen)
        w = torch.randn(200, K, generator=gen) / K ** 0.5
        ap, wp = ops.split3_bf16(a), ops.split3_bf16(w)
        pairs = ((0, 0), (1, 0), (2, 0), (0, 1), (1, 1), (0, 2))
        exact = a.double() @ w.double().T
        bound = (a.double().abs() @ w.double().abs().T) * 2.0 ** -24
        six64 = sum(ap[i].double() @ wp[j].double().T for i, j in pairs)
        assert float(((six64 - exact).abs() / bound).max()) <= 2.01, (K, scale)
        six32 = sum(ap[i].float() @ wp[j].float().T for i, j in pairs).double()
        assert float(((six32 - exact).abs() / bound).max()) <= 2.01 + K, (K, scale)
        # and it is an fp32-grade result, far from a single bf16 product
        one = (a.to(torch.bfloat16).double() @ w.to(torch.bfloat16).double().T)
        assert float((six32 - exact).abs().max()) * 1000 < float((one - exact).abs().max())


def test_f32_entry_points_reject_bad_arguments_before_touching_the_gpu():
    h = _lib.lib()
    kinds = (_lib.C.c_int * 2)(0, 1)
    ws = h.pope_coarse_tf_f32_workspace_bytes(2, 64, 48)
    assert ws > h.pope_coarse_tf_workspace_bytes(2, 64, 48) > 0
    assert h.pope_coarse_tf_f32_workspace_bytes(0, 64, 48) == 0 and h.pope_coarse_tf_f32_workspace_bytes(2, 0, 48) == 0
    assert h.pope_coarse_tf_f32_workspace_bytes(2, 64, -1) == 0 and h.pope_coarse_tf_f32_workspace_bytes(70000, 64, 48) == 0
    # feat0, feat1, n_pairs, L, S, weights, n_layers, layer_kinds, workspace, workspace_bytes, stream
    ok = [16, 16, 2, 64, 48, 16, 2, kinds, 16, ws, None]
    f = h.pope_coarse_transformer_f32
    for i in (0, 1, 5, 7, 8):                                      # null features, weights, kinds and workspace
        bad = list(ok); bad[i] = None
        assert f(*bad) == -1, i
    for i, v in ((2, -1), (3, 0), (4, 0), (6, -1)):                # negative / empty sizes
        bad = list(ok); bad[i] = v
        assert f(*bad) == -1, i
    bad = list(ok); bad[7] = (_lib.C.c_int * 2)(1, 3)              # layer kind other than 'self' / 'cross'
    assert f(*bad) == -1
    for i in (0, 1, 5, 8):                                         # misaligned pointers
        bad = list(ok); bad[i] = 40
        assert f(*bad) == -5, i
    bad = list(ok); bad[9] = ws - 1                                # workspace too small (the bf16 size, too)
    assert f(*bad) == -3
    bad = list(ok); bad[9] = h.pope_coarse_tf_workspace_bytes(2, 64, 48)
    assert f(*bad) == -3
    bad = list(ok); bad[2] = 70000                                 # more pairs than the attention grid holds
    assert f(*bad) == -4
    bad = list(ok); bad[2] = 0                                     # no pairs: a no-op
    assert f(*bad) == 0


def test_matcher_fp32_flag_wiring():
    cfg = pope_b200.make_default_cfg()
    stock = pope_b200.Matcher(cfg)
    m = pope_b200.Matcher(cfg, coarse_cuda_fp32=True)
    assert list(m.state_dict()) == list(stock.state_dict()) and len(m.state_dict()) == 211
    assert m.coarse_cuda_fp32 and m.loftr_coarse.cuda_fp32 and not m.coarse_cuda_bf16
    assert not stock.coarse_cuda_fp32 and not stock.loftr_coarse.cuda_fp32
    with pytest.raises(ValueError):
        pope_b200.Matcher(cfg, coarse_cuda_bf16=True, coarse_cuda_fp32=True)
    with pytest.raises(ValueError):
        m.set_coarse_cuda_bf16(True)
    b = pope_b200.Matcher(cfg, coarse_cuda_bf16=True)
    with pytest.raises(ValueError):
        b.set_coarse_cuda_fp32(True)
    b.set_coarse_cuda_bf16(False)
    b.set_coarse_cuda_fp32(True)                                  # switching over is fine
    assert b.coarse_cuda_fp32 and not b.coarse_cuda_bf16 and b.loftr_coarse.inplace
    b.set_coarse_cuda_fp32(False)
    assert not b.loftr_coarse.cuda_fp32 and not b.loftr_coarse.inplace
    for key, val in (("d_model", 128), ("nhead", 4), ("attention", "full")):
        bad = copy.deepcopy(cfg)
        bad["coarse"][key] = val
        if key == "d_model":
            bad["fine"]["d_model"] = 128
        with pytest.raises(NotImplementedError):
            pope_b200.Matcher(bad, coarse_cuda_fp32=True)
        pope_b200.Matcher(bad).set_coarse_cuda_fp32(False)


def test_cuda_fp32_mode_leaves_cpu_tensors_to_the_stock_layers():
    ref = _model(["self", "cross"], seed=2)
    m = CoarseTransformerB200(_coarse_cfg(["self", "cross"])).eval()
    m.load_state_dict(ref.state_dict())
    m.cuda_fp32 = True
    gen = torch.Generator().manual_seed(1)
    f0, f1 = torch.randn(2, 30, 256, generator=gen), torch.randn(2, 20, 256, generator=gen)
    with torch.no_grad():
        got, want = m(f0, f1), ref(f0, f1)
    assert got[0].dtype == torch.float32 and torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _errors(m, f0, f1, dev):
    """(CUDA fp32, stock fp32 with TF32 off, CUDA bf16) errors against the stock module in float64, per side."""
    names = m.layer_names
    ref = copy.deepcopy(m).to(dev).double()
    with torch.no_grad():
        want = ref(f0.to(dev, torch.float64), f1.to(dev, torch.float64))
    del ref
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        sm = copy.deepcopy(m).to(dev)
        with torch.no_grad():
            stock = sm(f0.to(dev), f1.to(dev))
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    sd = [layer.state_dict() for layer in m.layers]
    p32 = torch.cat([ops.pack_coarse_layer(l, dev, dtype=torch.float32) for l in sd])
    got = ops.coarse_transformer(f0.to(dev).contiguous(), f1.to(dev).contiguous(), p32, names)
    p16 = torch.cat([ops.pack_coarse_layer(l, dev) for l in sd])
    b16 = ops.coarse_transformer(f0.to(dev, torch.bfloat16), f1.to(dev, torch.bfloat16), p16, names)
    assert got[0].dtype == torch.float32 and got[0].shape == f0.shape and got[1].shape == f1.shape
    return [(_rel_err(got[s], want[s]), _rel_err(stock[s], want[s]), _rel_err(b16[s], want[s])) for s in range(2)]


CASES = [  # (n pairs, L, S, sigma): one / several pairs, L != S, ragged 128-row tiles, small / unit / large scales
    (1, 4800, 4800, 1.0), (3, 4800, 4800, 1.0), (1, 4800, 1024, 1.0), (2, 63, 1000, 0.1), (2, 1000, 200, 4.0),
    (1, 4800, 1024, 30.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("names", [DEFAULT, ["self"]], ids=["default", "self"])
@pytest.mark.parametrize("n,L,S,sigma", CASES)
def test_cuda_fp32_coarse_transformer_error_within_stock_fp32(names, n, L, S, sigma):
    m = _model(names, seed=L + S)
    f0, f1 = synth.coarse_features(13, n, L, S, sigma=sigma)
    for side, (e_cuda, e_stock, e_bf16) in enumerate(_errors(m, f0, f1, torch.device("cuda"))):
        print(f"{names} n={n} L={L} S={S} sigma={sigma} side {side}: cuda fp32 rms {e_cuda[0]:.3e} max {e_cuda[1]:.3e} | "
              f"stock fp32 rms {e_stock[0]:.3e} max {e_stock[1]:.3e} | cuda bf16 rms {e_bf16[0]:.3e} max {e_bf16[1]:.3e} | "
              f"ratios vs stock {e_cuda[0] / e_stock[0]:.2f} / {e_cuda[1] / e_stock[1]:.2f}, "
              f"bf16 / cuda {e_bf16[0] / e_cuda[0]:.0f} / {e_bf16[1] / e_cuda[1]:.0f}")
        for k in range(2):
            assert e_cuda[k] <= STOCK_FACTOR * e_stock[k], (side, e_cuda, e_stock)
            assert BF16_FACTOR * e_cuda[k] <= e_bf16[k], (side, e_cuda, e_bf16)


@pytest.mark.gpu
def test_cuda_fp32_coarse_transformer_is_deterministic_and_batch_independent():
    dev = torch.device("cuda")
    m = _model(DEFAULT, seed=7)
    packed = torch.cat([ops.pack_coarse_layer(l.state_dict(), dev, dtype=torch.float32) for l in m.layers])
    f0, f1 = synth.coarse_features(3, 3, 2400, 1500)
    g0, g1 = synth.coarse_features(4, 3, 2400, 1500)
    a = ops.coarse_transformer(f0.to(dev), f1.to(dev), packed, DEFAULT)
    b = ops.coarse_transformer(f0.to(dev), f1.to(dev), packed, DEFAULT)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for p in range(3):
        alone = ops.coarse_transformer(f0[p:p + 1].to(dev), f1[p:p + 1].to(dev), packed, DEFAULT)
        mixed0, mixed1 = g0.clone(), g1.clone()
        mixed0[p], mixed1[p] = f0[p], f1[p]
        batch = ops.coarse_transformer(mixed0.to(dev), mixed1.to(dev), packed, DEFAULT)
        assert torch.equal(batch[0][p], alone[0][0]) and torch.equal(batch[1][p], alone[1][0]), p


@pytest.mark.gpu
def test_coarse_transformer_rejects_a_dtype_packing_mismatch():
    dev = torch.device("cuda")
    sd = _model(["self"]).layers[0].state_dict()
    p16, p32 = ops.pack_coarse_layer(sd, dev), ops.pack_coarse_layer(sd, dev, dtype=torch.float32)
    f0, f1 = torch.randn(1, 64, 256, device=dev), torch.randn(1, 64, 256, device=dev)
    with pytest.raises(_lib.PopeError):
        ops.coarse_transformer(f0, f1, p16, ["self"])
    with pytest.raises(_lib.PopeError):
        ops.coarse_transformer(f0.to(torch.bfloat16), f1.to(torch.bfloat16), p32, ["self"])
    with pytest.raises(_lib.PopeError):
        ops.coarse_transformer(f0, f1.to(torch.bfloat16), p32, ["self"])


def _images(dev, seed, hw0=(480, 640), hw1=(480, 640), n=1):
    gen = torch.Generator().manual_seed(seed)
    return {"image0": torch.rand(n, 1, *hw0, generator=gen).to(dev), "image1": torch.rand(n, 1, *hw1, generator=gen).to(dev)}


@pytest.mark.gpu
def test_matcher_fp32_only_att_fea_returns_fp32_features():
    dev = torch.device("cuda")
    torch.manual_seed(0)
    cfg = pope_b200.make_default_cfg()
    stock = pope_b200.Matcher(cfg).eval().to(dev)
    m = pope_b200.Matcher(cfg, coarse_cuda_fp32=True).eval().to(dev)
    m.load_state_dict(stock.state_dict())
    data = _images(dev, 1, (480, 640), (256, 256))
    with torch.no_grad():
        got0, got1 = m(dict(data), only_att_fea=True)
        want0, want1 = stock(dict(data), only_att_fea=True)
        c0, c1 = m.backbone(data["image0"])[0], m.backbone(data["image1"])[0]
        f0 = m.pos_encoding(c0).flatten(2).transpose(1, 2).contiguous()
        f1 = m.pos_encoding(c1).flatten(2).transpose(1, 2).contiguous()
        packed = torch.cat([ops.pack_coarse_layer(l.state_dict(), dev, dtype=torch.float32) for l in m.loftr_coarse.layers])
        k0, k1 = ops.coarse_transformer(f0, f1, packed, m.loftr_coarse.layer_names)
    assert got0.dtype == got1.dtype == torch.float32 and got0.shape == (1, 4800, 256) and got1.shape == (1, 1024, 256)
    assert torch.equal(got0, k0) and torch.equal(got1, k1)
    for g, w in ((got0, want0), (got1, want1)):
        assert _rel_err(g, w.double())[0] < 1e-5


@pytest.mark.gpu
def test_matcher_fp32_flag_with_the_bf16_fine_level_writes_the_stock_keys():
    dev = torch.device("cuda")
    torch.manual_seed(0)
    cfg = pope_b200.make_default_cfg()
    stock = pope_b200.Matcher(cfg).eval().to(dev)
    runs = []
    for flags in ({}, {"coarse_cuda_fp32": True}, {"coarse_cuda_fp32": True, "fine_cuda_bf16": True}):
        mm = pope_b200.Matcher(cfg, **flags).eval().to(dev)
        mm.load_state_dict(stock.state_dict())
        data = _images(dev, 2, (480, 640), (256, 256))
        with torch.no_grad():
            mm(data)
        runs.append(data)
    for d in runs[1:]:
        assert list(d) == list(runs[0])
        for k, v in runs[0].items():
            if isinstance(v, torch.Tensor):
                assert d[k].dtype == v.dtype, k
    masked = pope_b200.Matcher(cfg, coarse_cuda_fp32=True).eval().to(dev)
    data = _images(dev, 3, (64, 64), (64, 64))
    data["mask0"] = data["mask1"] = torch.ones(1, 8, 8, dtype=torch.bool, device=dev)
    with torch.no_grad(), pytest.raises(NotImplementedError):
        masked(data)


@pytest.mark.gpu
def test_planted_matches_through_the_fp32_cuda_coarse_transformer():
    """Planted-correspondence features through 8 random-weight layers, then the coarse matcher: the Matcher with
    coarse_cuda_fp32 against the stock fp32 Matcher flow.  sigma is raised until the stock flow keeps > 1000 matches."""
    dev = torch.device("cuda")
    cfg = pope_b200.make_default_cfg()
    m = _model(DEFAULT, seed=3)
    stock, fast = pope_b200.Matcher(cfg).eval().to(dev), pope_b200.Matcher(cfg, coarse_cuda_fp32=True).eval().to(dev)
    for mm in (stock, fast):
        mm.loftr_coarse.load_state_dict(m.state_dict())
    hw0_i, hw_c = (480, 640), (60, 80)
    lists = []
    for sigma in (4.0, 8.0, 16.0, 32.0):
        f0, f1 = synth.coarse_features(21, 1, 4800, 4800, sigma=sigma)
        lists, feats = [], []
        for mm in (stock, fast):
            data = {"bs": 1, "hw0_i": hw0_i, "hw1_i": hw0_i, "hw0_c": hw_c, "hw1_c": hw_c}
            with torch.no_grad():
                x0, x1 = mm.loftr_coarse(f0.to(dev), f1.to(dev))
                mm.coarse_matching(x0, x1, data)
            assert x0.dtype == torch.float32
            lists.append(data)
            feats.append((x0, x1))
        if lists[0]["b_ids"].numel() > 1000:
            break
    want, got = lists
    assert want["b_ids"].numel() > 1000, sigma
    _, mg = parity_utils.oracle_with_margins(feats[0][0].cpu(), feats[0][1].cpu(), hw0_i, hw_c, hw_c)
    cpu = lambda d: {k: d[k].cpu() for k in ("b_ids", "i_ids", "j_ids")}
    same, near, bad = parity_utils.compare_match_lists(cpu(got), cpu(want), mg)
    print(f"sigma {sigma}: stock fp32 matches {want['b_ids'].numel()}, cuda fp32 {got['b_ids'].numel()}: "
          f"{same} identical, {len(near)} near-tie / near-threshold, {len(bad)} unexplained")
    assert not bad, bad[:10]
    key = lambda d: {(int(b), int(i), int(j)): float(c) for b, i, j, c in
                     zip(d["b_ids"].tolist(), d["i_ids"].tolist(), d["j_ids"].tolist(), d["mconf"].tolist())}
    kw, kg = key(want), key(got)
    common = set(kw) & set(kg)
    assert len(common) >= same
    assert max(abs(kw[k] - kg[k]) for k in common) <= 1e-4
