"""Coarse-level transformer in bf16 (csrc/coarse_tf.cu): pope_coarse_transformer / pope_coarse_pos_encode,
`ops.coarse_transformer`, `feature_net.CoarseTransformerB200`, `Matcher(config, coarse_cuda_bf16=True)`.

There is no fixture from the unmodified reference at d_model 256 (the reference tree is not available to generate one).
The fp32 reference here is `oracle.pope_oracle.fine_transformer` / `encoder_layer`, which is generic in width and pinned
to the reference's own fixture at d_model 128 (tests/test_fine_tf.py); the CPU test below ties it to the stock
`LocalFeatureTransformer(config['coarse'])` at d_model 256.

The bf16 path has no absolute error bound known in advance.  Its yardstick is the stock modules cast to bf16 on the same
inputs: the CUDA path's error against the fp32 reference (rms and max, relative to the output RMS) must not exceed 1.25x
the stock bf16 modules' error.
"""
import copy
import os
import re

import pytest
import torch

import pope_b200
from oracle import pope_oracle as O
from pope_b200 import _lib, ops, synth
from pope_b200.feature_net import LocalFeatureTransformer
from tests import parity_utils

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT = ["self", "cross"] * 4


def _coarse_cfg(names=None):
    cfg = copy.deepcopy(pope_b200.make_default_cfg()["coarse"])
    if names is not None:
        cfg["layer_names"] = list(names)
    return cfg


def _stock(names, seed=0):
    """A stock coarse transformer with random weights rounded to bf16 and perturbed LayerNorm parameters (so that the
    fp32 reference, the stock bf16 modules and the CUDA path all use the same values)."""
    torch.manual_seed(seed)
    m = LocalFeatureTransformer(_coarse_cfg(names)).eval()
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if p.dim() > 1:
                p.copy_(p.to(torch.bfloat16).float())
            elif name.endswith("weight"):
                p.copy_(1 + 0.2 * torch.randn(p.shape, generator=gen))
            else:
                p.copy_(0.1 * torch.randn(p.shape, generator=gen))
    return m


def _layers(m):
    return [{k: v.detach().clone() for k, v in layer.state_dict().items()} for layer in m.layers]


def _rel_err(got, want):
    rms = want.pow(2).mean().sqrt()
    d = (got.float() - want).abs()
    return float(d.pow(2).mean().sqrt() / rms), float(d.max() / rms)


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_oracle_matches_stock_coarse_transformer_at_d256():
    m = _stock(DEFAULT)
    gen = torch.Generator().manual_seed(5)
    f0 = torch.randn(2, 7 * 9, 256, generator=gen).to(torch.bfloat16).float()
    f1 = torch.randn(2, 10 * 12, 256, generator=gen).to(torch.bfloat16).float()
    with torch.no_grad():
        s0, s1 = m(f0, f1)
    o0, o1 = O.fine_transformer(f0, f1, _layers(m), m.layer_names)
    for o, s in ((o0, s0), (o1, s1)):
        assert torch.allclose(o, s, rtol=1e-5, atol=2e-5)
        assert torch.allclose(o.sum((1, 2)), s.sum((1, 2)), rtol=1e-4, atol=1e-2)


def test_pack_coarse_layer_puts_every_weight_at_the_header_offsets():
    header = open(os.path.join(ROOT, "include", "pope_b200.h")).read()
    assert int(re.search(r"#define POPE_COARSE_TF_LAYER_BYTES (\d+)", header).group(1)) == _lib.COARSE_TF_LAYER_BYTES
    sd = _layers(_stock(["self"]))[0]
    packed = ops.pack_coarse_layer(sd, "cpu")
    assert packed.numel() == _lib.COARSE_TF_LAYER_BYTES
    off = 0
    for key, shp in (("q_proj.weight", (256, 256)), ("k_proj.weight", (256, 256)), ("v_proj.weight", (256, 256)),
                     ("merge.weight", (256, 256)), ("mlp.0.weight", (512, 512)), ("mlp.2.weight", (256, 512))):
        n = shp[0] * shp[1] * 2
        got = packed[off:off + n].view(torch.bfloat16).view(shp)
        assert torch.equal(got.float(), sd[key].to(torch.bfloat16).float()), key
        off += n
    assert off == 1310720
    for key in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"):
        assert torch.equal(packed[off:off + 1024].view(torch.float32), sd[key]), key
        off += 1024
    bad = dict(sd)
    bad["mlp.0.weight"] = torch.zeros(256, 256)
    with pytest.raises(_lib.PopeError):
        ops.pack_coarse_layer(bad, "cpu")


def test_coarse_entry_points_reject_bad_arguments_before_touching_the_gpu():
    h = _lib.lib()
    kinds = (_lib.C.c_int * 2)(0, 1)
    ws = h.pope_coarse_tf_workspace_bytes(2, 64, 48)
    assert ws > 0 and h.pope_coarse_tf_workspace_bytes(0, 64, 48) == 0 and h.pope_coarse_tf_workspace_bytes(2, 0, 48) == 0
    # feat0, feat1, n_pairs, L, S, weights, n_layers, layer_kinds, workspace, workspace_bytes, stream
    ok = [16, 16, 2, 64, 48, None, 2, kinds, 16, ws, None]
    ok[5] = 16
    for i in (0, 1, 5, 7, 8):                                      # null features, weights, kinds and workspace
        bad = list(ok); bad[i] = None
        assert h.pope_coarse_transformer(*bad) == -1, i
    for i, v in ((2, -1), (3, 0), (4, 0), (6, -1)):                # negative / empty sizes
        bad = list(ok); bad[i] = v
        assert h.pope_coarse_transformer(*bad) == -1, i
    bad = list(ok); bad[7] = (_lib.C.c_int * 2)(0, 2)              # layer kind other than 'self' / 'cross'
    assert h.pope_coarse_transformer(*bad) == -1
    for i in (0, 1, 5, 8):                                         # misaligned pointers
        bad = list(ok); bad[i] = 24
        assert h.pope_coarse_transformer(*bad) == -5, i
    bad = list(ok); bad[9] = ws - 1                                # workspace too small
    assert h.pope_coarse_transformer(*bad) == -3
    bad = list(ok); bad[2] = 70000                                 # more pairs than the attention grid holds
    assert h.pope_coarse_transformer(*bad) == -4
    bad = list(ok); bad[2] = 0                                     # no pairs: a no-op
    assert h.pope_coarse_transformer(*bad) == 0

    # feat, pe, n, C, H, W, pe_h, pe_w, out, stream
    ok = [16, 16, 2, 256, 60, 80, 256, 256, 16, None]
    for i in (0, 1, 8):
        bad = list(ok); bad[i] = None
        assert h.pope_coarse_pos_encode(*bad) == -1, i
    for i, v in ((2, -1), (4, 0), (5, 0)):
        bad = list(ok); bad[i] = v
        assert h.pope_coarse_pos_encode(*bad) == -1, i
    for i, v in ((3, 128), (4, 257), (5, 300)):                    # C != 256, map larger than the encoding
        bad = list(ok); bad[i] = v
        assert h.pope_coarse_pos_encode(*bad) == -4, i
    for i, v in ((0, 18), (8, 24)):
        bad = list(ok); bad[i] = v
        assert h.pope_coarse_pos_encode(*bad) == -5, i
    bad = list(ok); bad[2] = 0
    assert h.pope_coarse_pos_encode(*bad) == 0


def test_matcher_coarse_flag_keeps_the_state_dict_and_rejects_unsupported_configs():
    cfg = pope_b200.make_default_cfg()
    stock = pope_b200.Matcher(cfg)
    m = pope_b200.Matcher(cfg, coarse_cuda_bf16=True)
    assert list(m.state_dict()) == list(stock.state_dict()) and len(m.state_dict()) == 211
    assert m.coarse_cuda_bf16 and not stock.coarse_cuda_bf16
    for key, val in (("d_model", 128), ("nhead", 4), ("attention", "full")):
        bad = copy.deepcopy(cfg)
        bad["coarse"][key] = val
        if key == "d_model":
            bad["fine"]["d_model"] = 128
        with pytest.raises(NotImplementedError):
            pope_b200.Matcher(bad, coarse_cuda_bf16=True)
        pope_b200.Matcher(bad).set_coarse_cuda_bf16(False)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def _run_all(m, f0, f1, dev):
    """(fp32 reference, stock bf16 modules, CUDA path) outputs on the same bf16-rounded inputs."""
    names = m.layer_names
    want = O.fine_transformer(f0.to(dev), f1.to(dev), [{k: v.to(dev) for k, v in l.items()} for l in _layers(m)], names)
    sb = copy.deepcopy(m).to(dev).to(torch.bfloat16)
    with torch.no_grad():
        stock = sb(f0.to(dev, torch.bfloat16), f1.to(dev, torch.bfloat16))
    packed = torch.cat([ops.pack_coarse_layer(l, dev) for l in _layers(m)])
    got = ops.coarse_transformer(f0.to(dev, torch.bfloat16), f1.to(dev, torch.bfloat16), packed, names)
    return want, stock, got


CASES = [  # (n pairs, L, S, sigma)
    (1, 4800, 4800, 1.0), (3, 4800, 4800, 1.0), (1, 4800, 1024, 1.0), (2, 63, 63, 1.0), (2, 63, 1024, 1.0),
    (1, 4800, 1024, 30.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("names", [DEFAULT, ["self"], ["cross"]], ids=["default", "self", "cross"])
@pytest.mark.parametrize("n,L,S,sigma", CASES)
def test_cuda_coarse_transformer_error_within_stock_bf16(names, n, L, S, sigma):
    dev = torch.device("cuda")
    m = _stock(names, seed=L + S)
    f0, f1 = synth.coarse_features(11, n, L, S, sigma=sigma, dtype=torch.bfloat16)
    want, stock, got = _run_all(m, f0.float(), f1.float(), dev)
    for side in range(2):
        e_cuda, e_stock = _rel_err(got[side], want[side]), _rel_err(stock[side], want[side])
        print(f"{names} n={n} L={L} S={S} sigma={sigma} side {side}: cuda rms {e_cuda[0]:.3e} max {e_cuda[1]:.3e} | "
              f"stock bf16 rms {e_stock[0]:.3e} max {e_stock[1]:.3e}")
        assert torch.isfinite(got[side].float()).all()
        assert e_cuda[0] <= 1.25 * e_stock[0], (side, e_cuda, e_stock)
        assert e_cuda[1] <= 1.25 * e_stock[1], (side, e_cuda, e_stock)


@pytest.mark.gpu
def test_cuda_coarse_transformer_is_deterministic_and_batch_independent():
    dev = torch.device("cuda")
    m = _stock(DEFAULT, seed=7)
    packed = torch.cat([ops.pack_coarse_layer(l, dev) for l in _layers(m)])
    f0, f1 = synth.coarse_features(3, 3, 2400, 1500, dtype=torch.bfloat16)
    g0, g1 = synth.coarse_features(4, 3, 2400, 1500, dtype=torch.bfloat16)
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
@pytest.mark.parametrize("temp_bug_fix", [True, False])
def test_pos_encode_kernel_is_bit_identical_to_torch(temp_bug_fix):
    dev = torch.device("cuda")
    pe = pope_b200.feature_net.PositionEncodingSine(256, temp_bug_fix=temp_bug_fix).to(dev)
    gen = torch.Generator().manual_seed(2)
    for n, h, w in ((2, 60, 80), (1, 32, 32), (3, 7, 9), (1, 256, 256)):
        x = (3 * torch.randn(n, 256, h, w, generator=gen)).to(dev)
        want = pe(x).flatten(2).transpose(1, 2).to(torch.bfloat16)
        got = ops.coarse_pos_encode(x, pe.pe)
        assert got.shape == want.shape and torch.equal(got.view(torch.int16), want.view(torch.int16)), (n, h, w)


def _images(dev, seed, hw0=(480, 640), hw1=(480, 640), n=1):
    gen = torch.Generator().manual_seed(seed)
    return {"image0": torch.rand(n, 1, *hw0, generator=gen).to(dev), "image1": torch.rand(n, 1, *hw1, generator=gen).to(dev)}


@pytest.mark.gpu
def test_matcher_only_att_fea_equals_the_kernels_on_the_backbone_output():
    dev = torch.device("cuda")
    torch.manual_seed(0)
    m = pope_b200.Matcher(pope_b200.make_default_cfg(), coarse_cuda_bf16=True).eval().to(dev)
    data = _images(dev, 1, (480, 640), (256, 256))
    with torch.no_grad():
        got0, got1 = m(dict(data), only_att_fea=True)
        c0, c1 = m.backbone(data["image0"])[0], m.backbone(data["image1"])[0]
        f0, f1 = ops.coarse_pos_encode(c0, m.pos_encoding.pe), ops.coarse_pos_encode(c1, m.pos_encoding.pe)
        packed = torch.cat([ops.pack_coarse_layer(l.state_dict(), dev) for l in m.loftr_coarse.layers])
        want0, want1 = ops.coarse_transformer(f0, f1, packed, m.loftr_coarse.layer_names)
    assert got0.dtype == torch.bfloat16 and got0.shape == (1, 4800, 256) and got1.shape == (1, 1024, 256)
    assert torch.equal(got0, want0) and torch.equal(got1, want1)


@pytest.mark.gpu
def test_matcher_forward_with_both_flags_writes_the_stock_keys():
    dev = torch.device("cuda")
    torch.manual_seed(0)
    cfg = pope_b200.make_default_cfg()
    stock = pope_b200.Matcher(cfg).eval().to(dev)
    fast = pope_b200.Matcher(cfg, fine_cuda_bf16=True, coarse_cuda_bf16=True).eval().to(dev)
    fast.load_state_dict(stock.state_dict())
    coarse_only = pope_b200.Matcher(cfg, coarse_cuda_bf16=True).eval().to(dev)
    coarse_only.load_state_dict(stock.state_dict())
    a, b, c = _images(dev, 2, (480, 640), (256, 256)), _images(dev, 2, (480, 640), (256, 256)), _images(dev, 2, (480, 640), (256, 256))
    with torch.no_grad():
        stock(a)
        fast(b)
        coarse_only(c)
    assert list(a) == list(b) == list(c)
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert a[k].dtype == b[k].dtype == c[k].dtype, k


@pytest.mark.gpu
def test_planted_matches_survive_the_cuda_coarse_transformer():
    """Random weights on images give no matches, so planted-correspondence features go through the transformer and then
    the coarse matcher.  sigma is raised until the fp32 stock path keeps more than 1000 matches through 8 layers."""
    dev = torch.device("cuda")
    m = _stock(DEFAULT, seed=3)
    hw0_i, hw_c = (480, 640), (60, 80)
    for sigma in (4.0, 8.0, 16.0, 32.0):
        f0, f1 = synth.coarse_features(21, 1, 4800, 4800, sigma=sigma, dtype=torch.bfloat16)
        want, stock, got = _run_all(m, f0.float(), f1.float(), dev)
        ref, mg = parity_utils.oracle_with_margins(want[0].cpu(), want[1].cpu(), hw0_i, hw_c, hw_c)
        if ref["b_ids"].numel() > 1000:
            break
    assert ref["b_ids"].numel() > 1000, sigma
    diffs = []
    for out in (stock, got):
        lst = O.coarse_match(out[0].float().cpu(), out[1].float().cpu(), hw0_i, hw_c, hw_c)
        same, near, bad = parity_utils.compare_match_lists(lst, ref, mg)
        diffs.append(len(near) + len(bad))
    print(f"sigma {sigma}: fp32 matches {ref['b_ids'].numel()}, rows differing: stock bf16 {diffs[0]}, cuda {diffs[1]}")
    assert diffs[1] <= 1.25 * diffs[0] + 1e-9, diffs
