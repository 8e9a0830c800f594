"""Fine-level transformer + FinePreprocess Linears (SURVEY.md 8(f) rank 1).

CPU: the oracle restatement (oracle/pope_oracle.py: fine_transformer, fine_merge_coarse) and the Matcher's `loftr_fine`
module against the fixture produced by the UNMODIFIED reference (oracle/gen_golden_fine_tf.py).  GPU: the bf16 CUDA path (pope_fine_transformer /
pope_fine_merge_coarse through the C ABI) against the same fixture and against the oracle on other shapes.

Tolerance of the bf16 path: weights and inputs are bf16 on both sides, but the CUDA path also rounds every activation
that crosses HBM to bf16 (q, k, v, message, hidden layer, layer outputs: ~12 roundings of 2^-9 along the deepest path),
so its outputs agree with the fp32 reference to a few 1e-2 of the output scale, not to 1e-4.  The bound asserted is on
the error relative to the RMS of the reference output (rms error < 1.5e-2, max error < 8e-2).
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import pope_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _bf16(bits: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(bits.view(np.int16).copy()).view(torch.bfloat16).float()


def _load():
    g = {}
    for name in ("fine_transformer.npz", "fine_merge_coarse.npz"):      # the transformer's fixture, the Linears' (`pre.`)
        g.update(np.load(os.path.join(GOLDEN, name)))
    meta = json.loads(str(g["meta"]))
    layers = []
    for l in range(len(meta["layer_names"])):
        sd = {}
        for k in g:
            pre = f"tf.layers.{l}."
            if k.startswith(pre):
                sd[k[len(pre):]] = _bf16(g[k]) if g[k].dtype == np.uint16 else torch.from_numpy(g[k])
        layers.append(sd)
    pre_sd = {k[4:]: (_bf16(g[k]) if g[k].dtype == np.uint16 else torch.from_numpy(g[k]))
              for k in g if k.startswith("pre.") and ("weight" in k or "bias" in k)}
    return g, meta, layers, pre_sd


def _inputs(seed, m, ww=25):
    gen = torch.Generator().manual_seed(seed)
    return (torch.randn(m, ww, 128, generator=gen).to(torch.bfloat16).float(),
            torch.randn(m, ww, 128, generator=gen).to(torch.bfloat16).float())


def _rel_err(got: torch.Tensor, want: torch.Tensor):
    rms = want.pow(2).mean().sqrt()
    d = (got.float() - want).abs()
    return float(d.pow(2).mean().sqrt() / rms), float(d.max() / rms)


# ---- CPU: the oracle is pinned to the reference's outputs -------------------------------------------------------------

def test_oracle_fine_transformer_matches_reference_fixture():
    g, meta, layers, _ = _load()
    f0, f1 = _inputs(meta["input_seed"], meta["m"])
    o0, o1 = O.fine_transformer(f0, f1, layers, meta["layer_names"])
    k = meta["kept"]
    assert torch.allclose(o0[:k], torch.from_numpy(g["out0"]), rtol=1e-5, atol=2e-5)
    assert torch.allclose(o1[:k], torch.from_numpy(g["out1"]), rtol=1e-5, atol=2e-5)
    assert torch.allclose(o0.sum((1, 2)), torch.from_numpy(g["out0_sum"]), rtol=1e-4, atol=1e-2)
    assert torch.allclose(o1.sum((1, 2)), torch.from_numpy(g["out1_sum"]), rtol=1e-4, atol=1e-2)


def test_fine_transformer_module_matches_reference_fixture():
    """The Matcher's own `loftr_fine` (stock PyTorch layers for fp32 input), loaded with the reference's weights through the
    state-dict layout, reproduces the reference's outputs."""
    import pope_b200
    g, meta, _, _ = _load()
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    sd = {k[3:]: (_bf16(v) if v.dtype == np.uint16 else torch.from_numpy(v)) for k, v in g.items() if k.startswith("tf.")}
    m.loftr_fine.load_state_dict(sd, strict=True)
    assert m.loftr_fine.layer_names == meta["layer_names"]
    f0, f1 = _inputs(meta["input_seed"], meta["m"])
    with torch.no_grad():
        o0, o1 = m.loftr_fine(f0, f1)
    k = meta["kept"]
    assert torch.allclose(o0[:k], torch.from_numpy(g["out0"]), rtol=1e-5, atol=2e-5)
    assert torch.allclose(o1[:k], torch.from_numpy(g["out1"]), rtol=1e-5, atol=2e-5)
    assert torch.allclose(o0.sum((1, 2)), torch.from_numpy(g["out0_sum"]), rtol=1e-4, atol=1e-2)
    assert torch.allclose(o1.sum((1, 2)), torch.from_numpy(g["out1_sum"]), rtol=1e-4, atol=1e-2)


def test_oracle_fine_merge_coarse_matches_reference_fixture():
    g, meta, _, pre_sd = _load()
    f0, f1 = _inputs(meta["input_seed"], meta["m"])
    fc0, fc1 = _bf16(g["pre.feat_c0"]), _bf16(g["pre.feat_c1"])
    ids = [torch.from_numpy(g["pre." + k]) for k in ("b_ids", "i_ids", "j_ids")]
    m0, m1 = O.fine_merge_coarse(f0, f1, fc0, fc1, *ids, pre_sd)
    k = meta["kept"]
    assert torch.allclose(m0[:k], torch.from_numpy(g["pre.merged0"]), rtol=1e-5, atol=2e-5)
    assert torch.allclose(m1[:k], torch.from_numpy(g["pre.merged1"]), rtol=1e-5, atol=2e-5)
    assert torch.allclose(torch.cat([m0, m1]).sum((1, 2)), torch.from_numpy(g["pre.merged_sum"]), rtol=1e-4, atol=1e-2)


def test_linear_attention_known_answers():
    """Identical keys -> the message is the mean value; a single source token -> the message is that token's value."""
    gen = torch.Generator().manual_seed(3)
    q = torch.randn(2, 5, 8, 16, generator=gen)
    v = torch.randn(2, 7, 8, 16, generator=gen)
    k = torch.randn(2, 1, 8, 16, generator=gen).expand(-1, 7, -1, -1)
    out = O.linear_attention(q, k, v)
    assert torch.allclose(out, v.mean(1, keepdim=True).expand(-1, 5, -1, -1), rtol=1e-4, atol=1e-5)
    out1 = O.linear_attention(q, k[:, :1], v[:, :1])
    assert torch.allclose(out1, v[:, :1].expand(-1, 5, -1, -1), rtol=1e-4, atol=1e-5)


# ---- GPU: the CUDA path through the C ABI -----------------------------------------------------------------------------

def _cuda_layers(layers, dev):
    from pope_b200 import ops
    return torch.cat([ops.pack_fine_layer(sd, dev) for sd in layers])


@pytest.mark.gpu
def test_cuda_fine_transformer_vs_reference_fixture():
    from pope_b200 import ops
    dev = torch.device("cuda:0")
    g, meta, layers, _ = _load()
    f0, f1 = _inputs(meta["input_seed"], meta["m"])
    d0, d1 = f0.to(dev, torch.bfloat16), f1.to(dev, torch.bfloat16)
    ops.fine_transformer(d0, d1, _cuda_layers(layers, dev), meta["layer_names"])
    torch.cuda.synchronize()
    k = meta["kept"]
    for got, want in ((d0[:k].cpu(), torch.from_numpy(g["out0"])), (d1[:k].cpu(), torch.from_numpy(g["out1"]))):
        rms, mx = _rel_err(got, want)
        assert rms < 1.5e-2 and mx < 8e-2, (rms, mx)
    want0, want1 = O.fine_transformer(f0, f1, layers, meta["layer_names"])        # all 37 windows incl. the ragged tile
    for got, want in ((d0.cpu(), want0), (d1.cpu(), want1)):
        rms, mx = _rel_err(got, want)
        assert rms < 1.5e-2 and mx < 8e-2, (rms, mx)


@pytest.mark.gpu
@pytest.mark.parametrize("m,names", [(1, ["self"]), (5, ["cross"]), (1003, ["self", "cross"]), (2048, ["cross", "self", "cross"])])
def test_cuda_fine_transformer_vs_oracle(m, names):
    """Other window counts (one window; a count whose 25*m is not a multiple of the 128-row tile; more tiles than SMs)
    and other layer schedules, with fresh random weights (LayerNorm scale/shift randomised)."""
    from pope_b200 import ops
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(100 + m)
    layers = []
    for _ in names:
        sd = {}
        for key, shp in (("q_proj.weight", (128, 128)), ("k_proj.weight", (128, 128)), ("v_proj.weight", (128, 128)),
                         ("merge.weight", (128, 128)), ("mlp.0.weight", (256, 256)), ("mlp.2.weight", (128, 256))):
            bound = (6.0 / (shp[0] + shp[1])) ** 0.5                                 # xavier_uniform_ (transformer.py:78-81)
            sd[key] = ((torch.rand(shp, generator=gen) * 2 - 1) * bound).to(torch.bfloat16).float()
        for key in ("norm1", "norm2"):
            sd[key + ".weight"] = 1 + 0.2 * torch.randn(128, generator=gen)
            sd[key + ".bias"] = 0.1 * torch.randn(128, generator=gen)
        layers.append(sd)
    f0, f1 = _inputs(200 + m, m)
    d0, d1 = f0.to(dev, torch.bfloat16), f1.to(dev, torch.bfloat16)
    r0, r1 = ops.fine_transformer(d0, d1, _cuda_layers(layers, dev), names)
    assert r0.data_ptr() == d0.data_ptr() and r1.data_ptr() == d1.data_ptr()
    torch.cuda.synchronize()
    want0, want1 = O.fine_transformer(f0, f1, layers, names)
    for got, want in ((d0.cpu(), want0), (d1.cpu(), want1)):
        assert torch.isfinite(got.float()).all()
        rms, mx = _rel_err(got, want)
        assert rms < 1.5e-2 and mx < 8e-2, (m, names, rms, mx)


@pytest.mark.gpu
def test_cuda_fine_transformer_empty_and_errors():
    from pope_b200 import _lib, ops
    dev = torch.device("cuda:0")
    _, meta, layers, _ = _load()
    packed = _cuda_layers(layers, dev)
    e0 = torch.empty(0, 25, 128, dtype=torch.bfloat16, device=dev)
    r0, r1 = ops.fine_transformer(e0, e0.clone(), packed, meta["layer_names"])
    assert r0.shape == (0, 25, 128)
    with pytest.raises(_lib.PopeError):
        ops.fine_transformer(torch.zeros(2, 25, 128, device=dev), torch.zeros(2, 25, 128, device=dev), packed, meta["layer_names"])
    with pytest.raises(_lib.PopeError):
        ops.fine_transformer(torch.zeros(2, 25, 128), torch.zeros(2, 25, 128), packed, meta["layer_names"])   # CPU tensors


@pytest.mark.gpu
def test_cuda_fine_merge_coarse_vs_reference_fixture():
    from pope_b200 import ops
    dev = torch.device("cuda:0")
    g, meta, _, pre_sd = _load()
    f0, f1 = _inputs(meta["input_seed"], meta["m"])
    fc0, fc1 = _bf16(g["pre.feat_c0"]), _bf16(g["pre.feat_c1"])
    ids = [torch.from_numpy(g["pre." + k]) for k in ("b_ids", "i_ids", "j_ids")]
    d0, d1 = f0.to(dev, torch.bfloat16), f1.to(dev, torch.bfloat16)
    ops.fine_merge_coarse(d0, d1, fc0.to(dev, torch.bfloat16), fc1.to(dev, torch.bfloat16), *[t.to(dev) for t in ids],
                          ops.pack_fine_pre(pre_sd, dev))
    torch.cuda.synchronize()
    want0, want1 = O.fine_merge_coarse(f0, f1, fc0, fc1, *ids, pre_sd)
    k = meta["kept"]
    assert _rel_err(d0[:k].cpu(), torch.from_numpy(g["pre.merged0"]))[1] < 2e-2
    for got, want in ((d0.cpu(), want0), (d1.cpu(), want1)):
        rms, mx = _rel_err(got, want)
        assert rms < 4e-3 and mx < 2e-2, (rms, mx)        # one bf16 rounding of c and one of the output


@pytest.mark.gpu
def test_matcher_bf16_fine_path_vs_fp32_module_flow():
    """Steps 3-5 of Matcher.forward with `fine_cuda_bf16=True` (bf16 window gather -> CUDA Linears -> CUDA fine transformer
    -> CUDA fine match) against the same modules in fp32 on the CPU (oracle for the hot-path stages, the weight-sharing
    torch modules for the Linears / transformer).  Match indices are identical (the coarse stage is untouched); the
    refined coordinates carry the bf16 fine level: |delta| is a small fraction of the +-4 px refinement range."""
    import copy
    import pope_b200
    from pope_b200 import synth
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m_cpu = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    m_gpu = copy.deepcopy(m_cpu).to(dev)
    m_gpu.set_fine_cuda_bf16(True)
    h, w, n = 20, 24, 2
    f0, f1 = synth.coarse_features(61, n, h * w, h * w, 256, sigma=0.85)
    ff0, ff1 = synth.fine_feature_maps(62, n, h * 4, w * 4, 128, channels_last=False)
    data = {"hw0_i": torch.Size([h * 8, w * 8]), "hw1_i": torch.Size([h * 8, w * 8]), "hw0_c": torch.Size([h, w]),
            "hw1_c": torch.Size([h, w]), "hw0_f": torch.Size([h * 4, w * 4]), "hw1_f": torch.Size([h * 4, w * 4]), "bs": n}
    with torch.no_grad():
        m_gpu.coarse_matching(f0.to(dev), f1.to(dev), data)
        w0, w1 = m_gpu.fine_preprocess(ff0.to(dev), ff1.to(dev), f0.to(dev), f1.to(dev), data)
        assert w0.dtype == torch.bfloat16
        w0, w1 = m_gpu.loftr_fine(w0, w1)
        m_gpu.fine_matching(w0, w1, data)
        want = O.coarse_match(f0, f1, data["hw0_i"], (h, w), (h, w))
        c0, c1 = O.fine_windows(ff0, want["b_ids"], want["i_ids"]), O.fine_windows(ff1, want["b_ids"], want["j_ids"])
        cw = m_cpu.fine_preprocess.down_proj(torch.cat([f0[want["b_ids"], want["i_ids"]], f1[want["b_ids"], want["j_ids"]]], 0))
        mg = m_cpu.fine_preprocess.merge_feat(torch.cat([torch.cat([c0, c1], 0), cw[:, None].expand(-1, 25, -1)], -1))
        c0, c1 = m_cpu.loftr_fine(*mg.chunk(2, 0))
        wf = O.fine_match(c0, c1, want["mkpts0_c"], want["mkpts1_c"], 2.0)
    for k in ("b_ids", "i_ids", "j_ids"):
        assert torch.equal(data[k].cpu(), want[k])
    assert data["mkpts1_f"].dtype == torch.float32 and data["expec_f"].shape == (want["b_ids"].numel(), 3)
    d = (data["mkpts1_f"].cpu() - wf["mkpts1_f"]).abs()
    assert want["b_ids"].numel() > 200
    assert float(d.mean()) < 0.03 and float(d.max()) < 0.3, (float(d.mean()), float(d.max()))     # pixels, range +-4
    # the state dict is the reference's whether or not the CUDA fine level is on
    assert list(m_gpu.state_dict().keys()) == list(m_cpu.state_dict().keys())


@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 300])
def test_cuda_fine_transformer_7x7_windows_vs_oracle(m):
    """7 x 7 windows (`fine_window_size` 7): 49 tokens exceed the 32-row tile of the mma.sync attention, so the fp32 SIMT
    attention kernel runs.  49 * m rows leave a ragged 128-row tile for both counts."""
    from pope_b200 import ops
    dev = torch.device("cuda:0")
    _, meta, layers, _ = _load()
    f0, f1 = _inputs(321 + m, m, 49)
    d0, d1 = f0.to(dev, torch.bfloat16), f1.to(dev, torch.bfloat16)
    ops.fine_transformer(d0, d1, _cuda_layers(layers, dev), meta["layer_names"])
    torch.cuda.synchronize()
    want0, want1 = O.fine_transformer(f0, f1, layers, meta["layer_names"])
    for got, want in ((d0.cpu(), want0), (d1.cpu(), want1)):
        assert torch.isfinite(got.float()).all()
        rms, mx = _rel_err(got, want)
        assert rms < 1.5e-2 and mx < 8e-2, (m, rms, mx)
