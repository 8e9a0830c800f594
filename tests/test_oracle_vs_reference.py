"""Live cross-checks against the UNMODIFIED reference, where its sources are present (POPE_REFERENCE_ROOT); skipped
elsewhere.  Its recorded outputs under tests/golden are checked everywhere (test_oracle_golden.py, test_fine_tf.py,
test_coarse_masked.py, test_host_logic.py).  CPU only."""
import contextlib
import copy
import io

import pytest
import torch

from oracle import pope_oracle as O
from oracle import ref_shim
from pope_b200 import synth

pytestmark = pytest.mark.skipif(not ref_shim.reference_available(),
                                reason="needs the unmodified reference sources (POPE_REFERENCE_ROOT), which are not part of this repository")


@pytest.fixture(scope="module")
def ref():
    return ref_shim.import_reference()


def test_oracle_coarse_equals_reference_on_fresh_seeds(ref):
    from src.matcher.utils.coarse_matching import CoarseMatching
    cm = CoarseMatching(copy.deepcopy(ref.default_cfg)["match_coarse"]).eval()
    for seed, (h0, w0, h1, w1) in enumerate([(9, 11, 9, 11), (12, 8, 7, 13), (16, 16, 16, 16)], start=100):
        f0, f1 = synth.coarse_features(seed, 2, h0 * w0, h1 * w1, 64, sigma=0.8)
        data = {"hw0_i": torch.Size([h0 * 8, w0 * 8]), "hw1_i": torch.Size([h1 * 8, w1 * 8]),
                "hw0_c": torch.Size([h0, w0]), "hw1_c": torch.Size([h1, w1])}
        with torch.no_grad():
            cm(f0, f1, data)
        out = O.coarse_match(f0, f1, data["hw0_i"], (h0, w0), (h1, w1))
        for k in ("b_ids", "i_ids", "j_ids", "m_bids", "gt_mask"):
            assert torch.equal(out[k], data[k]), k
        for k in ("mconf", "mkpts0_c", "mkpts1_c"):
            assert torch.allclose(out[k], data[k], rtol=1e-6, atol=0), k


def test_feature_modules_compute_the_reference_function(ref):
    """The stock-PyTorch part of the drop-in (backbone, position encoding, both transformers, the
    FinePreprocess Linears) must be the same function as the reference's once the reference's weights are
    loaded: identical state-dict keys and equal outputs."""
    import pope_b200
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        rm = ref.Matcher(copy.deepcopy(ref.default_cfg)).eval()
    mine = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    sd = {"matcher." + k: v.clone() for k, v in rm.state_dict().items()}      # exercise the prefix stripping
    missing, unexpected = mine.load_state_dict(sd, strict=False)
    assert not missing and not unexpected
    g = torch.Generator().manual_seed(3)
    img0, img1 = torch.rand(1, 1, 64, 96, generator=g), torch.rand(1, 1, 48, 64, generator=g)
    with torch.no_grad():
        a0, a1 = rm({"image0": img0, "image1": img1}, only_att_fea=True)
        b0, b1 = mine({"image0": img0, "image1": img1}, only_att_fea=True)
        assert torch.allclose(a0, b0, rtol=1e-5, atol=1e-5) and torch.allclose(a1, b1, rtol=1e-5, atol=1e-5)
        w0, w1 = torch.randn(7, 25, 128, generator=g), torch.randn(7, 25, 128, generator=g)
        r0, r1 = rm.loftr_fine(w0, w1)
        m0, m1 = mine.loftr_fine(w0, w1)
        assert torch.allclose(r0, m0, rtol=1e-5, atol=1e-5) and torch.allclose(r1, m1, rtol=1e-5, atol=1e-5)
        fr, ff = rm.backbone(img0), mine.backbone(img0)
        assert torch.allclose(fr[0], ff[0], rtol=1e-5, atol=1e-5) and torch.allclose(fr[1], ff[1], rtol=1e-5, atol=1e-5)


def test_reference_random_init_gives_zero_matches(ref):
    """The 'vacuous parity trap' (SURVEY.md section 7): images + random weights -> M = 0, which is why parity is
    driven with synthetic features at the stage boundary."""
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        rm = ref.Matcher(copy.deepcopy(ref.default_cfg)).eval()
    batch = {"image0": torch.rand(1, 1, 64, 96), "image1": torch.rand(1, 1, 64, 96)}
    with torch.no_grad():
        rm(batch)
    assert batch["mconf"].numel() == 0 and batch["mkpts0_f"].shape == (0, 2) and batch["expec_f"].shape == (0, 3)


def test_oracle_masked_coarse_equals_reference_on_fresh_seeds(ref):
    """Padded batches: the -1e9 fill (coarse_matching.py:115-118) and mask_border_with_padding (:28-43), live."""
    from src.matcher.utils.coarse_matching import CoarseMatching
    cm = CoarseMatching(copy.deepcopy(ref.default_cfg)["match_coarse"]).eval()
    g = torch.Generator().manual_seed(9)
    for seed, (h0, w0, h1, w1) in enumerate([(12, 14, 10, 15), (16, 16, 16, 16)], start=300):
        n = 3
        f0, f1 = synth.coarse_features(seed, n, h0 * w0, h1 * w1, 64, sigma=0.8, planted=0.9)
        m0, m1 = torch.zeros(n, h0, w0, dtype=torch.bool), torch.zeros(n, h1, w1, dtype=torch.bool)
        for b in range(n):
            m0[b, : int(torch.randint(6, h0 + 1, (1,), generator=g)), : int(torch.randint(6, w0 + 1, (1,), generator=g))] = True
            m1[b, : int(torch.randint(6, h1 + 1, (1,), generator=g)), : int(torch.randint(6, w1 + 1, (1,), generator=g))] = True
        data = {"hw0_i": torch.Size([h0 * 8, w0 * 8]), "hw1_i": torch.Size([h1 * 8, w1 * 8]),
                "hw0_c": torch.Size([h0, w0]), "hw1_c": torch.Size([h1, w1]), "mask0": m0, "mask1": m1}
        with torch.no_grad():
            cm(f0, f1, data, mask_c0=m0.flatten(-2), mask_c1=m1.flatten(-2))
        out = O.coarse_match_masked(f0, f1, data["hw0_i"], (h0, w0), (h1, w1), m0, m1)
        for k in ("b_ids", "i_ids", "j_ids", "m_bids", "gt_mask"):
            assert torch.equal(out[k], data[k]), k
        for k in ("mconf", "mkpts0_c", "mkpts1_c"):
            assert torch.allclose(out[k], data[k], rtol=1e-6, atol=0), k
        assert data["b_ids"].numel() > 5


def test_coarse_transformer_with_masks_computes_the_reference_function(ref):
    """Matcher.forward hands the padding masks to the coarse transformer (matcher.py:60-63); ours is stock PyTorch and must
    be the same function there too."""
    import pope_b200
    torch.manual_seed(1)
    with contextlib.redirect_stdout(io.StringIO()):
        rm = ref.Matcher(copy.deepcopy(ref.default_cfg)).eval()
    mine = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    mine.load_state_dict(rm.state_dict(), strict=False)
    g = torch.Generator().manual_seed(4)
    c0, c1 = torch.randn(2, 8 * 12, 256, generator=g), torch.randn(2, 6 * 8, 256, generator=g)
    m0, m1 = torch.zeros(2, 8, 12, dtype=torch.bool), torch.zeros(2, 6, 8, dtype=torch.bool)
    m0[0, :8, :12], m0[1, :5, :9], m1[0, :6, :8], m1[1, :6, :4] = True, True, True, True
    with torch.no_grad():
        r0, r1 = rm.loftr_coarse(c0, c1, m0.flatten(-2), m1.flatten(-2))
        a0, a1 = mine.loftr_coarse(c0, c1, m0.flatten(-2), m1.flatten(-2))
    assert torch.allclose(r0, a0, rtol=1e-5, atol=1e-5) and torch.allclose(r1, a1, rtol=1e-5, atol=1e-5)
