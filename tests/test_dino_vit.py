"""Batched DINOv2 ViT-S/14 (SURVEY.md 8(f) rank 2): pope_b200.dino_vit.DinoViT against the UNMODIFIED reference module
(dinov2/dinov2/models/vision_transformer.py `vit_small`), where /root/reference is mounted; and the batched retrieval
driver against the per-crop loop of eval_linemod_json.py."""
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import pope_oracle as O
from oracle import ref_shim
from pope_b200.dino_vit import DinoViT, cls_tokens


def _small():
    torch.manual_seed(0)
    m = DinoViT(img_size=518, patch_size=14, embed_dim=384, depth=12, num_heads=6, init_values=1.0).eval()
    with torch.no_grad():                                  # random but non-degenerate weights
        for p in m.parameters():
            if p.dim() > 1:
                p.normal_(0, 0.05)
    return m


def test_state_dict_layout_of_vit_small():
    m = DinoViT()
    keys = set(m.state_dict().keys())
    assert {"cls_token", "pos_embed", "mask_token", "patch_embed.proj.weight", "patch_embed.proj.bias", "norm.weight",
            "blocks.0.norm1.weight", "blocks.0.attn.qkv.weight", "blocks.0.attn.qkv.bias", "blocks.0.attn.proj.weight",
            "blocks.0.ls1.gamma", "blocks.0.norm2.bias", "blocks.0.mlp.fc1.weight", "blocks.0.mlp.fc2.bias",
            "blocks.11.ls2.gamma"} <= keys
    assert m.pos_embed.shape == (1, 37 * 37 + 1, 384) and sum(p.numel() for p in m.parameters()) == 22_056_576


@pytest.mark.skipif(not ref_shim.reference_available(),
                    reason="needs the unmodified reference sources (POPE_REFERENCE_ROOT), which are not part of this repository")
def test_dino_vit_equals_reference_module():
    if ref_shim.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, ref_shim.REFERENCE_ROOT)
    from dinov2.dinov2.models.vision_transformer import vit_small   # the reference's own class, unmodified
    torch.manual_seed(1)
    ref = vit_small(patch_size=14, img_size=518, init_values=1.0, block_chunks=0).eval()
    with torch.no_grad():
        for p in ref.parameters():
            if p.dim() > 1:
                p.normal_(0, 0.05)
    mine = DinoViT().eval()
    missing, unexpected = mine.load_state_dict(ref.state_dict(), strict=True)
    assert not missing and not unexpected
    g = torch.Generator().manual_seed(2)
    for shape in ((3, 3, 224, 224), (2, 3, 518, 518), (1, 3, 224, 280)):
        x = torch.randn(shape, generator=g)
        with torch.no_grad():
            want = ref(x, is_training=True)
            got = mine(x, is_training=True)
        for k in ("x_norm_clstoken", "x_norm_patchtokens"):
            assert torch.allclose(got[k], want[k], rtol=1e-4, atol=2e-5), (shape, k, float((got[k] - want[k]).abs().max()))


def test_batched_tokens_equal_per_crop_loop_and_retrieval_slots():
    """One batched forward == R batch-1 forwards, and the slots of the device top-k == the eval loop's (oracle)."""
    m = _small()
    g = torch.Generator().manual_seed(3)
    ref_img, crops = torch.randn(1, 3, 224, 224, generator=g), torch.randn(9, 3, 224, 224, generator=g)
    with torch.no_grad():
        one_by_one = torch.cat([m(crops[r:r + 1], is_training=True)["x_norm_clstoken"] for r in range(9)])
    batched = cls_tokens(m, crops, batch=4)
    assert torch.allclose(batched, one_by_one, rtol=1e-4, atol=1e-5)
    q = cls_tokens(m, ref_img)
    scores = O.cosine_scores(q, batched)
    slot_s, slot_i = O.running_topk(scores.tolist(), 3)
    loop = [float(F.cosine_similarity(q, one_by_one[r:r + 1], dim=1, eps=1e-8)) for r in range(9)]
    assert torch.allclose(scores, torch.tensor(loop), rtol=1e-5, atol=1e-6)
    assert sorted(i for i in slot_i if i >= 0) == sorted(torch.tensor(loop).topk(3).indices.tolist()) or min(slot_s) <= 0


@pytest.mark.gpu
def test_retrieve_topk_images_on_device():
    import pope_b200
    dev = torch.device("cuda:0")
    m = _small().to(dev)
    g = torch.Generator().manual_seed(4)
    ref_img, crops = torch.randn(1, 3, 224, 224, generator=g).to(dev), torch.randn(37, 3, 224, 224, generator=g).to(dev)
    scores, slot_s, slot_i = pope_b200.retrieve_topk_images(m, ref_img, crops, k=3, batch=16)
    with torch.no_grad():
        q = m(ref_img, is_training=True)["x_norm_clstoken"]
        loop = torch.cat([F.cosine_similarity(q, m(crops[r:r + 1], is_training=True)["x_norm_clstoken"], dim=1, eps=1e-8)
                          for r in range(37)])
    assert torch.allclose(scores, loop, rtol=1e-3, atol=1e-4)
    want_s, want_i = O.running_topk(loop.tolist(), 3)
    assert slot_i == want_i
