"""Matcher -- drop-in for src/matcher/matcher.py:12-85 (reference tree).

Same constructor (`Matcher(config)`), same `forward(data, only_att_fea=False)` mutating `data` in place with the
reference's key order (bs, hw0_i, hw1_i, hw0_c, hw1_c, hw0_f, hw1_f, b_ids, i_ids, j_ids, gt_mask, m_bids,
mkpts0_c, mkpts1_c, mconf, W, expec_f, mkpts0_f, mkpts1_f), same sub-module names and therefore the same 211
state-dict keys, and the same `load_state_dict` that strips a leading 'matcher.' (:81-85).

Steps 3-5 of the forward (coarse match, fine-window gather, fine match; matcher.py:71-79) run in
libpope_b200.so; the backbone and the two transformers are stock PyTorch modules (feature_net.py) unless the bf16
CUDA paths are switched on (`fine_cuda_bf16`, `coarse_cuda_bf16`).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .coarse_matching import CoarseMatching
from .feature_net import CoarseTransformerB200, FineTransformerB200, PositionEncodingSine, build_backbone
from .fine_matching import FineMatching
from .fine_preprocess import FinePreprocess


class Matcher(nn.Module):
    def __init__(self, config: dict, fine_cuda_bf16: bool = False, coarse_cuda_bf16: bool = False):
        """`fine_cuda_bf16` (not in the reference): run the fine level -- window gather, FinePreprocess Linears, fine
        transformer, fine matching -- in bfloat16 inside libpope_b200.so instead of fp32 torch modules between the CUDA
        stages.  `coarse_cuda_bf16` (not in the reference): add the position encoding, lay the coarse maps out token-major
        and run the coarse transformer in bfloat16 inside libpope_b200.so; the coarse matcher then takes the bf16
        features, and `forward(data, only_att_fea=True)` returns them as bfloat16.  Parameters and state-dict keys are
        unchanged either way."""
        super().__init__()
        self.config = config
        self.backbone = build_backbone(config)
        self.pos_encoding = PositionEncodingSine(config["coarse"]["d_model"],
                                                 temp_bug_fix=config["coarse"]["temp_bug_fix"])
        self.loftr_coarse = CoarseTransformerB200(config["coarse"])
        self.coarse_matching = CoarseMatching(config["match_coarse"])
        self.fine_preprocess = FinePreprocess(config)
        self.loftr_fine = FineTransformerB200(config["fine"])
        self.fine_matching = FineMatching()
        self.set_fine_cuda_bf16(fine_cuda_bf16)
        self.set_coarse_cuda_bf16(coarse_cuda_bf16)

    def set_fine_cuda_bf16(self, on: bool) -> None:
        if on and not self.loftr_fine.cuda_supported():
            raise NotImplementedError("the CUDA fine transformer covers d_model 128 / 8 heads / linear attention")
        self.fine_cuda_bf16 = bool(on)
        self.fine_preprocess.cuda_bf16 = bool(on)
        self.loftr_fine.inplace = bool(on)

    def set_coarse_cuda_bf16(self, on: bool) -> None:
        if on and not self.loftr_coarse.cuda_supported():
            raise NotImplementedError("the CUDA coarse transformer covers d_model 256 / 8 heads / linear attention")
        self.coarse_cuda_bf16 = bool(on)
        self.loftr_coarse.inplace = bool(on)

    def fine_level(self, device) -> dict:
        """The packed bf16 weights of the fine level for `ops.match_pairs_device(..., fine_level=...)` (and the driver's
        batched steps built on it): {"pre": FinePreprocess' down_proj + merge_feat (None when fine_concat_coarse_feat is
        off), "layers": the fine transformer's layers, "layer_names": their 'self' / 'cross' schedule}.  The packed
        tensors are the modules' own caches, repacked only when a parameter changes."""
        if not self.loftr_fine.cuda_supported():
            raise NotImplementedError("the CUDA fine transformer covers d_model 128 / 8 heads / linear attention")
        dev = torch.device(device)
        pre = self.fine_preprocess._packed_weights(dev) if self.fine_preprocess.cat_c_feat else None
        return {"pre": pre, "layers": self.loftr_fine._packed_weights(dev), "layer_names": list(self.loftr_fine.layer_names)}

    def forward(self, data: dict, only_att_fea: bool = False):
        img0, img1 = data["image0"], data["image1"]
        data.update({"bs": img0.size(0), "hw0_i": img0.shape[2:], "hw1_i": img1.shape[2:]})
        if data["hw0_i"] == data["hw1_i"]:
            feats_c, feats_f = self.backbone(torch.cat([img0, img1], dim=0))
            (feat_c0, feat_c1), (feat_f0, feat_f1) = feats_c.split(data["bs"]), feats_f.split(data["bs"])
        else:
            (feat_c0, feat_f0), (feat_c1, feat_f1) = self.backbone(img0), self.backbone(img1)
        data.update({"hw0_c": feat_c0.shape[2:], "hw1_c": feat_c1.shape[2:],
                     "hw0_f": feat_f0.shape[2:], "hw1_f": feat_f1.shape[2:]})

        mask_c0 = mask_c1 = None
        if "mask0" in data:
            mask_c0, mask_c1 = data["mask0"].flatten(-2), data["mask1"].flatten(-2)
        # [N, C, H, W] -> [N, HW, C] after adding the position encoding
        if self.coarse_cuda_bf16 and feat_c0.is_cuda:      # (with masks, loftr_coarse raises NotImplementedError)
            from . import ops
            feat_c0 = ops.coarse_pos_encode(feat_c0, self.pos_encoding.pe)
            feat_c1 = ops.coarse_pos_encode(feat_c1, self.pos_encoding.pe)
        else:
            feat_c0 = self.pos_encoding(feat_c0).flatten(2).transpose(1, 2)
            feat_c1 = self.pos_encoding(feat_c1).flatten(2).transpose(1, 2)
        feat_c0, feat_c1 = self.loftr_coarse(feat_c0, feat_c1, mask_c0, mask_c1)
        if only_att_fea:
            return feat_c0, feat_c1

        self.coarse_matching(feat_c0, feat_c1, data, mask_c0=mask_c0, mask_c1=mask_c1)
        if feat_c0.dtype != feat_f0.dtype and not self.fine_cuda_bf16:     # the stock fine level runs in the maps' dtype
            feat_c0, feat_c1 = feat_c0.to(feat_f0.dtype), feat_c1.to(feat_f0.dtype)
        win0, win1 = self.fine_preprocess(feat_f0, feat_f1, feat_c0, feat_c1, data)
        if win0.size(0) != 0:
            win0, win1 = self.loftr_fine(win0, win1)
        self.fine_matching(win0, win1, data)

    def load_state_dict(self, state_dict, *args, **kwargs):
        for k in list(state_dict.keys()):
            if k.startswith("matcher."):
                state_dict[k.replace("matcher.", "", 1)] = state_dict.pop(k)
        return super().load_state_dict(state_dict, *args, **kwargs)
