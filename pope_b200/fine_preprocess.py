"""FinePreprocess -- drop-in for src/matcher/loftr_module/fine_preprocess.py:8-59.

The window extraction (F.unfold of both fine maps + gather of the matched cells, :40-47) runs in
libpope_b200.so (`pope_fine_gather`): only the M matched 5x5 windows are read.  The two small Linears that mix
in the coarse feature (:50-57) stay torch/cuBLAS in the reference's fp32 precision; with `cuda_bf16 = True` the windows
are gathered in bfloat16 and the Linears run in libpope_b200.so too (`pope_fine_merge_coarse`, csrc/fine_tf.cu); with
`cuda_fp32 = True` the fp32 windows go through the Linears in libpope_b200.so at fp32 accuracy
(`pope_fine_merge_coarse_f32`).
Parameter names (`down_proj`, `merge_feat`) are the reference's.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops


class FinePreprocess(nn.Module):
    def __init__(self, config: dict):
        super().__init__()
        self.config = config
        self.cat_c_feat = config["fine_concat_coarse_feat"]
        self.W = config["fine_window_size"]
        d_model_c = config["coarse"]["d_model"]
        self.d_model_f = config["fine"]["d_model"]
        if self.cat_c_feat:
            self.down_proj = nn.Linear(d_model_c, self.d_model_f, bias=True)
            self.merge_feat = nn.Linear(2 * self.d_model_f, self.d_model_f, bias=True)
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.kaiming_normal_(p, mode="fan_out", nonlinearity="relu")
        self.cuda_bf16 = False          # bf16 windows + CUDA Linears (set by Matcher(config, fine_cuda_bf16=True))
        self.cuda_fp32 = False          # fp32 windows + CUDA Linears at fp32 accuracy (Matcher(config, fine_cuda_fp32=True))
        self._packed = {}
        self._packed_key = {}

    def _packed_weights(self, dev, dtype: torch.dtype = torch.bfloat16):
        key = (str(dev),) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        if dtype not in self._packed or self._packed_key[dtype] != key:
            self._packed[dtype] = ops.pack_fine_pre(self.state_dict(), dev, dtype)
            self._packed_key[dtype] = key
        return self._packed[dtype]

    def forward(self, feat_f0, feat_f1, feat_c0, feat_c1, data):
        W = self.W
        stride = data["hw0_f"][0] // data["hw0_c"][0]
        data.update({"W": W})
        b_ids, i_ids, j_ids = data["b_ids"], data["i_ids"], data["j_ids"]
        if b_ids.shape[0] == 0:
            empty = torch.empty(0, W * W, self.d_model_f, device=feat_f0.device)
            return empty, empty.clone()
        # the CUDA gather is coalesced on channels-last maps (a window pixel = one contiguous Cf-vector); the stock
        # backbone emits NCHW, so re-layout once per call (one pass over the map, far cheaper than F.unfold's 25x blow-up)
        bf16 = self.cuda_bf16 and feat_f0.is_cuda and self.d_model_f == 128
        if bf16:
            feat_f0, feat_f1 = feat_f0.to(torch.bfloat16), feat_f1.to(torch.bfloat16)
        feat_f0 = feat_f0.contiguous(memory_format=torch.channels_last)
        feat_f1 = feat_f1.contiguous(memory_format=torch.channels_last)
        win0, win1 = ops.fine_gather(feat_f0, feat_f1, b_ids, i_ids, j_ids, data["hw0_c"][1], data["hw1_c"][1],
                                     stride, W)
        if self.cat_c_feat and bf16 and feat_c0.shape[2] == 256:
            win0, win1 = ops.fine_merge_coarse(win0, win1, feat_c0.to(torch.bfloat16).contiguous(),
                                               feat_c1.to(torch.bfloat16).contiguous(), b_ids, i_ids, j_ids,
                                               self._packed_weights(win0.device))
        elif self.cat_c_feat and self.cuda_fp32 and win0.is_cuda and win0.dtype == torch.float32 \
                and self.d_model_f == 128 and feat_c0.shape[2] == 256:
            win0, win1 = ops.fine_merge_coarse(win0, win1, feat_c0.float().contiguous(), feat_c1.float().contiguous(), b_ids,
                                               i_ids, j_ids, self._packed_weights(win0.device, torch.float32))
        elif self.cat_c_feat:
            m = b_ids.shape[0]
            c_win = self.down_proj(torch.cat([feat_c0[b_ids, i_ids], feat_c1[b_ids, j_ids]], 0))      # [2M, Cf]
            both = torch.cat([win0, win1], 0).to(c_win.dtype)                                          # [2M, WW, Cf]
            merged = self.merge_feat(torch.cat([both, c_win[:, None, :].expand(-1, W * W, -1)], -1))
            win0, win1 = merged[:m], merged[m:]
        return win0, win1
