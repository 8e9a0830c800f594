"""Feature producers of the Matcher that stay stock PyTorch (cuDNN / cuBLAS): the ResNet-FPN backbone, the
sinusoidal position encoding and the linear-attention LoFTR transformer.  They are OUT of the accelerated hot
path (SURVEY.md section 8) but are part of the drop-in boundary: module/parameter names reproduce the reference's
state-dict layout (211 entries) so `weights/matcher.pth` loads unchanged.

Reference: src/matcher/backbone/resnet_fpn.py:15-199, src/matcher/utils/position_encoding.py:6-42,
src/matcher/loftr_module/transformer.py:7-106, src/matcher/loftr_module/linear_attention.py:14-81.
"""
from __future__ import annotations

import math
from typing import List, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F


# ---- ResNet-FPN -----------------------------------------------------------------------------------------------

def _conv(cin: int, cout: int, k: int, stride: int = 1) -> nn.Conv2d:
    return nn.Conv2d(cin, cout, kernel_size=k, stride=stride, padding=k // 2, bias=False)


class ResidualBlock(nn.Module):
    """Two 3x3 conv+BN with identity (or strided 1x1 projection) shortcut (resnet_fpn.py:15-40)."""

    def __init__(self, cin: int, cout: int, stride: int = 1):
        super().__init__()
        self.conv1 = _conv(cin, cout, 3, stride)
        self.conv2 = _conv(cout, cout, 3)
        self.bn1 = nn.BatchNorm2d(cout)
        self.bn2 = nn.BatchNorm2d(cout)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = None if stride == 1 else nn.Sequential(_conv(cin, cout, 1, stride), nn.BatchNorm2d(cout))

    def forward(self, x):
        y = self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x)))))
        return self.relu((x if self.downsample is None else self.downsample(x)) + y)


class ResNetFPN(nn.Module):
    """ResNet stem + `len(block_dims)` stages + top-down FPN.  Returns [coarsest map, map of stage `fine_stage`].

    3 stages / fine_stage 1  == the reference's ResNetFPN_8_2  (resnet_fpn.py:43-118): outputs 1/8 and 1/2;
    4 stages / fine_stage 2  == ResNetFPN_16_4 (:121-199): outputs 1/16 and 1/4.
    Sub-module names (layerK, layerK_outconv, layerK_outconv2) are the reference's, they fix the checkpoint keys."""

    def __init__(self, config: dict, fine_stage: int = 1):
        super().__init__()
        dims: List[int] = list(config["block_dims"])
        stem = config["initial_dim"]
        self.n_stages, self.fine_stage = len(dims), fine_stage
        self.conv1 = nn.Conv2d(1, stem, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = nn.BatchNorm2d(stem)
        self.relu = nn.ReLU(inplace=True)
        cin = stem
        for k, d in enumerate(dims, start=1):
            setattr(self, f"layer{k}", nn.Sequential(ResidualBlock(cin, d, 1 if k == 1 else 2), ResidualBlock(d, d)))
            cin = d
        top = self.n_stages
        setattr(self, f"layer{top}_outconv", _conv(dims[-1], dims[-1], 1))
        for k in range(top - 1, fine_stage - 1, -1):       # lateral 1x1 + smoothing convs, top-down
            up, here = dims[k], dims[k - 1]
            setattr(self, f"layer{k}_outconv", _conv(here, up, 1))
            setattr(self, f"layer{k}_outconv2",
                    nn.Sequential(_conv(up, up, 3), nn.BatchNorm2d(up), nn.LeakyReLU(), _conv(up, here, 3)))
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.ones_(m.weight)
                nn.init.zeros_(m.bias)

    def forward(self, x):
        feats = []
        x = self.relu(self.bn1(self.conv1(x)))
        for k in range(1, self.n_stages + 1):
            x = getattr(self, f"layer{k}")(x)
            feats.append(x)
        top = self.n_stages
        coarse = getattr(self, f"layer{top}_outconv")(feats[-1])
        y = coarse
        for k in range(top - 1, self.fine_stage - 1, -1):
            up = F.interpolate(y, scale_factor=2.0, mode="bilinear", align_corners=True)
            y = getattr(self, f"layer{k}_outconv2")(getattr(self, f"layer{k}_outconv")(feats[k - 1]) + up)
        return [coarse, y]


def build_backbone(config: dict) -> nn.Module:
    """src/matcher/backbone/__init__.py:4-11."""
    if config["backbone_type"] != "ResNetFPN":
        raise ValueError(f"LOFTR.BACKBONE_TYPE {config['backbone_type']} not supported.")
    res = tuple(config["resolution"])
    if res == (8, 2):
        return ResNetFPN(config["resnetfpn"], fine_stage=1)
    if res == (16, 4):
        return ResNetFPN(config["resnetfpn"], fine_stage=2)
    raise ValueError(f"resolution {res} not supported")


# ---- position encoding ---------------------------------------------------------------------------------------

class PositionEncodingSine(nn.Module):
    """2-D sinusoidal encoding added to the coarse map (position_encoding.py:6-42).  With temp_bug_fix=False the
    frequency term keeps the reference's operator-precedence bug ((-ln 1e4 / d) // 2), which the released
    weights were trained with (:25-28)."""

    def __init__(self, d_model: int, max_shape=(256, 256), temp_bug_fix: bool = True):
        super().__init__()
        ys = torch.arange(1, max_shape[0] + 1, dtype=torch.float32).view(1, -1, 1).expand(1, *max_shape)
        xs = torch.arange(1, max_shape[1] + 1, dtype=torch.float32).view(1, 1, -1).expand(1, *max_shape)
        k = torch.arange(0, d_model // 2, 2).float()
        if temp_bug_fix:
            freq = torch.exp(k * (-math.log(10000.0) / (d_model // 2)))
        else:
            freq = torch.exp(k * (-math.log(10000.0) / d_model // 2))
        freq = freq.view(-1, 1, 1)
        pe = torch.zeros(d_model, *max_shape)
        pe[0::4] = torch.sin(xs * freq)
        pe[1::4] = torch.cos(xs * freq)
        pe[2::4] = torch.sin(ys * freq)
        pe[3::4] = torch.cos(ys * freq)
        self.register_buffer("pe", pe.unsqueeze(0), persistent=False)

    def forward(self, x):
        return x + self.pe[:, :, : x.size(2), : x.size(3)]


# ---- linear-attention transformer -----------------------------------------------------------------------------

class LinearAttention(nn.Module):
    """O(L d^2) attention with the elu(x)+1 feature map (linear_attention.py:14-47)."""

    def __init__(self, eps: float = 1e-6):
        super().__init__()
        self.eps = eps

    def forward(self, queries, keys, values, q_mask=None, kv_mask=None):
        q = F.elu(queries) + 1
        k = F.elu(keys) + 1
        if q_mask is not None:
            q = q * q_mask[:, :, None, None]
        if kv_mask is not None:
            k = k * kv_mask[:, :, None, None]
            values = values * kv_mask[:, :, None, None]
        s = values.size(1)
        kv = torch.einsum("nshd,nshv->nhdv", k, values / s)
        z = 1 / (torch.einsum("nlhd,nhd->nlh", q, k.sum(dim=1)) + self.eps)
        return (torch.einsum("nlhd,nhdv,nlh->nlhv", q, kv, z) * s).contiguous()


class FullAttention(nn.Module):
    """Softmax attention (linear_attention.py:50-81); selectable through config['attention'] == 'full'."""

    def forward(self, queries, keys, values, q_mask=None, kv_mask=None):
        qk = torch.einsum("nlhd,nshd->nlsh", queries, keys)
        if kv_mask is not None:
            qk.masked_fill_(~(q_mask[:, :, None, None] * kv_mask[:, None, :, None]), float("-inf"))
        a = torch.softmax(qk / queries.size(3) ** 0.5, dim=2)
        return torch.einsum("nlsh,nshd->nlhd", a, values).contiguous()


class LoFTREncoderLayer(nn.Module):
    def __init__(self, d_model: int, nhead: int, attention: str = "linear"):
        super().__init__()
        self.dim, self.nhead = d_model // nhead, nhead
        self.q_proj = nn.Linear(d_model, d_model, bias=False)
        self.k_proj = nn.Linear(d_model, d_model, bias=False)
        self.v_proj = nn.Linear(d_model, d_model, bias=False)
        self.attention = LinearAttention() if attention == "linear" else FullAttention()
        self.merge = nn.Linear(d_model, d_model, bias=False)
        self.mlp = nn.Sequential(nn.Linear(2 * d_model, 2 * d_model, bias=False), nn.ReLU(True),
                                 nn.Linear(2 * d_model, d_model, bias=False))
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)

    def forward(self, x, source, x_mask=None, source_mask=None):
        n = x.size(0)
        q = self.q_proj(x).view(n, -1, self.nhead, self.dim)
        k = self.k_proj(source).view(n, -1, self.nhead, self.dim)
        v = self.v_proj(source).view(n, -1, self.nhead, self.dim)
        msg = self.attention(q, k, v, q_mask=x_mask, kv_mask=source_mask)
        msg = self.norm1(self.merge(msg.view(n, -1, self.nhead * self.dim)))
        msg = self.norm2(self.mlp(torch.cat([x, msg], dim=2)))
        return x + msg


class LocalFeatureTransformer(nn.Module):
    """Stack of self/cross LoFTR layers (transformer.py:61-106).  Unlike the reference it neither prints the layer
    names (:72) nor mutates the config it is given (:68-71)."""

    def __init__(self, config: dict, d_model: Optional[int] = None, LAYER_NAMES: Optional[List[str]] = None):
        super().__init__()
        self.config = config
        self.d_model = d_model if d_model is not None else config["d_model"]
        self.nhead = config["nhead"]
        self.layer_names = list(LAYER_NAMES if LAYER_NAMES is not None else config["layer_names"])
        self.layers = nn.ModuleList([LoFTREncoderLayer(self.d_model, self.nhead, config["attention"])
                                     for _ in self.layer_names])
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)

    def forward(self, feat0, feat1, mask0=None, mask1=None):
        assert self.d_model == feat0.size(2), "the feature number of src and transformer must be equal"
        for layer, name in zip(self.layers, self.layer_names):
            if name == "self":
                feat0 = layer(feat0, feat0, mask0, mask0)
                feat1 = layer(feat1, feat1, mask1, mask1)
            elif name == "cross":
                feat0 = layer(feat0, feat1, mask0, mask1)
                feat1 = layer(feat1, feat0, mask1, mask0)
            else:
                raise KeyError(name)
        return feat0, feat1


class FineTransformerB200(LocalFeatureTransformer):
    """`loftr_fine` with the encoder layers running in libpope_b200.so (csrc/fine_tf.cu: tcgen05 Linears with fused
    epilogues + tensor-core linear attention) when it is handed CUDA bfloat16 windows; same parameters, same state-dict
    keys as LocalFeatureTransformer (transformer.py:61-106).  fp32 windows keep the stock PyTorch layers (the
    reference's precision) unless `cuda_fp32` is set: then CUDA fp32 windows run the fp32-accuracy fine transformer (every
    GEMM operand split into three bf16 terms, fp32 activations) and come back fp32.  Masks are not supported by the CUDA
    paths (no inference caller passes them to the fine level).

    `inplace`: update the given window tensors (the Matcher owns them) instead of working on copies."""

    def __init__(self, config: dict, d_model: Optional[int] = None, LAYER_NAMES: Optional[List[str]] = None):
        super().__init__(config, d_model, LAYER_NAMES)
        self.inplace = False
        self.cuda_fp32 = False
        self._packed = {}
        self._packed_key = {}
        self._workspace = None

    def cuda_supported(self) -> bool:
        return self.d_model == 128 and self.nhead == 8 and self.config["attention"] == "linear"

    def _packed_weights(self, dev, dtype: torch.dtype = torch.bfloat16):
        from . import ops
        key = (str(dev),) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        if dtype not in self._packed or self._packed_key[dtype] != key:
            self._packed[dtype] = torch.cat([ops.pack_fine_layer(layer.state_dict(), dev, dtype) for layer in self.layers])
            self._packed_key[dtype] = key
        return self._packed[dtype]

    def forward(self, feat0, feat1, mask0=None, mask1=None):
        bf16 = feat0.dtype == torch.bfloat16 and feat1.dtype == torch.bfloat16
        fp32 = self.cuda_fp32 and feat0.dtype == torch.float32 and feat1.dtype == torch.float32
        if not (feat0.is_cuda and (bf16 or fp32)):
            return super().forward(feat0, feat1, mask0, mask1)
        if mask0 is not None or mask1 is not None or not self.cuda_supported():
            raise NotImplementedError("the CUDA fine transformer covers d_model 128 / 8 heads / linear attention without masks")
        from . import ops
        assert self.d_model == feat0.size(2), "the feature number of src and transformer must be equal"
        if not self.inplace:
            feat0, feat1 = feat0.clone(), feat1.clone()
        feat0, feat1 = feat0.contiguous(), feat1.contiguous()
        self._workspace = ops.fine_level_workspace(feat0.shape[0], feat0.shape[1], feat0.device, self._workspace,
                                                   merge=False, dtype=feat0.dtype)
        return ops.fine_transformer(feat0, feat1, self._packed_weights(feat0.device, feat0.dtype), self.layer_names,
                                    self._workspace)


class CoarseTransformerB200(LocalFeatureTransformer):
    """`loftr_coarse` with the encoder layers running in libpope_b200.so (csrc/coarse_tf.cu: tcgen05 Linears with fused
    feature-map / LayerNorm / ReLU / residual epilogues + global linear attention reduced in a fixed order) when it is
    handed CUDA bfloat16 features [N, L, 256] / [N, S, 256]; same parameters, same state-dict keys as
    LocalFeatureTransformer (transformer.py:61-106).  fp32 features keep the stock PyTorch layers (the reference's
    precision) unless `cuda_fp32` is set: then CUDA fp32 features run the fp32-accuracy transformer (every GEMM operand
    split into three bf16 terms, fp32 activations) and come back fp32.  Masks (padded batches) are not supported by the
    CUDA paths.

    `inplace`: update the given feature tensors (the Matcher owns them) instead of working on copies."""

    def __init__(self, config: dict, d_model: Optional[int] = None, LAYER_NAMES: Optional[List[str]] = None):
        super().__init__(config, d_model, LAYER_NAMES)
        self.inplace = False
        self.cuda_fp32 = False
        self._packed = {}
        self._packed_key = {}
        self._workspace = None

    def cuda_supported(self) -> bool:
        return self.d_model == 256 and self.nhead == 8 and self.config["attention"] == "linear"

    def _packed_weights(self, dev, dtype: torch.dtype = torch.bfloat16):
        from . import ops
        key = (str(dev),) + tuple((p.data_ptr(), p._version) for p in self.parameters())
        if dtype not in self._packed or self._packed_key[dtype] != key:
            self._packed[dtype] = torch.cat([ops.pack_coarse_layer(layer.state_dict(), dev, dtype) for layer in self.layers])
            self._packed_key[dtype] = key
        return self._packed[dtype]

    def forward(self, feat0, feat1, mask0=None, mask1=None):
        bf16 = feat0.dtype == torch.bfloat16 and feat1.dtype == torch.bfloat16
        fp32 = self.cuda_fp32 and feat0.dtype == torch.float32 and feat1.dtype == torch.float32
        if not (feat0.is_cuda and (bf16 or fp32)):
            return super().forward(feat0, feat1, mask0, mask1)
        if mask0 is not None or mask1 is not None or not self.cuda_supported():
            raise NotImplementedError("the CUDA coarse transformer covers d_model 256 / 8 heads / linear attention without masks")
        from . import ops
        assert self.d_model == feat0.size(2), "the feature number of src and transformer must be equal"
        if not self.inplace:
            feat0, feat1 = feat0.clone(), feat1.clone()
        feat0, feat1 = feat0.contiguous(), feat1.contiguous()
        self._workspace = ops.coarse_tf_workspace(feat0.shape[0], feat0.shape[1], feat1.shape[1], feat0.device,
                                                  self._workspace, dtype=feat0.dtype)
        return ops.coarse_transformer(feat0, feat1, self._packed_weights(feat0.device, feat0.dtype), self.layer_names,
                                      self._workspace)
