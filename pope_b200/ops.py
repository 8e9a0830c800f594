"""Functional wrappers over the C ABI (device tensors in, device tensors out).

Each function is the CUDA replacement of one reference function (paths relative to the reference tree):
  coarse_match  <- CoarseMatching.forward/get_coarse_match   src/matcher/utils/coarse_matching.py:87-261
  fine_gather   <- FinePreprocess unfold + gather              src/matcher/loftr_module/fine_preprocess.py:40-47
  fine_match    <- FineMatching.forward/get_fine_match         src/matcher/utils/fine_matching.py:15-74
  cosine_topk   <- retrieval loop                              eval_linemod_json.py:72-101
Nothing here computes on the CPU; tensors that are not on a CUDA device are rejected.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import check, dtype_code, lib, ptr, require_cuda, stream_ptr


class CoarseResult(dict):
    """dict of device tensors at full capacity plus `counts` (int32 [n+2] on device).  `.sliced()` performs the
    one host sync (reads the total) and returns views of length M, in the reference's key order."""

    def total(self) -> int:
        return int(self["counts"][self["n_pairs"]].item())

    def flags(self) -> int:
        return int(self["counts"][self["n_pairs"] + 1].item())

    def sliced(self) -> Dict[str, torch.Tensor]:
        n = self["n_pairs"]
        m, fl = self["counts"][n:n + 2].tolist()          # one transfer: the total and the flag word
        if fl & ~_lib.FLAG_ROBUST_PATH:                   # ROBUST_PATH is informational; anything else the caller must hear of
            import warnings
            what = [name for bit, name in ((_lib.FLAG_NONFINITE_LSE, "inf / nan in the features (non-finite log-sum-exp)"),
                                           (_lib.FLAG_CAND_OVERFLOW, "candidate list overflow (nan in the features)"),
                                           (_lib.FLAG_CAPACITY, "more matches than the output capacity: list truncated"))
                    if fl & bit]
            warnings.warn("pope_coarse_match: " + "; ".join(what), RuntimeWarning, stacklevel=2)
        out = {k: self[k][:m] for k in ("b_ids", "i_ids", "j_ids")}
        mconf = self["mconf"][:m]
        out["gt_mask"] = mconf == 0
        out["m_bids"] = out["b_ids"]
        out["mkpts0_c"] = self["mkpts0_c"][:m]
        out["mkpts1_c"] = self["mkpts1_c"][:m]
        out["mconf"] = mconf
        return out


def coarse_match(feat_c0: torch.Tensor, feat_c1: torch.Tensor, hw0_c: Sequence[int], hw1_c: Sequence[int],
                 pixel_scale: float, thr: float = 0.2, border_rm: int = 2, temperature: float = 0.1,
                 impl: int = _lib.COARSE_AUTO, workspace: Optional[torch.Tensor] = None) -> CoarseResult:
    dev = require_cuda(feat_c0, feat_c1)
    if feat_c0.dtype != feat_c1.dtype:
        raise _lib.PopeError("feat_c0 and feat_c1 must have the same dtype")
    feat_c0, feat_c1 = feat_c0.contiguous(), feat_c1.contiguous()
    n, L, Cc = feat_c0.shape
    S = feat_c1.shape[1]
    if feat_c1.shape[0] != n or feat_c1.shape[2] != Cc:
        raise _lib.PopeError(f"shape mismatch {tuple(feat_c0.shape)} vs {tuple(feat_c1.shape)}")
    h = lib()
    # fp32 features: the larger workspace enables the tensor-core path (three-way bf16 split) unless SIMT is requested
    need = (h.pope_coarse_workspace_bytes(n, L, S) if impl == _lib.COARSE_SIMT
            else h.pope_coarse_workspace_bytes_ex(n, L, S, feat_c0.shape[2], dtype_code(feat_c0)))
    if workspace is None or workspace.numel() < need or workspace.device != dev:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    cap = n * L           # one match per row: never truncated (the C ABI's documented minimum is n * min(L, S))
    i64 = dict(dtype=torch.int64, device=dev)
    f32 = dict(dtype=torch.float32, device=dev)
    res = CoarseResult(
        b_ids=torch.empty(cap, **i64), i_ids=torch.empty(cap, **i64), j_ids=torch.empty(cap, **i64),
        mconf=torch.empty(cap, **f32), mkpts0_c=torch.empty(cap, 2, **f32), mkpts1_c=torch.empty(cap, 2, **f32),
        counts=torch.empty(n + 2, dtype=torch.int32, device=dev), n_pairs=n, workspace=workspace)
    with torch.cuda.device(dev):
        st = h.pope_coarse_match(ptr(feat_c0), ptr(feat_c1), dtype_code(feat_c0), n, L, S, Cc,
                                 int(hw0_c[0]), int(hw0_c[1]), int(hw1_c[0]), int(hw1_c[1]),
                                 float(pixel_scale), float(temperature), float(thr), int(border_rm), int(impl),
                                 ptr(workspace), workspace.numel(),
                                 ptr(res["b_ids"]), ptr(res["i_ids"]), ptr(res["j_ids"]), ptr(res["mconf"]),
                                 ptr(res["mkpts0_c"]), ptr(res["mkpts1_c"]), ptr(res["counts"]), cap, stream_ptr(dev))
    check(st, "pope_coarse_match")
    return res


def _strides4(t: torch.Tensor):
    return (C.c_int64 * 4)(*t.stride())


def fine_gather(feat_f0: torch.Tensor, feat_f1: torch.Tensor, b_ids: torch.Tensor, i_ids: torch.Tensor,
                j_ids: torch.Tensor, w0c: int, w1c: int, stride: int, W: int = 5,
                m_dev: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Returns (win0, win1) of shape [M, W*W, Cf] (M = len(b_ids); with `m_dev` rows >= *m_dev are left
    uninitialised).  feat_f* are logical [N, Cf, Hf, Wf] with any strides (channels-last is the fast path)."""
    dev = require_cuda(feat_f0, feat_f1, b_ids, i_ids, j_ids)
    if feat_f0.dtype != feat_f1.dtype:
        raise _lib.PopeError("feat_f0 and feat_f1 must have the same dtype")
    n, Cf, Hf0, Wf0 = feat_f0.shape
    _, _, Hf1, Wf1 = feat_f1.shape
    M = b_ids.shape[0]
    win0 = torch.empty(M, W * W, Cf, dtype=feat_f0.dtype, device=dev)
    win1 = torch.empty(M, W * W, Cf, dtype=feat_f0.dtype, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_fine_gather(ptr(feat_f0), ptr(feat_f1), dtype_code(feat_f0), n, Cf, Hf0, Wf0, _strides4(feat_f0),
                                    Hf1, Wf1, _strides4(feat_f1), int(w0c), int(w1c), int(stride), int(W),
                                    ptr(b_ids), ptr(i_ids), ptr(j_ids), M, ptr(m_dev), ptr(win0), ptr(win1),
                                    stream_ptr(dev))
    check(st, "pope_fine_gather")
    return win0, win1


def fine_match(win0: torch.Tensor, win1: torch.Tensor, mkpts1_c: torch.Tensor, coord_scale: float,
               m_dev: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Returns (expec_f [M,3], mkpts1_f [M,2]);  coord_scale = (W//2) * hw0_i[0]/hw0_f[0]."""
    dev = require_cuda(win0, win1, mkpts1_c)
    if win0.dtype != win1.dtype or win0.shape != win1.shape:
        raise _lib.PopeError("win0 and win1 must have the same dtype and shape")
    win0, win1, mkpts1_c = win0.contiguous(), win1.contiguous(), mkpts1_c.contiguous().float()
    M, WW, Cf = win0.shape
    expec = torch.empty(M, 3, dtype=torch.float32, device=dev)
    mk1f = torch.empty(M, 2, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_fine_match(ptr(win0), ptr(win1), dtype_code(win0), M, ptr(m_dev), WW, Cf, ptr(mkpts1_c),
                                   float(coord_scale), ptr(expec), ptr(mk1f), stream_ptr(dev))
    check(st, "pope_fine_match")
    return expec, mk1f


def _split_packed(mats, device) -> torch.Tensor:
    """Matrices -> their three bf16 planes each (split3_bf16), consecutive: the fp32-accuracy packed layouts."""
    return torch.cat([p.reshape(-1) for t in mats for p in split3_bf16(t.detach().to(device=device, dtype=torch.float32))
                      ]).view(torch.uint8)


def _check_pack_dtype(dtype, what) -> None:
    if dtype not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError(f"the {what} packs for torch.bfloat16 or torch.float32, not {dtype}")


def pack_fine_layer(sd: Dict[str, torch.Tensor], device, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """One LoFTREncoderLayer state dict (d_model 128) -> the packed byte layout of include/pope_b200.h:
    POPE_FINE_TF_LAYER_BYTES for dtype=torch.bfloat16 (the bf16 fine transformer), POPE_FINE_TF_F32_LAYER_BYTES for
    dtype=torch.float32 (the fp32-accuracy one: every matrix as its three bf16 planes, split3_bf16, q | k | v split as one
    stacked [384, 128] matrix)."""
    _check_pack_dtype(dtype, "fine transformer")
    mats = [sd["q_proj.weight"], sd["k_proj.weight"], sd["v_proj.weight"], sd["merge.weight"], sd["mlp.0.weight"],
            sd["mlp.2.weight"]]
    shapes = [(128, 128)] * 4 + [(256, 256), (128, 256)]
    for t, shp in zip(mats, shapes):
        if tuple(t.shape) != shp:
            raise _lib.PopeError(f"fine transformer weight of shape {tuple(t.shape)}, expected {shp} (d_model 128, 8 heads)")
    if dtype == torch.bfloat16:
        w = torch.cat([t.detach().to(device=device, dtype=torch.bfloat16).reshape(-1) for t in mats]).view(torch.uint8)
        size = _lib.FINE_TF_LAYER_BYTES
    else:
        w = _split_packed([torch.cat(mats[:3])] + mats[3:], device)
        size = _lib.FINE_TF_F32_LAYER_BYTES
    ln = torch.cat([sd[k].detach().to(device=device, dtype=torch.float32).reshape(-1)
                    for k in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias")]).view(torch.uint8)
    out = torch.cat([w, ln])
    assert out.numel() == size
    return out


def pack_fine_pre(sd: Dict[str, torch.Tensor], device, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """FinePreprocess state dict (down_proj, merge_feat) -> the packed byte layout of include/pope_b200.h:
    POPE_FINE_PRE_BYTES for dtype=torch.bfloat16, POPE_FINE_PRE_F32_BYTES for dtype=torch.float32 (each matrix as its
    three bf16 planes)."""
    _check_pack_dtype(dtype, "FinePreprocess")
    mats = [sd["down_proj.weight"], sd["merge_feat.weight"]]
    if dtype == torch.bfloat16:
        w = torch.cat([t.detach().to(device=device, dtype=torch.bfloat16).reshape(-1) for t in mats]).view(torch.uint8)
        size = _lib.FINE_PRE_BYTES
    else:
        w = _split_packed(mats, device)
        size = _lib.FINE_PRE_F32_BYTES
    b = torch.cat([sd[k].detach().to(device=device, dtype=torch.float32).reshape(-1)
                   for k in ("down_proj.bias", "merge_feat.bias")]).view(torch.uint8)
    out = torch.cat([w, b])
    assert out.numel() == size
    return out


def _check_m_dev(m_dev: Optional[torch.Tensor], dev) -> None:
    if m_dev is not None and (m_dev.dtype != torch.int32 or m_dev.numel() < 1 or m_dev.device != dev):
        raise _lib.PopeError("m_dev must be a device int32 tensor (the live count) on the device of the windows")


def _fine_dtype(what: str, *tensors: torch.Tensor) -> bool:
    """True for fp32 tensors, False for bf16 ones; anything else (or a mix) raises."""
    dt = tensors[0].dtype
    if dt not in (torch.bfloat16, torch.float32) or any(t.dtype != dt for t in tensors):
        raise _lib.PopeError(f"{what} takes bfloat16 or float32 tensors (all alike)")
    return dt == torch.float32


def _check_packing(packed: torch.Tensor, count: int, f32: bool, bf16_bytes: int, f32_bytes: int, what: str, packer: str):
    per, other = (f32_bytes, bf16_bytes) if f32 else (bf16_bytes, f32_bytes)
    if packed.numel() != count * per:
        if packed.numel() == count * other:
            dt = torch.float32 if f32 else torch.bfloat16
            raise _lib.PopeError(f"{dt} tensors need {what} packed with {packer}(..., dtype={dt})")
        raise _lib.PopeError(f"{what} does not hold the packed bytes of {packer}")


def fine_transformer(feat0: torch.Tensor, feat1: torch.Tensor, packed_layers: torch.Tensor, layer_names,
                     workspace: Optional[torch.Tensor] = None, m_dev: Optional[torch.Tensor] = None
                     ) -> Tuple[torch.Tensor, torch.Tensor]:
    """LocalFeatureTransformer.forward on windows [M, WW, 128], IN PLACE (returns the same tensors).  bfloat16 windows run
    the bf16 fine transformer, float32 windows the fp32-accuracy one; `packed_layers`: concatenation of
    pack_fine_layer(..., dtype=<the windows' dtype>) of every layer, `layer_names`: 'self' / 'cross'.
    `m_dev` (device int32, bf16 only): live window count; M is then the capacity and windows >= *m_dev are left untouched."""
    if m_dev is not None and (feat0.dtype == torch.float32 or feat1.dtype == torch.float32):
        raise _lib.PopeError("the fp32 fine transformer has no device-count bound (m_dev): it runs on all M windows")
    return _fine_transformer(feat0, feat1, packed_layers, layer_names, workspace, m_dev)


def _fine_transformer(feat0, feat1, packed_layers, layer_names, workspace, m_dev):
    """fine_transformer with a device-count bound for either dtype (the fp32 one through pope_fine_transformer_f32_ex,
    which ops.match_pairs_device uses)."""
    dev = require_cuda(feat0, feat1, packed_layers)
    _check_m_dev(m_dev, dev)
    f32 = _fine_dtype("the CUDA fine transformer", feat0, feat1)
    if feat0.shape != feat1.shape or feat0.dim() != 3 or feat0.shape[2] != 128:
        raise _lib.PopeError("feat0 / feat1 must both be [M, WW, 128]")
    if not (feat0.is_contiguous() and feat1.is_contiguous()):
        raise _lib.PopeError("the CUDA fine transformer updates its inputs in place: pass contiguous tensors")
    kinds = []
    for name in layer_names:
        if name not in ("self", "cross"):
            raise KeyError(name)
        kinds.append(0 if name == "self" else 1)
    _check_packing(packed_layers, len(kinds), f32, _lib.FINE_TF_LAYER_BYTES, _lib.FINE_TF_F32_LAYER_BYTES,
                   "packed_layers", "pack_fine_layer")
    M, WW, _ = feat0.shape
    if M == 0:
        return feat0, feat1
    workspace = fine_level_workspace(M, WW, dev, workspace, merge=False, dtype=feat0.dtype)
    arr = (_lib.C.c_int * max(len(kinds), 1))(*kinds)
    fn = lib().pope_fine_transformer_f32_ex if f32 else lib().pope_fine_transformer_ex
    with torch.cuda.device(dev):
        st = fn(ptr(feat0), ptr(feat1), M, ptr(m_dev), WW, ptr(packed_layers), len(kinds), arr, ptr(workspace),
                workspace.numel(), stream_ptr(dev))
    check(st, "pope_fine_transformer_f32" if f32 else "pope_fine_transformer")
    return feat0, feat1


def split3_bf16(w: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """fp32 -> three bf16 terms w1 + w2 + w3 (8 mantissa bits each, every residual exact in fp32): the operand split of the
    fp32-accuracy tensor-core paths (csrc/split3.cuh).  The sum is w exactly for fp32 values down to 2^-110 in
    magnitude; below that the third term runs into the bf16 subnormal range and the sum is w to within 2^-134."""
    w = w.to(torch.float32)
    w1 = w.to(torch.bfloat16)
    r1 = w - w1.float()
    w2 = r1.to(torch.bfloat16)
    w3 = (r1 - w2.float()).to(torch.bfloat16)
    return w1, w2, w3


def pack_coarse_layer(sd: Dict[str, torch.Tensor], device, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """One LoFTREncoderLayer state dict (d_model 256) -> the packed byte layout of include/pope_b200.h:
    POPE_COARSE_TF_LAYER_BYTES for dtype=torch.bfloat16 (the bf16 transformer), POPE_COARSE_TF_F32_LAYER_BYTES for
    dtype=torch.float32 (the fp32-accuracy transformer: every matrix as its three bf16 planes, split3_bf16)."""
    if dtype not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError(f"the coarse transformer packs for torch.bfloat16 or torch.float32, not {dtype}")
    mats = [sd["q_proj.weight"], sd["k_proj.weight"], sd["v_proj.weight"], sd["merge.weight"], sd["mlp.0.weight"],
            sd["mlp.2.weight"]]
    shapes = [(256, 256)] * 4 + [(512, 512), (256, 512)]
    for t, shp in zip(mats, shapes):
        if tuple(t.shape) != shp:
            raise _lib.PopeError(f"coarse transformer weight of shape {tuple(t.shape)}, expected {shp} (d_model 256, 8 heads)")
    for k in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"):
        if tuple(sd[k].shape) != (256,):
            raise _lib.PopeError(f"coarse transformer {k} of shape {tuple(sd[k].shape)}, expected (256,)")
    if dtype == torch.bfloat16:
        w = torch.cat([t.detach().to(device=device, dtype=torch.bfloat16).reshape(-1) for t in mats]).view(torch.uint8)
        size = _lib.COARSE_TF_LAYER_BYTES
    else:
        # q | k | v stacked as one [768, 256] matrix, then split: plane p of a matrix holds term p of every element
        qkv = torch.cat([t.detach().to(device=device, dtype=torch.float32) for t in mats[:3]])
        groups = [qkv] + [t.detach().to(device=device, dtype=torch.float32) for t in mats[3:]]
        w = torch.cat([p.reshape(-1) for g in groups for p in split3_bf16(g)]).view(torch.uint8)
        size = _lib.COARSE_TF_F32_LAYER_BYTES
    ln = torch.cat([sd[k].detach().to(device=device, dtype=torch.float32).reshape(-1)
                    for k in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias")]).view(torch.uint8)
    out = torch.cat([w, ln])
    assert out.numel() == size
    return out


def coarse_transformer(feat0: torch.Tensor, feat1: torch.Tensor, packed_layers: torch.Tensor, layer_names,
                       workspace: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """LocalFeatureTransformer.forward (d_model 256, 8 heads, linear attention, no masks) on token-major features
    feat0 [N, L, 256] and feat1 [N, S, 256], IN PLACE (returns the same tensors).  bfloat16 features run the bf16
    transformer, float32 features the fp32-accuracy one; `packed_layers`: concatenation of
    pack_coarse_layer(..., dtype=<the features' dtype>) of every layer, `layer_names`: 'self' / 'cross'.
    `workspace`: reused when large enough."""
    dev = require_cuda(feat0, feat1, packed_layers)
    if feat0.dtype != feat1.dtype or feat0.dtype not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError("the CUDA coarse transformer takes bfloat16 or float32 features (both sides alike)")
    f32 = feat0.dtype == torch.float32
    if feat0.dim() != 3 or feat1.dim() != 3 or feat0.shape[0] != feat1.shape[0] or feat0.shape[2] != 256 \
            or feat1.shape[2] != 256:
        raise _lib.PopeError("feat0 / feat1 must be [N, L, 256] / [N, S, 256]")
    if not (feat0.is_contiguous() and feat1.is_contiguous()):
        raise _lib.PopeError("the CUDA coarse transformer updates its inputs in place: pass contiguous tensors")
    kinds = []
    for name in layer_names:
        if name not in ("self", "cross"):
            raise KeyError(name)
        kinds.append(0 if name == "self" else 1)
    per_layer = _lib.COARSE_TF_F32_LAYER_BYTES if f32 else _lib.COARSE_TF_LAYER_BYTES
    if packed_layers.numel() != len(kinds) * per_layer:
        other = _lib.COARSE_TF_LAYER_BYTES if f32 else _lib.COARSE_TF_F32_LAYER_BYTES
        if packed_layers.numel() == len(kinds) * other:
            raise _lib.PopeError(f"{feat0.dtype} features need layers packed with pack_coarse_layer(..., dtype={feat0.dtype})")
        raise _lib.PopeError("packed_layers does not hold one packed layer per layer name")
    n, L, S = feat0.shape[0], feat0.shape[1], feat1.shape[1]
    if n == 0 or L == 0 or S == 0:
        return feat0, feat1
    workspace = coarse_tf_workspace(n, L, S, dev, workspace, dtype=feat0.dtype)
    arr = (_lib.C.c_int * max(len(kinds), 1))(*kinds)
    fn, name = ((lib().pope_coarse_transformer_f32, "pope_coarse_transformer_f32") if f32 else
                (lib().pope_coarse_transformer, "pope_coarse_transformer"))
    with torch.cuda.device(dev):
        st = fn(ptr(feat0), ptr(feat1), n, L, S, ptr(packed_layers), len(kinds), arr, ptr(workspace), workspace.numel(),
                stream_ptr(dev))
    check(st, name)
    return feat0, feat1


def coarse_tf_workspace(n: int, L: int, S: int, dev, workspace: Optional[torch.Tensor] = None,
                        dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """Scratch of the CUDA coarse transformer (bf16, or fp32 accuracy for dtype=torch.float32) for n pairs of L and S
    tokens; `workspace` is returned when large enough."""
    if dtype not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError(f"the CUDA coarse transformer runs in torch.bfloat16 or torch.float32, not {dtype}")
    query = lib().pope_coarse_tf_f32_workspace_bytes if dtype == torch.float32 else lib().pope_coarse_tf_workspace_bytes
    need = query(int(n), int(L), int(S))
    if need == 0:
        raise _lib.PopeError(f"coarse transformer shape n={n}, L={L}, S={S} is outside what the kernels index")
    if workspace is None or workspace.numel() < need or workspace.device != dev:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    return workspace


def coarse_pos_encode(feat: torch.Tensor, pe: torch.Tensor, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """PositionEncodingSine + flatten(2).transpose(1, 2) + .to(dtype) in one kernel: feat [N, 256, H, W] fp32 ->
    [N, H*W, 256] contiguous, bit-identical to `(feat + pe[..., :H, :W]).flatten(2).transpose(1, 2).to(dtype)`.
    dtype=torch.bfloat16 (the input of the bf16 coarse transformer) or torch.float32 (the fp32 sum itself, the input of the
    fp32-accuracy one).  `pe`: the encoding's `pe` buffer [1, 256, Hmax, Wmax] fp32."""
    if dtype not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError(f"coarse_pos_encode writes torch.bfloat16 or torch.float32, not {dtype}")
    dev = require_cuda(feat, pe)
    if feat.dtype != torch.float32 or pe.dtype != torch.float32 or feat.dim() != 4 or pe.dim() != 4 or pe.shape[0] != 1:
        raise _lib.PopeError("coarse_pos_encode takes an fp32 [N, C, H, W] map and the fp32 [1, C, Hmax, Wmax] encoding")
    if pe.shape[1] != feat.shape[1]:
        raise _lib.PopeError("the encoding and the map differ in channels")
    feat, pe = feat.contiguous(), pe.contiguous()
    n, c, h, w = feat.shape
    out = torch.empty(n, h * w, c, dtype=dtype, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_coarse_pos_encode_ex(ptr(feat), ptr(pe), n, c, h, w, pe.shape[2], pe.shape[3], ptr(out),
                                             dtype_code(out), stream_ptr(dev))
    check(st, "pope_coarse_pos_encode")
    return out


def fine_merge_coarse(win0: torch.Tensor, win1: torch.Tensor, feat_c0: torch.Tensor, feat_c1: torch.Tensor, b_ids, i_ids,
                      j_ids, packed_pre: torch.Tensor, workspace: Optional[torch.Tensor] = None,
                      m_dev: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """FinePreprocess' down_proj / merge_feat on windows [M, WW, 128], IN PLACE (returns the same tensors): bfloat16
    tensors in bf16, float32 tensors at fp32 accuracy (`packed_pre` from pack_fine_pre(..., dtype=<their dtype>)).
    `m_dev` (device int32, bf16 only): live window count; M is then the capacity and windows / ids >= *m_dev are never
    touched."""
    if m_dev is not None and any(t.dtype == torch.float32 for t in (win0, win1, feat_c0, feat_c1)):
        raise _lib.PopeError("the fp32 fine_merge_coarse has no device-count bound (m_dev): it runs on all M windows")
    return _fine_merge_coarse(win0, win1, feat_c0, feat_c1, b_ids, i_ids, j_ids, packed_pre, workspace, m_dev)


def _fine_merge_coarse(win0, win1, feat_c0, feat_c1, b_ids, i_ids, j_ids, packed_pre, workspace, m_dev):
    """fine_merge_coarse with a device-count bound for either dtype (the fp32 one through pope_fine_merge_coarse_f32_ex,
    which ops.match_pairs_device uses)."""
    dev = require_cuda(win0, win1, feat_c0, feat_c1, b_ids, i_ids, j_ids, packed_pre)
    _check_m_dev(m_dev, dev)
    f32 = _fine_dtype("fine_merge_coarse", win0, win1, feat_c0, feat_c1)
    if not all(t.is_contiguous() for t in (win0, win1, feat_c0, feat_c1)):
        raise _lib.PopeError("fine_merge_coarse takes contiguous tensors")
    _check_packing(packed_pre, 1, f32, _lib.FINE_PRE_BYTES, _lib.FINE_PRE_F32_BYTES, "packed_pre", "pack_fine_pre")
    M, WW, _ = win0.shape
    if M == 0:
        return win0, win1
    n, L, C_ = feat_c0.shape
    S = feat_c1.shape[1]
    workspace = fine_level_workspace(M, WW, dev, workspace, transformer=False, dtype=win0.dtype)
    ids = (ptr(b_ids.contiguous()), ptr(i_ids.contiguous()), ptr(j_ids.contiguous()))
    fn = lib().pope_fine_merge_coarse_f32_ex if f32 else lib().pope_fine_merge_coarse_ex
    with torch.cuda.device(dev):
        st = fn(ptr(win0), ptr(win1), M, ptr(m_dev), WW, ptr(feat_c0), ptr(feat_c1), L, S, C_, *ids, ptr(packed_pre),
                ptr(workspace), workspace.numel(), stream_ptr(dev))
    check(st, "pope_fine_merge_coarse_f32" if f32 else "pope_fine_merge_coarse")
    return win0, win1


def match_order_by_ref(counts: torch.Tensor, n_pairs: int, S: int, j_ids: torch.Tensor) -> torch.Tensor:
    """order[k] = index of the k-th match in (pair, reference cell) order; see pope_match_order_by_ref."""
    dev = require_cuda(counts, j_ids)
    order = torch.empty(j_ids.shape[0], dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_match_order_by_ref(ptr(counts), int(n_pairs), int(S), ptr(j_ids), ptr(order), stream_ptr(dev))
    check(st, "pope_match_order_by_ref")
    return order


def fine_match_maps(feat_f0: torch.Tensor, feat_f1: torch.Tensor, b_ids, i_ids, j_ids, mkpts1_c: torch.Tensor,
                    w0c: int, w1c: int, stride: int, coord_scale: float, W: int = 5,
                    m_dev: Optional[torch.Tensor] = None, order: Optional[torch.Tensor] = None
                    ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Fused fine_gather + fine_match on channels-last maps (no windows materialised); same results.  `order`:
    optional processing order from `match_order_by_ref` (outputs do not depend on it)."""
    dev = require_cuda(feat_f0, feat_f1, b_ids, i_ids, j_ids, mkpts1_c)
    if feat_f0.dtype != feat_f1.dtype:
        raise _lib.PopeError("feat_f0 and feat_f1 must have the same dtype")
    n, Cf, Hf0, Wf0 = feat_f0.shape
    _, _, Hf1, Wf1 = feat_f1.shape
    M = b_ids.shape[0]
    expec = torch.empty(M, 3, dtype=torch.float32, device=dev)
    mk1f = torch.empty(M, 2, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_fine_match_maps(ptr(feat_f0), ptr(feat_f1), dtype_code(feat_f0), n, Cf, Hf0, Wf0,
                                        _strides4(feat_f0), Hf1, Wf1, _strides4(feat_f1), int(w0c), int(w1c),
                                        int(stride), int(W), ptr(b_ids), ptr(i_ids), ptr(j_ids), M, ptr(m_dev),
                                        ptr(order), ptr(mkpts1_c), float(coord_scale), ptr(expec), ptr(mk1f),
                                        stream_ptr(dev))
    check(st, "pope_fine_match_maps")
    return expec, mk1f


def match_scores(mconf: torch.Tensor, counts: torch.Tensor, n_pairs: int, group: int = 3, thr: float = 0.9
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
    """(scores [n_pairs] int32, best [ceil(n_pairs/group)] int32): per-pair count of mconf > thr and, per group of
    consecutive pairs, the first arg-max -- the `matching_score` / `np.argmax` of eval_linemod_json.py:118-119,146."""
    dev = require_cuda(mconf, counts)
    scores = torch.empty(n_pairs, dtype=torch.int32, device=dev)
    best = torch.empty((n_pairs + group - 1) // group, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_match_scores(ptr(mconf), ptr(counts), int(n_pairs), int(group), float(thr), ptr(scores), ptr(best),
                                     stream_ptr(dev))
    check(st, "pope_match_scores")
    return scores, best


def cosine_topk(q: torch.Tensor, refs: torch.Tensor, k: int = 3, eps: float = 1e-8):
    """q [1,D] or [D], refs [R,D] -> (scores [R], slot_scores [k], slot_idx [k] int32; -1 = empty slot)."""
    dev = require_cuda(q, refs)
    q, refs = q.reshape(-1).contiguous(), refs.contiguous()
    if q.dtype != refs.dtype or q.shape[0] != refs.shape[1]:
        raise _lib.PopeError("q and refs must share dtype and feature dimension")
    R, D = refs.shape
    scores = torch.empty(R, dtype=torch.float32, device=dev)
    slot_s = torch.empty(k, dtype=torch.float32, device=dev)
    slot_i = torch.empty(k, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_cosine_topk(ptr(q), ptr(refs), dtype_code(q), R, D, k, float(eps), ptr(scores), ptr(slot_s),
                                    ptr(slot_i), stream_ptr(dev))
    check(st, "pope_cosine_topk")
    return scores, slot_s, slot_i


def running_topk(scores: torch.Tensor, k: int = 3):
    """The running top-k of eval_linemod_json.py:95-101 over device scores [R] in crop order -> (slot_scores [k],
    slot_idx [k] int32; -1 = empty slot)."""
    dev = require_cuda(scores)
    scores = scores.reshape(-1).contiguous().float()
    slot_s = torch.empty(k, dtype=torch.float32, device=dev)
    slot_i = torch.empty(k, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_running_topk(ptr(scores), scores.numel(), k, ptr(slot_s), ptr(slot_i), stream_ptr(dev))
    check(st, "pope_running_topk")
    return slot_s, slot_i


def fine_level_workspace(m: int, ww: int, dev, workspace: Optional[torch.Tensor] = None, merge: bool = True,
                         transformer: bool = True, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """Scratch of the fine level for m windows of ww tokens (bf16, or fp32 accuracy for dtype=torch.float32), sized for
    the stages that will use it: the FinePreprocess Linears (`merge`) and the fine transformer (`transformer`, 5 planes of
    [m * ww, 128] bf16; in fp32, 5 fp32 planes and 9 bf16 split planes).  They run one after the other on one stream, so
    with both the scratch is shared (at 25 tokens its size is the transformer's).  A stage that is handed no scratch gets
    one of its own size only, so a caller that does not share pays for no more than it uses."""
    if dtype not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError(f"the CUDA fine level runs in torch.bfloat16 or torch.float32, not {dtype}")
    h = lib()
    tf, mg = ((h.pope_fine_tf_f32_workspace_bytes, h.pope_fine_merge_f32_workspace_bytes) if dtype == torch.float32 else
              (h.pope_fine_tf_workspace_bytes, h.pope_fine_merge_workspace_bytes))
    need = max(tf(int(m), int(ww)) if transformer else 0, mg(int(m)) if merge else 0, 16)
    if workspace is None or workspace.numel() < need or workspace.device != dev:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    return workspace


def _fine_level_dtype(fine_level: dict) -> torch.dtype:
    """The packing of a fine-level bundle (`Matcher.fine_level`): its "dtype" entry; a bundle without one is bf16."""
    dt = fine_level.get("dtype", torch.bfloat16)
    if dt not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError(f"a fine level is packed for torch.bfloat16 or torch.float32, not {dt}")
    return dt


def _check_fine_level_inputs(feat_c0, feat_c1, feat_f0, feat_f1, W, dtype, coarse_features: bool = True) -> None:
    """`coarse_features=False`: feat_c0 / feat_c1 are backbone maps that a coarse level turns into the features."""
    require_cuda(feat_c0, feat_c1, feat_f0, feat_f1)
    name = "bf16" if dtype == torch.bfloat16 else "fp32"
    if coarse_features and (feat_c0.dtype != dtype or feat_c1.dtype != dtype or feat_c0.shape[-1] != 256):
        raise _lib.PopeError(f"the {name} fine level takes {dtype} coarse features with C = 256")
    if feat_f0.dtype != dtype or feat_f1.dtype != dtype or feat_f0.shape[1] != 128 or feat_f1.shape[1] != 128:
        raise _lib.PopeError(f"the {name} fine level takes {dtype} fine maps with Cf = 128")
    if W != 5:
        raise _lib.PopeError(f"the {name} fine level takes 5 x 5 windows")


def _check_coarse_level(coarse_level: dict, fine_level: Optional[dict], feat_c0, feat_c1, hw0_c, hw1_c) -> torch.dtype:
    """What the coarse level of the step needs, checked before any launch; returns the bundle's dtype."""
    dt = coarse_level.get("dtype")
    if dt not in (torch.bfloat16, torch.float32):
        raise _lib.PopeError(f"a coarse level is packed for torch.bfloat16 or torch.float32, not {dt}")
    if fine_level is not None and _fine_level_dtype(fine_level) != dt:
        raise _lib.PopeError(f"a coarse level of {dt} with a fine level of {_fine_level_dtype(fine_level)}: the step runs "
                             "both levels in one dtype")
    pe, layers, names = coarse_level["pe"], coarse_level["layers"], list(coarse_level["layer_names"])
    for t in (feat_c0, feat_c1):
        if t.dtype != torch.float32 or t.dim() != 4:
            raise _lib.PopeError("with a coarse level, feat_c0 / feat_c1 are the backbone's fp32 maps [N, 256, Hc, Wc]")
        if t.shape[1] != 256:
            raise _lib.PopeError(f"the coarse level takes maps with C = 256, not {t.shape[1]}")
    if feat_c0.shape[0] != feat_c1.shape[0]:
        raise _lib.PopeError("feat_c0 and feat_c1 hold different numbers of pairs")
    for t, hw in ((feat_c0, hw0_c), (feat_c1, hw1_c)):
        if tuple(t.shape[2:]) != (int(hw[0]), int(hw[1])):
            raise _lib.PopeError(f"a coarse map of grid {tuple(t.shape[2:])} with hw_c = {tuple(hw)}")
        if pe.dim() != 4 or pe.shape[1] != 256 or t.shape[2] > pe.shape[2] or t.shape[3] > pe.shape[3]:
            raise _lib.PopeError(f"a coarse grid of {tuple(t.shape[2:])} is larger than the position encoding "
                                 f"{tuple(pe.shape[2:])}")
    per_layer = _lib.COARSE_TF_F32_LAYER_BYTES if dt == torch.float32 else _lib.COARSE_TF_LAYER_BYTES
    if not names or any(nm not in ("self", "cross") for nm in names) or layers.numel() != len(names) * per_layer:
        raise _lib.PopeError("the coarse level's layer names and packed layers do not agree")
    require_cuda(feat_c0, feat_c1, pe, layers)
    return dt


def match_pairs_device(feat_c0, feat_c1, feat_f0, feat_f1, hw0_i, hw0_c, hw1_c, thr=0.2, border_rm=2,
                       temperature=0.1, W=5, impl=_lib.COARSE_AUTO, workspace=None, fused_fine=None, fine_level=None,
                       fine_workspace=None, coarse_level=None, coarse_workspace=None) -> CoarseResult:
    """The hot path on device-resident inputs with NO host synchronisation: coarse match -> window gather ->
    fine match, the match count staying on the device (`m_dev`).  Returns the capacity-sized CoarseResult
    extended with `expec_f`, `mkpts0_f`, `mkpts1_f` (and `win0`, `win1` on the unfused route).

    `fine_level` (`Matcher.fine_level(device)`): also run what Matcher.forward runs between gather and fine matching --
    FinePreprocess' two Linears and the fine transformer, in bf16 (csrc/fine_tf.cu) -- so that the step computes what
    `Matcher(config, fine_cuda_bf16=True)` computes, bit for bit on the live rows, still without a host sync: every launch
    is bounded by the device match count.  Needs bf16 coarse features (C = 256), bf16 fine maps (Cf = 128) and W = 5, and
    takes the unfused route.  The result then also holds `fine_workspace` (pass it back in to reuse it).  Memory is sized
    by the capacity n * L, not by the match count: at 64 pairs x 480x640 (307 200 windows) that is 3.9 GB of windows plus
    9.8 GB of fine scratch per call, about 13.8 GB; the Matcher flow, sized by the count, needs about half of that at the
    synthetic inputs' match rate.

    `fine_level=Matcher.fine_level(device, dtype=torch.float32)`: the fp32-accuracy level instead (gather -> FinePreprocess
    Linears -> fine transformer -> fine match, every launch bounded by the device count, no host sync), which computes what
    `Matcher(config, fine_cuda_fp32=True)` computes, bit for bit on the live rows.  The bundle's dtype selects the level;
    coarse features and fine maps must then both be float32 (any mix raises).  Its cost, from the workspace formulas (not
    measured): at 64 pairs x 480x640 (307 200 windows) 7.9 GB of fp32 windows plus 37.4 GB of fine scratch per call.

    `coarse_level` (`Matcher.coarse_level(device, dtype)`): start where the backbone stops.  feat_c0 / feat_c1 are then the
    backbone's fp32 coarse maps [N, 256, Hc, Wc] with (Hc, Wc) = hw0_c / hw1_c; the step adds the position encoding and lays
    them out token-major in the bundle's dtype (`coarse_pos_encode`), runs the coarse transformer on them in place
    (`coarse_transformer`), and continues as above on the transformed features -- what
    `Matcher(config, coarse_cuda_bf16=True)` (bf16 bundle) or `coarse_cuda_fp32=True` (fp32 bundle) computes after its
    backbone, bit for bit, still without a host sync.  The result also holds `feat_c0` / `feat_c1` (the transformed
    features, what `Matcher.forward(data, only_att_fea=True)` returns) and `coarse_workspace` (pass it back in to reuse
    it; from the workspace formulas about 0.8 GB in bf16 and 3.0 GB in fp32 at 64 pairs x 480x640, not measured).  A
    coarse level goes alone or with a fine level of the same dtype; any other mix, maps that are not fp32 4-D, C != 256,
    a grid other than hw_c or larger than the encoding raise `PopeError` before any launch."""
    coarse_dtype = None
    if coarse_level is not None:
        coarse_dtype = _check_coarse_level(coarse_level, fine_level, feat_c0, feat_c1, hw0_c, hw1_c)
    if fine_level is not None:
        level_dtype = _fine_level_dtype(fine_level)
        _check_fine_level_inputs(feat_c0, feat_c1, feat_f0, feat_f1, W, level_dtype, coarse_features=coarse_dtype is None)
        if fused_fine:
            raise _lib.PopeError("fine_level runs between window gather and fine matching: it takes the unfused route")
        fused_fine = False
    if coarse_level is not None:
        feat_c0 = coarse_pos_encode(feat_c0, coarse_level["pe"], coarse_dtype)
        feat_c1 = coarse_pos_encode(feat_c1, coarse_level["pe"], coarse_dtype)
        coarse_workspace = coarse_tf_workspace(feat_c0.shape[0], feat_c0.shape[1], feat_c1.shape[1], feat_c0.device,
                                               coarse_workspace, dtype=coarse_dtype)
        coarse_transformer(feat_c0, feat_c1, coarse_level["layers"], coarse_level["layer_names"], coarse_workspace)
    res = coarse_match(feat_c0, feat_c1, hw0_c, hw1_c, hw0_i[0] / hw0_c[0], thr, border_rm, temperature, impl, workspace)
    if coarse_level is not None:
        res.update(feat_c0=feat_c0, feat_c1=feat_c1, coarse_workspace=coarse_workspace)
    n = res["n_pairs"]
    m_dev = res["counts"][n:n + 1]
    stride = feat_f0.shape[2] // hw0_c[0]
    coord_scale = (W // 2) * (hw0_i[0] / feat_f0.shape[2])
    if fused_fine is None:      # fused kernel needs channels-last maps; plain NCHW takes the two-kernel route
        fused_fine = feat_f0.stride(1) == 1 and feat_f1.stride(1) == 1 and feat_f0.shape[1] == 128 and W == 5
    if fine_level is not None:
        win0, win1 = fine_gather(feat_f0, feat_f1, res["b_ids"], res["i_ids"], res["j_ids"], hw0_c[1], hw1_c[1],
                                 stride, W, m_dev)
        cap = win0.shape[0]
        fine_workspace = fine_level_workspace(cap, W * W, win0.device, fine_workspace, dtype=level_dtype)
        if fine_level["pre"] is not None:
            _fine_merge_coarse(win0, win1, feat_c0.contiguous(), feat_c1.contiguous(), res["b_ids"], res["i_ids"],
                               res["j_ids"], fine_level["pre"], fine_workspace, m_dev)
        _fine_transformer(win0, win1, fine_level["layers"], fine_level["layer_names"], fine_workspace, m_dev)
        expec, mk1f = fine_match(win0, win1, res["mkpts1_c"], coord_scale, m_dev)
        res.update(win0=win0, win1=win1, fine_workspace=fine_workspace)
    elif fused_fine:
        # (match_order_by_ref + order= was measured neutral on B200: 10 us of sorting buys 13 us of gather; not used)
        expec, mk1f = fine_match_maps(feat_f0, feat_f1, res["b_ids"], res["i_ids"], res["j_ids"], res["mkpts1_c"],
                                      hw0_c[1], hw1_c[1], stride, coord_scale, W, m_dev)
    else:
        win0, win1 = fine_gather(feat_f0, feat_f1, res["b_ids"], res["i_ids"], res["j_ids"], hw0_c[1], hw1_c[1],
                                 stride, W, m_dev)
        expec, mk1f = fine_match(win0, win1, res["mkpts1_c"], coord_scale, m_dev)
        res.update(win0=win0, win1=win1)
    res.update(expec_f=expec, mkpts0_f=res["mkpts0_c"], mkpts1_f=mk1f)
    return res


def scratch_views(workspace: torch.Tensor, n: int, L: int, S: int) -> Dict[str, torch.Tensor]:
    """Debug/test view of the coarse scratch (layout of carve_coarse_scratch in csrc/common.cuh): the row/column
    log-sum-exp (log2 units), the best-candidate records, and the single sweep's column partial sums / shifts / per-pair
    flags left by the last pope_coarse_match call."""
    def up(x):
        return (x + 255) // 256 * 256
    G, B = (L + 31) // 32, (S + 31) // 32
    off, out = 0, {}
    for name, nbytes, dt, shape in (("rowbest", 8 * n * L, torch.int64, (n, L)), ("colbest", 8 * n * S, torch.int64, (n, S)),
                                    ("cand_cnt", 8 * n * L, torch.int16, (n, L, 4)), ("ready", 4 * (n + 1), torch.int32, (n + 1,)),
                                    ("lse_r", 4 * n * L, torch.float32, (n, L)), ("lse_c", 4 * n * S, torch.float32, (n, S)),
                                    ("cand", 8 * n * L * 4 * 24, torch.int64, (n, L, 16, 6)),
                                    ("cbound", 4 * n * G * 32, torch.float32, (n, G * 32)), ("cminb", 4 * n * G, torch.float32, (n, G)),
                                    ("colpart", 4 * n * G * S, torch.float32, (n, G, S)), ("cshift", 4 * n * G * B, torch.float32, (n, G, B)),
                                    ("pairflag", 4 * n, torch.int32, (n,))):
        out[name] = workspace[off:off + nbytes].view(dt).view(*shape)
        off += up(nbytes)
    return out
