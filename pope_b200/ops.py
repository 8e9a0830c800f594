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


def pack_fine_layer(sd: Dict[str, torch.Tensor], device) -> torch.Tensor:
    """One LoFTREncoderLayer state dict (d_model 128) -> the packed byte layout of include/pope_b200.h."""
    mats = [sd["q_proj.weight"], sd["k_proj.weight"], sd["v_proj.weight"], sd["merge.weight"], sd["mlp.0.weight"],
            sd["mlp.2.weight"]]
    shapes = [(128, 128)] * 4 + [(256, 256), (128, 256)]
    for t, shp in zip(mats, shapes):
        if tuple(t.shape) != shp:
            raise _lib.PopeError(f"fine transformer weight of shape {tuple(t.shape)}, expected {shp} (d_model 128, 8 heads)")
    w = torch.cat([t.detach().to(device=device, dtype=torch.bfloat16).reshape(-1) for t in mats]).view(torch.uint8)
    ln = torch.cat([sd[k].detach().to(device=device, dtype=torch.float32).reshape(-1)
                    for k in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias")]).view(torch.uint8)
    out = torch.cat([w, ln])
    assert out.numel() == _lib.FINE_TF_LAYER_BYTES
    return out


def pack_fine_pre(sd: Dict[str, torch.Tensor], device) -> torch.Tensor:
    """FinePreprocess state dict (down_proj, merge_feat) -> the packed byte layout of include/pope_b200.h."""
    w = torch.cat([sd[k].detach().to(device=device, dtype=torch.bfloat16).reshape(-1)
                   for k in ("down_proj.weight", "merge_feat.weight")]).view(torch.uint8)
    b = torch.cat([sd[k].detach().to(device=device, dtype=torch.float32).reshape(-1)
                   for k in ("down_proj.bias", "merge_feat.bias")]).view(torch.uint8)
    out = torch.cat([w, b])
    assert out.numel() == _lib.FINE_PRE_BYTES
    return out


def _check_m_dev(m_dev: Optional[torch.Tensor], dev) -> None:
    if m_dev is not None and (m_dev.dtype != torch.int32 or m_dev.numel() < 1 or m_dev.device != dev):
        raise _lib.PopeError("m_dev must be a device int32 tensor (the live count) on the device of the windows")


def fine_transformer(feat0: torch.Tensor, feat1: torch.Tensor, packed_layers: torch.Tensor, layer_names,
                     workspace: Optional[torch.Tensor] = None, m_dev: Optional[torch.Tensor] = None
                     ) -> Tuple[torch.Tensor, torch.Tensor]:
    """LocalFeatureTransformer.forward on bf16 windows [M, WW, 128], IN PLACE (returns the same tensors).
    `packed_layers`: concatenation of pack_fine_layer() of every layer, `layer_names`: 'self' / 'cross'.
    `m_dev` (device int32): live window count; M is then the capacity and windows >= *m_dev are left untouched."""
    dev = require_cuda(feat0, feat1, packed_layers)
    _check_m_dev(m_dev, dev)
    if feat0.dtype != torch.bfloat16 or feat1.dtype != torch.bfloat16:
        raise _lib.PopeError("the CUDA fine transformer takes bfloat16 windows")
    if feat0.shape != feat1.shape or feat0.dim() != 3 or feat0.shape[2] != 128:
        raise _lib.PopeError("feat0 / feat1 must both be [M, WW, 128]")
    if not (feat0.is_contiguous() and feat1.is_contiguous()):
        raise _lib.PopeError("the CUDA fine transformer updates its inputs in place: pass contiguous tensors")
    kinds = []
    for name in layer_names:
        if name not in ("self", "cross"):
            raise KeyError(name)
        kinds.append(0 if name == "self" else 1)
    if packed_layers.numel() != len(kinds) * _lib.FINE_TF_LAYER_BYTES:
        raise _lib.PopeError("packed_layers does not hold one packed layer per layer name")
    M, WW, _ = feat0.shape
    if M == 0:
        return feat0, feat1
    workspace = fine_level_workspace(M, WW, dev, workspace, merge=False)
    arr = (_lib.C.c_int * max(len(kinds), 1))(*kinds)
    with torch.cuda.device(dev):
        st = lib().pope_fine_transformer_ex(ptr(feat0), ptr(feat1), M, ptr(m_dev), WW, ptr(packed_layers), len(kinds), arr,
                                            ptr(workspace), workspace.numel(), stream_ptr(dev))
    check(st, "pope_fine_transformer")
    return feat0, feat1


def pack_coarse_layer(sd: Dict[str, torch.Tensor], device) -> torch.Tensor:
    """One LoFTREncoderLayer state dict (d_model 256) -> the packed byte layout of include/pope_b200.h
    (POPE_COARSE_TF_LAYER_BYTES)."""
    mats = [sd["q_proj.weight"], sd["k_proj.weight"], sd["v_proj.weight"], sd["merge.weight"], sd["mlp.0.weight"],
            sd["mlp.2.weight"]]
    shapes = [(256, 256)] * 4 + [(512, 512), (256, 512)]
    for t, shp in zip(mats, shapes):
        if tuple(t.shape) != shp:
            raise _lib.PopeError(f"coarse transformer weight of shape {tuple(t.shape)}, expected {shp} (d_model 256, 8 heads)")
    for k in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"):
        if tuple(sd[k].shape) != (256,):
            raise _lib.PopeError(f"coarse transformer {k} of shape {tuple(sd[k].shape)}, expected (256,)")
    w = torch.cat([t.detach().to(device=device, dtype=torch.bfloat16).reshape(-1) for t in mats]).view(torch.uint8)
    ln = torch.cat([sd[k].detach().to(device=device, dtype=torch.float32).reshape(-1)
                    for k in ("norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias")]).view(torch.uint8)
    out = torch.cat([w, ln])
    assert out.numel() == _lib.COARSE_TF_LAYER_BYTES
    return out


def coarse_transformer(feat0: torch.Tensor, feat1: torch.Tensor, packed_layers: torch.Tensor, layer_names,
                       workspace: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """LocalFeatureTransformer.forward (d_model 256, 8 heads, linear attention, no masks) on bf16 token-major features
    feat0 [N, L, 256] and feat1 [N, S, 256], IN PLACE (returns the same tensors).  `packed_layers`: concatenation of
    pack_coarse_layer() of every layer, `layer_names`: 'self' / 'cross'.  `workspace`: reused when large enough."""
    dev = require_cuda(feat0, feat1, packed_layers)
    if feat0.dtype != torch.bfloat16 or feat1.dtype != torch.bfloat16:
        raise _lib.PopeError("the CUDA coarse transformer takes bfloat16 features")
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
    if packed_layers.numel() != len(kinds) * _lib.COARSE_TF_LAYER_BYTES:
        raise _lib.PopeError("packed_layers does not hold one packed layer per layer name")
    n, L, S = feat0.shape[0], feat0.shape[1], feat1.shape[1]
    if n == 0 or L == 0 or S == 0:
        return feat0, feat1
    workspace = coarse_tf_workspace(n, L, S, dev, workspace)
    arr = (_lib.C.c_int * max(len(kinds), 1))(*kinds)
    with torch.cuda.device(dev):
        st = lib().pope_coarse_transformer(ptr(feat0), ptr(feat1), n, L, S, ptr(packed_layers), len(kinds), arr,
                                           ptr(workspace), workspace.numel(), stream_ptr(dev))
    check(st, "pope_coarse_transformer")
    return feat0, feat1


def coarse_tf_workspace(n: int, L: int, S: int, dev, workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Scratch of the CUDA coarse transformer for n pairs of L and S tokens; `workspace` is returned when large enough."""
    need = lib().pope_coarse_tf_workspace_bytes(int(n), int(L), int(S))
    if need == 0:
        raise _lib.PopeError(f"coarse transformer shape n={n}, L={L}, S={S} is outside what the kernels index")
    if workspace is None or workspace.numel() < need or workspace.device != dev:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    return workspace


def coarse_pos_encode(feat: torch.Tensor, pe: torch.Tensor) -> torch.Tensor:
    """PositionEncodingSine + flatten(2).transpose(1, 2) + .to(torch.bfloat16) in one kernel: feat [N, 256, H, W] fp32 ->
    [N, H*W, 256] bf16, bit-identical to `(feat + pe[..., :H, :W]).flatten(2).transpose(1, 2).to(torch.bfloat16)`.
    `pe`: the encoding's `pe` buffer [1, 256, Hmax, Wmax] fp32."""
    dev = require_cuda(feat, pe)
    if feat.dtype != torch.float32 or pe.dtype != torch.float32 or feat.dim() != 4 or pe.dim() != 4 or pe.shape[0] != 1:
        raise _lib.PopeError("coarse_pos_encode takes an fp32 [N, C, H, W] map and the fp32 [1, C, Hmax, Wmax] encoding")
    if pe.shape[1] != feat.shape[1]:
        raise _lib.PopeError("the encoding and the map differ in channels")
    feat, pe = feat.contiguous(), pe.contiguous()
    n, c, h, w = feat.shape
    out = torch.empty(n, h * w, c, dtype=torch.bfloat16, device=dev)
    with torch.cuda.device(dev):
        st = lib().pope_coarse_pos_encode(ptr(feat), ptr(pe), n, c, h, w, pe.shape[2], pe.shape[3], ptr(out), stream_ptr(dev))
    check(st, "pope_coarse_pos_encode")
    return out


def fine_merge_coarse(win0: torch.Tensor, win1: torch.Tensor, feat_c0: torch.Tensor, feat_c1: torch.Tensor, b_ids, i_ids,
                      j_ids, packed_pre: torch.Tensor, workspace: Optional[torch.Tensor] = None,
                      m_dev: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """FinePreprocess' down_proj / merge_feat on bf16 windows [M, WW, 128], IN PLACE (returns the same tensors).
    `m_dev` (device int32): live window count; M is then the capacity and windows / ids >= *m_dev are never touched."""
    dev = require_cuda(win0, win1, feat_c0, feat_c1, b_ids, i_ids, j_ids, packed_pre)
    _check_m_dev(m_dev, dev)
    for t in (win0, win1, feat_c0, feat_c1):
        if t.dtype != torch.bfloat16 or not t.is_contiguous():
            raise _lib.PopeError("fine_merge_coarse takes contiguous bfloat16 tensors")
    M, WW, _ = win0.shape
    if M == 0:
        return win0, win1
    n, L, C_ = feat_c0.shape
    S = feat_c1.shape[1]
    workspace = fine_level_workspace(M, WW, dev, workspace, transformer=False)
    with torch.cuda.device(dev):
        st = lib().pope_fine_merge_coarse_ex(ptr(win0), ptr(win1), M, ptr(m_dev), WW, ptr(feat_c0), ptr(feat_c1), L, S, C_,
                                             ptr(b_ids.contiguous()), ptr(i_ids.contiguous()), ptr(j_ids.contiguous()),
                                             ptr(packed_pre), ptr(workspace), workspace.numel(), stream_ptr(dev))
    check(st, "pope_fine_merge_coarse")
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
                         transformer: bool = True) -> torch.Tensor:
    """Scratch of the bf16 fine level for m windows of ww tokens, sized for the stages that will use it: the FinePreprocess
    Linears (`merge`) and the fine transformer (`transformer`, 5 planes of [m * ww, 128] bf16).  They run one after the
    other on one stream, so with both the scratch is shared (at 25 tokens its size is the transformer's).  A stage that
    is handed no scratch gets one of its own size only, so a caller that does not share pays for no more than it uses."""
    need = max(lib().pope_fine_tf_workspace_bytes(int(m), int(ww)) if transformer else 0,
               lib().pope_fine_merge_workspace_bytes(int(m)) if merge else 0, 16)
    if workspace is None or workspace.numel() < need or workspace.device != dev:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    return workspace


def _check_fine_level_inputs(feat_c0, feat_c1, feat_f0, feat_f1, W) -> None:
    require_cuda(feat_c0, feat_c1, feat_f0, feat_f1)
    if feat_c0.dtype != torch.bfloat16 or feat_c1.dtype != torch.bfloat16 or feat_c0.shape[-1] != 256:
        raise _lib.PopeError("the bf16 fine level takes bfloat16 coarse features with C = 256")
    if feat_f0.dtype != torch.bfloat16 or feat_f1.dtype != torch.bfloat16 or feat_f0.shape[1] != 128 \
            or feat_f1.shape[1] != 128:
        raise _lib.PopeError("the bf16 fine level takes bfloat16 fine maps with Cf = 128")
    if W != 5:
        raise _lib.PopeError("the bf16 fine level takes 5 x 5 windows")


def match_pairs_device(feat_c0, feat_c1, feat_f0, feat_f1, hw0_i, hw0_c, hw1_c, thr=0.2, border_rm=2,
                       temperature=0.1, W=5, impl=_lib.COARSE_AUTO, workspace=None, fused_fine=None, fine_level=None,
                       fine_workspace=None) -> CoarseResult:
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
    synthetic inputs' match rate."""
    if fine_level is not None:
        _check_fine_level_inputs(feat_c0, feat_c1, feat_f0, feat_f1, W)
        if fused_fine:
            raise _lib.PopeError("fine_level runs between window gather and fine matching: it takes the unfused route")
        fused_fine = False
    res = coarse_match(feat_c0, feat_c1, hw0_c, hw1_c, hw0_i[0] / hw0_c[0], thr, border_rm, temperature, impl, workspace)
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
        fine_workspace = fine_level_workspace(cap, W * W, win0.device, fine_workspace)
        if fine_level["pre"] is not None:
            fine_merge_coarse(win0, win1, feat_c0.contiguous(), feat_c1.contiguous(), res["b_ids"], res["i_ids"],
                              res["j_ids"], fine_level["pre"], fine_workspace, m_dev)
        fine_transformer(win0, win1, fine_level["layers"], fine_level["layer_names"], fine_workspace, m_dev)
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
