"""ctypes binding of libpope_b200.so (include/pope_b200.h).  No fallback: a missing library, a missing
symbol or a non-zero status raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpope_b200.so")

POPE_F32, POPE_BF16 = 0, 1
COARSE_AUTO, COARSE_SIMT, COARSE_TCGEN05 = 0, 1, 2
FLAG_NONFINITE_LSE = 1
FLAG_CAND_OVERFLOW = 2
FLAG_ROBUST_PATH = 4
FLAG_CAPACITY = 8
FINE_TF_LAYER_BYTES = 329728      # include/pope_b200.h: packed weights of one LoFTREncoderLayer (d_model 128)
FINE_PRE_BYTES = 132096           # ... of FinePreprocess' down_proj + merge_feat
COARSE_TF_LAYER_BYTES = 1314816   # ... of one d_model-256 LoFTREncoderLayer (the coarse transformer)

_p, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/pope_b200.h one to one
SIGNATURES = {
    "pope_abi_version": (_i, []),
    "pope_status_string": (C.c_char_p, [_i]),
    "pope_coarse_auto_impl": (_i, [_i, _i, _i, _i]),
    "pope_coarse_workspace_bytes": (_sz, [_i, _i, _i]),
    "pope_coarse_workspace_bytes_ex": (_sz, [_i, _i, _i, _i, _i]),
    "pope_coarse_match": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _i, _i, _p, _sz,
                               _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "pope_fine_gather": (_i, [_p, _p, _i, _i, _i, _i, _i, C.POINTER(_i64), _i, _i, C.POINTER(_i64),
                              _i, _i, _i, _i, _p, _p, _p, _i64, _p, _p, _p, _p]),
    "pope_fine_match": (_i, [_p, _p, _i, _i64, _p, _i, _i, _p, _f, _p, _p, _p]),
    "pope_fine_match_maps": (_i, [_p, _p, _i, _i, _i, _i, _i, C.POINTER(_i64), _i, _i, C.POINTER(_i64),
                                  _i, _i, _i, _i, _p, _p, _p, _i64, _p, _p, _p, _f, _p, _p, _p]),
    "pope_fine_tf_workspace_bytes": (_sz, [_i64, _i]),
    "pope_fine_merge_workspace_bytes": (_sz, [_i64]),
    "pope_fine_transformer": (_i, [_p, _p, _i64, _i, _p, _i, C.POINTER(_i), _p, _sz, _p]),
    "pope_fine_merge_coarse": (_i, [_p, _p, _i64, _i, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "pope_fine_transformer_ex": (_i, [_p, _p, _i64, _p, _i, _p, _i, C.POINTER(_i), _p, _sz, _p]),
    "pope_fine_merge_coarse_ex": (_i, [_p, _p, _i64, _p, _i, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "pope_coarse_tf_workspace_bytes": (_sz, [_i64, _i, _i]),
    "pope_coarse_transformer": (_i, [_p, _p, _i64, _i, _i, _p, _i, C.POINTER(_i), _p, _sz, _p]),
    "pope_coarse_pos_encode": (_i, [_p, _p, _i64, _i, _i, _i, _i, _i, _p, _p]),
    "pope_match_order_by_ref": (_i, [_p, _i, _i, _p, _p, _p]),
    "pope_savetxt_f32": (_i, [C.c_char_p, _p, _i64, _i]),
    "pope_savetxt_f64": (_i, [C.c_char_p, _p, _i64, _i]),
    "pope_write_match_files": (_i, [C.c_char_p, C.POINTER(C.c_char_p), _i, _p, _p, _p, _i64, _i, _i, C.POINTER(C.c_int32)]),
    "pope_loadtxt_f64": (_i, [C.c_char_p, _p, _i64, C.POINTER(_i64), C.POINTER(_i)]),
    "pope_read_match_files": (_i, [C.c_char_p, C.POINTER(C.c_char_p), _i, _p, _p, _p, _i64, _i]),
    "pope_write_png": (_i, [C.c_char_p, _p, _i, _i, _i, _i64, _i]),
    "pope_write_png_batch": (_i, [C.POINTER(C.c_char_p), C.POINTER(_p), _p, _p, _i, _i, _i, _i]),
    "pope_pack_records": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _p, _p, _p]),
    "pope_pack_records_compact": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i, _p, _p, _p]),
    "pope_match_scores": (_i, [_p, _p, _i, _i, _f, _p, _p, _p]),
    "pope_pose_workspace_bytes": (_sz, [_i, _i64]),
    "pope_estimate_pose_batch": (_i, [_p, _p, _p, _i, _i64, _p, _p, C.c_double, C.c_double, _i, C.c_uint64, _p, _p, _p, _p,
                                      _p, _p, _p, _p, _sz, _p]),
    "pope_running_topk": (_i, [_p, _i, _i, _p, _p, _p]),
    "pope_cosine_topk": (_i, [_p, _p, _i, _i, _i, _i, _f, _p, _p, _p, _p]),
    "pope_pipeline_create": (_i, [C.POINTER(_p), _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _f, _i, _i]),
    "pope_pipeline_run": (_i, [_p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p]),
    "pope_pipeline_destroy": (_i, [_p]),
    "pope_pipeline_last_h2d_bytes": (_i64, [_p]),
    "pope_pipeline_last_f1_mode": (_i, [_p]),
    "pope_pipeline_set_fine_level": (_i, [_p, _p, _p, _i, C.POINTER(_i)]),
    "pope_match_pairs_host": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _f, _i, _i,
                                   _i, _i, _p, _p, _p, _p, _p, _p, _p]),
}

# kernels launched by one hot-path step (bench.py `gpu_launches`).  tcgen05 (thr > 0.15): single sweep, column-sum
# reduction, gated two-sweep launch (a no-op unless the fallback flag is raised), list evaluation, count+emit, fused fine
# match.  SIMT: row sweep, candidate bounds, column sweep, candidate evaluation, count+emit, fused fine match.
# fp32 on tcgen05: 2 split launches, sweep, column-sum reduction, list evaluation, 5 gated fp32-FMA fallback launches (no-ops
# unless the fallback flag is raised), count+emit, fused fine match.
KERNELS_PER_STEP = {"tcgen05": 6, "tcgen05_f32": 12, "simt": 6}


def single_sweep_is_split(n_pairs: int, L: int, sms: int = 148) -> bool:
    """Does the bf16 single sweep run as two launches (head + tail, csrc/coarse_tc.cu::coarse_tc_run)?  One more kernel per step
    then: the head's pairs fill whole rounds of the static unit schedule, the tail's fit the last, part-empty round, and the
    column merge of the head runs beside the tail."""
    cta_pairs, upp = sms // 2, -(-L // 256)
    units = n_pairs * upp
    if n_pairs <= 1 or units <= cta_pairs or units % cta_pairs == 0:
        return False
    head = ((units // cta_pairs) * cta_pairs) // upp
    ua, ub = head * upp, units - head * upp
    rounds = lambda u: -(-u // cta_pairs)
    return 0 < head < n_pairs and rounds(ua) + rounds(ub) == rounds(units) and 2 * ub <= cta_pairs + cta_pairs // 2

_lib: Optional[C.CDLL] = None


class PopeError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Loads the CUDA library once.  Raises if it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PopeError(f"{LIB_PATH} not found: build it with `make -C pope_b200/csrc` "
                            "(there is no CPU or PyTorch fallback for the Matcher hot path)")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)        # AttributeError if the symbol is missing
            fn.restype, fn.argtypes = res, args
        if h.pope_abi_version() != 1:
            raise PopeError("libpope_b200.so ABI version mismatch")
        _lib = h
    return _lib


def tcgen05_available(L: int = 4800, S: int = 4800, C_: int = 256) -> bool:
    """True when POPE_COARSE_AUTO resolves to the tcgen05 kernels for bf16 features of this shape."""
    return lib().pope_coarse_auto_impl(POPE_BF16, L, S, C_) == COARSE_TCGEN05


def check(status: int, what: str) -> None:
    if status != 0:
        raise PopeError(f"{what} failed: status {status} ({lib().pope_status_string(status).decode()})")


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return POPE_F32
    if t.dtype == torch.bfloat16:
        return POPE_BF16
    raise PopeError(f"unsupported feature dtype {t.dtype}: the CUDA path takes float32 or bfloat16")


def require_cuda(*tensors: torch.Tensor) -> torch.device:
    dev = tensors[0].device
    for t in tensors:
        if not t.is_cuda:
            raise PopeError("pope_b200 runs on a CUDA device only (no CPU fallback); got a tensor on " + str(t.device))
        if t.device != dev:
            raise PopeError("all tensors of one call must live on the same device")
    return dev


def stream_ptr(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()
