"""TEST INFRASTRUCTURE ONLY -- tests/golden/fine_transformer.npz and fine_merge_coarse.npz from the UNMODIFIED reference.

    POPE_REFERENCE_ROOT=<reference checkout> python oracle/gen_golden_fine_tf.py

Runs the reference's own `LocalFeatureTransformer(config['fine'])` (src/matcher/loftr_module/transformer.py:61-106,
d_model 128, 8 heads, layers ['self', 'cross'], linear attention) and `FinePreprocess` (fine_preprocess.py:8-59) with
seeded weights whose matrices are rounded to bf16 (so that the bf16 CUDA path and the fp32 reference use the same
weights) on seeded bf16-rounded inputs.  Stored: the weights (bf16 bit patterns / fp32), the seeds of the inputs and the
reference's fp32 outputs.
"""
from __future__ import annotations

import contextlib
import copy
import io
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
M_WINDOWS, KEPT = 37, 12          # 37 * 25 = 925 token rows: 7 full 128-row tiles + a ragged one


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).float()


def bf16_bits(t: torch.Tensor) -> np.ndarray:
    return t.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def inputs(seed: int, m: int = M_WINDOWS):
    g = torch.Generator().manual_seed(seed)
    return bf16_round(torch.randn(m, 25, 128, generator=g)), bf16_round(torch.randn(m, 25, 128, generator=g))


def main():
    ref = ref_shim.import_reference()
    from src.matcher.loftr_module.fine_preprocess import FinePreprocess
    from src.matcher.loftr_module.transformer import LocalFeatureTransformer
    cfg = copy.deepcopy(ref.default_cfg)
    torch.manual_seed(7)
    with contextlib.redirect_stdout(io.StringIO()):
        tf = LocalFeatureTransformer(copy.deepcopy(cfg["fine"])).eval()
    g = torch.Generator().manual_seed(8)
    with torch.no_grad():
        for name, p in tf.named_parameters():
            if p.dim() > 1:
                p.copy_(bf16_round(p))
            elif name.endswith("weight"):          # LayerNorm scale / shift away from the (1, 0) default
                p.copy_(1.0 + 0.2 * torch.randn(p.shape, generator=g))
            else:
                p.copy_(0.1 * torch.randn(p.shape, generator=g))
    f0, f1 = inputs(9)
    with torch.no_grad():
        o0, o1 = tf(f0.clone(), f1.clone())
    out = {"meta": json.dumps(dict(input_seed=9, m=M_WINDOWS, kept=KEPT, layer_names=list(tf.layer_names))),
           "out0": o0[:KEPT].numpy(), "out1": o1[:KEPT].numpy(),
           "out0_sum": o0.sum((1, 2)).numpy(), "out1_sum": o1.sum((1, 2)).numpy()}
    for k, v in tf.state_dict().items():
        out["tf." + k] = bf16_bits(v) if v.dim() > 1 else v.numpy()

    # FinePreprocess Linears on the same windows + seeded coarse features
    torch.manual_seed(10)
    fp = FinePreprocess(copy.deepcopy(cfg)).eval()
    with torch.no_grad():
        for name, p in fp.named_parameters():
            p.copy_(bf16_round(p) if p.dim() > 1 else 0.1 * torch.randn(p.shape, generator=g))
    n, L, S = 2, 48, 40
    fc0, fc1 = bf16_round(torch.randn(n, L, 256, generator=g)), bf16_round(torch.randn(n, S, 256, generator=g))
    b_ids = torch.randint(0, n, (M_WINDOWS,), generator=g).sort().values
    i_ids = torch.randint(0, L, (M_WINDOWS,), generator=g)
    j_ids = torch.randint(0, S, (M_WINDOWS,), generator=g)
    both = torch.cat([f0, f1], 0)
    with torch.no_grad():                           # fine_preprocess.py:50-57 with the reference's own modules
        c_win = fp.down_proj(torch.cat([fc0[b_ids, i_ids], fc1[b_ids, j_ids]], 0))
        merged = fp.merge_feat(torch.cat([both, c_win[:, None, :].expand(-1, 25, -1)], -1))
    pre = {"pre.meta": json.dumps(dict(n=n, L=L, S=S)), "pre.feat_c0": bf16_bits(fc0), "pre.feat_c1": bf16_bits(fc1),
           "pre.b_ids": b_ids.numpy(), "pre.i_ids": i_ids.numpy(), "pre.j_ids": j_ids.numpy(),
           "pre.merged0": merged[:KEPT].numpy(), "pre.merged1": merged[M_WINDOWS:M_WINDOWS + KEPT].numpy(),
           "pre.merged_sum": merged.sum((1, 2)).numpy()}
    for k, v in fp.state_dict().items():
        pre["pre." + k] = bf16_bits(v) if v.dim() > 1 else v.numpy()
    # two files, each below 1 MB; the Linears' fixture shares the inputs (`meta`) of the transformer's
    for name, arrays in (("fine_transformer.npz", out), ("fine_merge_coarse.npz", pre)):
        np.savez_compressed(os.path.join(GOLDEN, name), **arrays)
        print(name + ":", {k: getattr(v, "shape", None) for k, v in arrays.items() if not k.endswith("meta")})


if __name__ == "__main__":
    main()
