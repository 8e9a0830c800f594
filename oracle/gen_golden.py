"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/*.npz by running the UNMODIFIED reference.

Run in the build container (where /root/reference is mounted):

    python oracle/gen_golden.py

It imports the reference's own `CoarseMatching`, `FinePreprocess`, `FineMatching` and `Matcher`
(src/matcher/..., via oracle/ref_shim.py), feeds them the seeded synthetic inputs of
`pope_b200/synth.py` and stores inputs' seeds + the reference's outputs.  The fixtures pin the oracle
(tests/test_oracle_golden.py) and, on the GPU box where /root/reference does not exist, the CUDA path
(tests/test_gpu_parity.py).  Inputs are regenerated from the seed at test time; only outputs are stored.
"""
from __future__ import annotations

import copy
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402
from pope_b200 import synth  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# name -> generator kwargs.  hw*_c are coarse grids (cells), image size = 8 * grid.
COARSE_CASES = {
    "coarse_small":     dict(seed=11, n=2, hw0_c=(12, 16), hw1_c=(12, 16), C=256, kind="plain", sigma=0.8),
    "coarse_ragged":    dict(seed=12, n=3, hw0_c=(10, 14), hw1_c=(8, 9),   C=64,  kind="plain", sigma=0.8),
    "coarse_hard":      dict(seed=13, n=2, hw0_c=(20, 24), hw1_c=(18, 28), C=64,  kind="hard",  sigma=0.9),
    "coarse_bf16":      dict(seed=14, n=2, hw0_c=(12, 16), hw1_c=(12, 16), C=256, kind="bf16",  sigma=0.8),
    "coarse_nomatch":   dict(seed=15, n=1, hw0_c=(6, 8),   hw1_c=(6, 8),   C=64,  kind="noise", sigma=0.05),
    "coarse_mid":       dict(seed=16, n=2, hw0_c=(30, 40), hw1_c=(32, 32), C=256, kind="plain", sigma=0.9),
    # BASELINE.json configs[0]: one 480x640 pair, 60x80 coarse tokens, d=256 (fp32 and bf16-rounded inputs)
    "coarse_full":      dict(seed=17, n=1, hw0_c=(60, 80), hw1_c=(60, 80), C=256, kind="plain", sigma=1.0),
    "coarse_full_bf16": dict(seed=18, n=1, hw0_c=(60, 80), hw1_c=(60, 80), C=256, kind="bf16",  sigma=1.0),
}


def coarse_inputs(case):
    L = case["hw0_c"][0] * case["hw0_c"][1]
    S = case["hw1_c"][0] * case["hw1_c"][1]
    sg = case["sigma"]
    if case["kind"] == "hard":
        return synth.hard_coarse_features(case["seed"], case["n"], L, S, case["C"], sigma=sg)
    if case["kind"] == "bf16":
        f0, f1 = synth.coarse_features(case["seed"], case["n"], L, S, case["C"], sigma=sg, dtype=torch.bfloat16)
        return f0.float(), f1.float()
    if case["kind"] == "noise":   # no planted correspondences, tiny norm -> conf << thr -> M = 0
        return synth.coarse_features(case["seed"], case["n"], L, S, case["C"], sigma=sg, planted=0.0)
    return synth.coarse_features(case["seed"], case["n"], L, S, case["C"], sigma=sg)


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    ref = ref_shim.import_reference()
    from src.matcher.utils.coarse_matching import CoarseMatching
    from src.matcher.utils.fine_matching import FineMatching
    from src.matcher.loftr_module.fine_preprocess import FinePreprocess

    cfg = copy.deepcopy(ref.default_cfg)
    torch.set_grad_enabled(False)

    # ---- coarse matching -------------------------------------------------------------------------
    cm = CoarseMatching(cfg["match_coarse"]).eval()
    for name, case in COARSE_CASES.items():
        f0, f1 = coarse_inputs(case)
        hw0_c, hw1_c = case["hw0_c"], case["hw1_c"]
        data = {"hw0_i": torch.Size([hw0_c[0] * 8, hw0_c[1] * 8]), "hw1_i": torch.Size([hw1_c[0] * 8, hw1_c[1] * 8]),
                "hw0_c": torch.Size(hw0_c), "hw1_c": torch.Size(hw1_c)}
        cm(f0, f1, data)
        conf = data["conf_matrix"]
        # margins used by the parity tests to classify near-ties / near-threshold cells
        top2_row = conf.topk(2, dim=2)[0]
        top2_col = conf.topk(2, dim=1)[0]
        np.savez_compressed(
            os.path.join(GOLDEN, name + ".npz"),
            meta=json.dumps(case),
            b_ids=data["b_ids"].numpy(), i_ids=data["i_ids"].numpy(), j_ids=data["j_ids"].numpy(),
            mconf=data["mconf"].numpy(), mkpts0_c=data["mkpts0_c"].numpy(), mkpts1_c=data["mkpts1_c"].numpy(),
            gt_mask=data["gt_mask"].numpy(), m_bids=data["m_bids"].numpy(),
            conf_rowmax=top2_row[..., 0].numpy(), conf_row2nd=top2_row[..., 1].numpy(),
            conf_colmax=top2_col[:, 0].numpy(), conf_col2nd=top2_col[:, 1].numpy(),
        )
        print(f"{name}: M={data['b_ids'].numel()} mconf[min,max]="
              f"{(data['mconf'].min().item() if data['mconf'].numel() else 0):.3f},"
              f"{(data['mconf'].max().item() if data['mconf'].numel() else 0):.3f}")

    # ---- fine preprocess (window unfold + gather, without the coarse-feature Linears: gen_golden_fine_tf.py has those) ----
    case = COARSE_CASES["coarse_small"]
    f0, f1 = coarse_inputs(case)
    g = np.load(os.path.join(GOLDEN, "coarse_small.npz"))
    b_ids, i_ids, j_ids = (torch.from_numpy(g[k]) for k in ("b_ids", "i_ids", "j_ids"))
    hw_c = case["hw0_c"]
    ff0, ff1 = synth.fine_feature_maps(21, case["n"], hw_c[0] * 4, hw_c[1] * 4, 128, channels_last=False)
    data = {"hw0_f": ff0.shape[2:], "hw0_c": torch.Size(hw_c), "b_ids": b_ids, "i_ids": i_ids, "j_ids": j_ids}
    cfg_nocat = copy.deepcopy(cfg)
    cfg_nocat["fine_concat_coarse_feat"] = False
    w0, w1 = FinePreprocess(cfg_nocat).eval()(ff0, ff1, f0, f1, dict(data))
    keep = slice(0, 40)          # 40 of the 64 windows in full (the fixture stays below 1 MB), the sums of all of them
    np.savez_compressed(
        os.path.join(GOLDEN, "fine_preprocess.npz"),
        meta=json.dumps(dict(coarse_case="coarse_small", fine_seed=21, kept=40)),
        win0=w0[keep].numpy(), win1=w1[keep].numpy(), win0_sum=w0.sum((1, 2)).numpy(), win1_sum=w1.sum((1, 2)).numpy(),
    )
    print(f"fine_preprocess: M={w0.shape[0]}")

    # ---- fine matching ---------------------------------------------------------------------------
    fm = FineMatching().eval()
    for name, (seed, M, gain) in {"fine_match_soft": (31, 96, 1.0), "fine_match_peaked": (32, 96, 3.0)}.items():
        a, b = synth.fine_windows(seed, M, 25, 128, gain=gain)
        gg = torch.Generator().manual_seed(seed + 1)
        mk0 = (torch.randint(0, 80, (M, 2), generator=gg) * 8).float()
        mk1 = (torch.randint(0, 80, (M, 2), generator=gg) * 8).float()
        data = {"hw0_i": torch.Size([480, 640]), "hw0_f": torch.Size([240, 320]),
                "mkpts0_c": mk0, "mkpts1_c": mk1, "mconf": torch.ones(M)}
        fm(a, b, data)
        np.savez_compressed(os.path.join(GOLDEN, name + ".npz"),
                            meta=json.dumps(dict(seed=seed, M=M, gain=gain)),
                            mkpts0_c=mk0.numpy(), mkpts1_c=mk1.numpy(),
                            expec_f=data["expec_f"].numpy(), mkpts0_f=data["mkpts0_f"].numpy(),
                            mkpts1_f=data["mkpts1_f"].numpy())
        print(f"{name}: expec range {data['expec_f'][:, :2].min().item():.3f}..{data['expec_f'][:, :2].max().item():.3f}")
    # M == 0 branch (fine_matching.py:33-41)
    data = {"hw0_i": torch.Size([480, 640]), "hw0_f": torch.Size([240, 320]),
            "mkpts0_c": torch.empty(0, 2), "mkpts1_c": torch.empty(0, 2), "mconf": torch.empty(0)}
    fm(torch.empty(0, 25, 128), torch.empty(0, 25, 128), data)
    assert data["expec_f"].shape == (0, 3) and data["mkpts1_f"].shape == (0, 2)

    # ---- whole-Matcher structure: state-dict layout and output-dict key order -------------------------
    torch.manual_seed(0)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        m = ref.Matcher(copy.deepcopy(ref.default_cfg)).eval()
    sd = m.state_dict()
    batch = {"image0": torch.rand(1, 1, 64, 96, generator=torch.Generator().manual_seed(1)),
             "image1": torch.rand(1, 1, 64, 64, generator=torch.Generator().manual_seed(2))}
    m(batch)
    layout = {
        "state_dict": {k: list(v.shape) for k, v in sd.items()},
        "n_params": int(sum(p.numel() for p in m.parameters())),
        "data_keys": list(batch.keys()),
        "data_types": {k: (str(v.dtype) + str(list(v.shape)) if torch.is_tensor(v) else type(v).__name__)
                       for k, v in batch.items()},
        "default_cfg": json.loads(json.dumps(ref.default_cfg)),
    }
    with open(os.path.join(GOLDEN, "matcher_layout.json"), "w") as f:
        json.dump(layout, f, indent=1, sort_keys=False)
    print(f"matcher_layout: {len(sd)} state-dict entries, {layout['n_params']} params, keys {layout['data_keys']}")


if __name__ == "__main__":
    main()
