"""The bf16 fine level (FinePreprocess Linears + fine transformer) inside the sync-free device step, bounded by the match
count kept on the device: `pope_fine_transformer_ex` / `pope_fine_merge_coarse_ex`, `ops.match_pairs_device(fine_level=)`,
`Matcher.fine_level`, `DeviceBatchRunner.submit(fine_level=)`.

The bounded launches run the same kernels with the same per-row arithmetic as the unbounded ones (every Linear row, every
attention window and every LayerNorm row is computed from its own inputs only), so live rows are compared bit for bit,
and rows at or past the live count must keep what they held before."""
import pytest
import torch

import pope_b200
from pope_b200 import _lib, ops, synth

CAP = 2048
LIVE = (0, 1, 5, 1003, 2048)


def _random_layer(gen):
    sd = {}
    for key, shp in (("q_proj.weight", (128, 128)), ("k_proj.weight", (128, 128)), ("v_proj.weight", (128, 128)),
                     ("merge.weight", (128, 128)), ("mlp.0.weight", (256, 256)), ("mlp.2.weight", (128, 256))):
        bound = (6.0 / (shp[0] + shp[1])) ** 0.5
        sd[key] = (torch.rand(shp, generator=gen) * 2 - 1) * bound
    for key in ("norm1", "norm2"):
        sd[key + ".weight"] = 1 + 0.2 * torch.randn(128, generator=gen)
        sd[key + ".bias"] = 0.1 * torch.randn(128, generator=gen)
    return sd


def _random_pre(gen):
    return {"down_proj.weight": torch.randn(128, 256, generator=gen) * 0.06, "down_proj.bias": 0.1 * torch.randn(128, generator=gen),
            "merge_feat.weight": torch.randn(128, 256, generator=gen) * 0.06, "merge_feat.bias": 0.1 * torch.randn(128, generator=gen)}


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _sentinel_windows(gen, dev, live):
    """[CAP, 25, 128] bf16 windows: random rows below `live`, NaN from there on (a NaN that reached a live row through a
    shared tile would show in the comparison)."""
    w = torch.randn(CAP, 25, 128, generator=gen).to(torch.bfloat16)
    w[live:] = float("nan")
    return w.to(dev)


# ---- CPU: argument checking and the weight bundle ------------------------------------------------------------------

def test_ex_entry_points_reject_bad_arguments_before_touching_the_gpu():
    h = _lib.lib()
    kinds = (_lib.C.c_int * 2)(0, 1)
    ws = h.pope_fine_tf_workspace_bytes(8, 25)
    # feat0, feat1, m_windows, m_dev, window_tokens, weights, n_layers, layer_kinds, workspace, workspace_bytes, stream
    ok = [16, 16, 8, None, 25, 16, 2, kinds, 16, ws, None]
    for i in (0, 1, 5, 8):                                         # null feature, weight and workspace pointers
        bad = list(ok); bad[i] = None
        assert h.pope_fine_transformer_ex(*bad) == -1, i
    bad = list(ok); bad[2] = -1                                    # negative capacity
    assert h.pope_fine_transformer_ex(*bad) == -1
    bad = list(ok); bad[4] = 0                                     # no tokens per window
    assert h.pope_fine_transformer_ex(*bad) == -1
    bad = list(ok); bad[7] = (_lib.C.c_int * 2)(0, 2)              # layer kind other than 'self' / 'cross'
    assert h.pope_fine_transformer_ex(*bad) == -1
    bad = list(ok); bad[9] = ws - 1                                # workspace too small
    assert h.pope_fine_transformer_ex(*bad) == -3
    bad = list(ok); bad[0] = 24                                    # misaligned windows
    assert h.pope_fine_transformer_ex(*bad) == -5
    bad = list(ok); bad[2] = 0                                     # capacity 0 is a no-op
    assert h.pope_fine_transformer_ex(*bad) == 0

    mw = h.pope_fine_merge_workspace_bytes(8)
    # win0, win1, m_windows, m_dev, window_tokens, feat_c0, feat_c1, L, S, C, b_ids, i_ids, j_ids, weights, workspace, bytes, stream
    ok = [16, 16, 8, None, 25, 16, 16, 64, 64, 256, 16, 16, 16, 16, 16, mw, None]
    for i in (0, 1, 5, 6, 10, 11, 12, 13, 14):
        bad = list(ok); bad[i] = None
        assert h.pope_fine_merge_coarse_ex(*bad) == -1, i
    bad = list(ok); bad[2] = -5
    assert h.pope_fine_merge_coarse_ex(*bad) == -1
    bad = list(ok); bad[9] = 128                                   # coarse width other than 256
    assert h.pope_fine_merge_coarse_ex(*bad) == -4
    bad = list(ok); bad[15] = mw - 1
    assert h.pope_fine_merge_coarse_ex(*bad) == -3
    bad = list(ok); bad[2] = 0
    assert h.pope_fine_merge_coarse_ex(*bad) == 0


@pytest.mark.parametrize("m,S", [(1, 25), (3, 25), (8, 25), (1003, 25), (307200, 25), (5, 49), (77, 9)])
def test_fine_tf_workspace_is_five_planes(m, S):
    """The transformer's scratch is q, k, v, message and merged message: five 256-byte-aligned [m * S, 128] bf16 planes.
    At S = 25 it also covers the merge's scratch, so the fine level's shared scratch is the transformer's size."""
    h = _lib.lib()
    plane = (m * S * 128 * 2 + 255) // 256 * 256
    assert h.pope_fine_tf_workspace_bytes(m, S) == 5 * plane
    if S == 25:
        assert h.pope_fine_tf_workspace_bytes(m, S) >= h.pope_fine_merge_workspace_bytes(m)
    assert h.pope_fine_tf_workspace_bytes(0, S) == 0 and h.pope_fine_tf_workspace_bytes(m, 0) == 0


def test_fine_level_workspace_is_sized_for_the_stages_that_use_it():
    """The Matcher flow hands the merge no scratch: it must get the merge's bytes, not the transformer's five planes.
    A scratch that is large enough is reused, one that is too small is replaced."""
    h, cpu = _lib.lib(), torch.device("cpu")
    m = 1003
    tf, mg = h.pope_fine_tf_workspace_bytes(m, 25), h.pope_fine_merge_workspace_bytes(m)
    assert mg < tf
    assert ops.fine_level_workspace(m, 25, cpu, transformer=False).numel() == mg
    assert ops.fine_level_workspace(m, 25, cpu, merge=False).numel() == tf
    shared = ops.fine_level_workspace(m, 25, cpu)
    assert shared.numel() == tf
    assert ops.fine_level_workspace(m, 25, cpu, shared, transformer=False) is shared
    assert ops.fine_level_workspace(m, 25, cpu, shared[:mg - 1], transformer=False).numel() == mg


def test_fine_level_packs_the_matcher_weights_and_rejects_what_it_cannot_run():
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    fl = m.fine_level("cpu")
    assert fl["layer_names"] == m.loftr_fine.layer_names
    assert fl["layers"].numel() == len(fl["layer_names"]) * _lib.FINE_TF_LAYER_BYTES
    assert fl["pre"].numel() == _lib.FINE_PRE_BYTES
    assert fl["layers"] is m.fine_level("cpu")["layers"]          # the module's cache, not a new packing
    cfg = pope_b200.make_default_cfg()
    cfg["fine_concat_coarse_feat"] = False
    assert pope_b200.Matcher(cfg).fine_level("cpu")["pre"] is None
    cfg = pope_b200.make_default_cfg()
    cfg["fine"]["attention"] = "full"
    with pytest.raises(NotImplementedError):
        pope_b200.Matcher(cfg).fine_level("cpu")


def test_fine_level_step_rejects_cpu_tensors():
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    f0, f1 = synth.coarse_features(5, 1, 64, 64, 256, dtype=torch.bfloat16)
    ff0, ff1 = synth.fine_feature_maps(6, 1, 32, 32, 128, dtype=torch.bfloat16)
    with pytest.raises(_lib.PopeError):
        ops.match_pairs_device(f0, f1, ff0, ff1, (64, 64), (8, 8), (8, 8), fine_level=m.fine_level("cpu"))
    with pytest.raises(_lib.PopeError):
        ops.fine_transformer(torch.zeros(2, 25, 128, dtype=torch.bfloat16), torch.zeros(2, 25, 128, dtype=torch.bfloat16),
                             m.fine_level("cpu")["layers"], m.loftr_fine.layer_names, m_dev=torch.ones(1, dtype=torch.int32))


# ---- GPU -----------------------------------------------------------------------------------------------------------

DEV = torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("names", [["self"], ["cross"]])
@pytest.mark.parametrize("live", LIVE)
def test_bounded_transformer_equals_unbounded_on_the_live_windows(names, live):
    gen = torch.Generator().manual_seed(7 + live)
    packed = torch.cat([ops.pack_fine_layer(_random_layer(gen), DEV) for _ in names])
    w0, w1 = _sentinel_windows(gen, DEV, live), _sentinel_windows(gen, DEV, live)
    before0, before1 = w0.clone(), w1.clone()
    want0, want1 = w0[:live].clone(), w1[:live].clone()
    ops.fine_transformer(want0, want1, packed, names)
    m_dev = torch.tensor([live], dtype=torch.int32, device=DEV)
    ops.fine_transformer(w0, w1, packed, names, m_dev=m_dev)
    torch.cuda.synchronize()
    for got, want, before in ((w0, want0, before0), (w1, want1, before1)):
        assert torch.equal(_bits(got[:live]), _bits(want)), live
        assert torch.equal(_bits(got[live:]), _bits(before[live:])), live
        assert torch.isfinite(got[:live].float()).all()


@pytest.mark.gpu
@pytest.mark.parametrize("live", LIVE)
def test_bounded_merge_equals_unbounded_on_both_sides(live):
    gen = torch.Generator().manual_seed(31 + live)
    n, L, S = 3, 300, 280
    fc0 = torch.randn(n, L, 256, generator=gen).to(DEV, torch.bfloat16)
    fc1 = torch.randn(n, S, 256, generator=gen).to(DEV, torch.bfloat16)
    b = torch.randint(0, n, (CAP,), generator=gen).to(DEV)
    i = torch.randint(0, L, (CAP,), generator=gen).to(DEV)
    j = torch.randint(0, S, (CAP,), generator=gen).to(DEV)
    pre = ops.pack_fine_pre(_random_pre(gen), DEV)
    w0, w1 = _sentinel_windows(gen, DEV, live), _sentinel_windows(gen, DEV, live)
    before0, before1 = w0.clone(), w1.clone()
    want0, want1 = w0[:live].clone(), w1[:live].clone()
    ops.fine_merge_coarse(want0, want1, fc0, fc1, b[:live], i[:live], j[:live], pre)
    ops.fine_merge_coarse(w0, w1, fc0, fc1, b, i, j, pre, m_dev=torch.tensor([live], dtype=torch.int32, device=DEV))
    torch.cuda.synchronize()
    for side, (got, want, before) in enumerate(((w0, want0, before0), (w1, want1, before1))):
        assert torch.equal(_bits(got[:live]), _bits(want)), (live, side)
        assert torch.equal(_bits(got[live:]), _bits(before[live:])), (live, side)


def _shapes(h, w, n):
    return {"hw0_i": torch.Size([h * 8, w * 8]), "hw1_i": torch.Size([h * 8, w * 8]), "hw0_c": torch.Size([h, w]),
            "hw1_c": torch.Size([h, w]), "hw0_f": torch.Size([h * 4, w * 4]), "hw1_f": torch.Size([h * 4, w * 4]), "bs": n}


def _matcher(seed=0):
    torch.manual_seed(seed)
    return pope_b200.Matcher(pope_b200.make_default_cfg(), fine_cuda_bf16=True).eval().to(DEV)


def _inputs(seed, n, h, w, channels_last=True):
    f0, f1 = synth.coarse_features(seed, n, h * w, h * w, 256, sigma=0.9, dtype=torch.bfloat16)
    ff0, ff1 = synth.fine_feature_maps(seed + 1, n, h * 4, w * 4, 128, dtype=torch.bfloat16, channels_last=channels_last)
    return [t.to(DEV) for t in (f0, f1, ff0, ff1)]


KEYS = ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f", "expec_f")


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w", [(2, 20, 24), (8, 60, 80)])
def test_step_with_fine_level_equals_the_matcher(n, h, w):
    m = _matcher()
    f0, f1, ff0, ff1 = _inputs(40 + n, n, h, w, channels_last=False)
    data = _shapes(h, w, n)
    with torch.no_grad():
        m.coarse_matching(f0, f1, data)
        w0, w1 = m.fine_preprocess(ff0, ff1, f0, f1, data)
        w0, w1 = m.loftr_fine(w0, w1)
        m.fine_matching(w0, w1, data)
    res = ops.match_pairs_device(f0, f1, ff0, ff1, data["hw0_i"], (h, w), (h, w), fine_level=m.fine_level(DEV))
    k = res.total()
    assert k == data["b_ids"].numel() and k > 100 and res.flags() == 0
    for key in ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f"):
        assert torch.equal(res[key][:k], data[key]), key
    for key in ("expec_f", "mkpts1_f"):
        assert torch.equal(_bits(res[key][:k]), _bits(data[key])), key
    # the fine level really ran: without it the refinement differs
    plain = ops.match_pairs_device(f0, f1, ff0, ff1, data["hw0_i"], (h, w), (h, w), fused_fine=False)
    assert not torch.equal(plain["mkpts1_f"][:k], res["mkpts1_f"][:k])


@pytest.mark.gpu
def test_step_with_fine_level_is_graph_capturable():
    """Same shape as tests/test_gpu_parity.py::test_hot_path_step_is_graph_capturable: with the fine level the step still
    has no host sync, so it is captured into a CUDA graph; replays on new feature contents equal eager calls bit for bit."""
    n, h, w = 24, 40, 48
    m = _matcher(1)
    fl = m.fine_level(DEV)
    sets = [_inputs(seed, n, h, w) for seed in (301, 302)]
    hw_i = (h * 8, w * 8)
    want = []
    for s in sets:
        r = ops.match_pairs_device(*s, hw_i, (h, w), (h, w), fine_level=fl)
        k = r.total()
        assert k > 5000 and r.flags() == 0
        want.append((k, {key: r[key][:k].clone() for key in KEYS}))
    static = [t.clone() for t in sets[0]]
    ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, h * w, h * w, 256, 1), dtype=torch.uint8, device=DEV)
    fws = ops.fine_level_workspace(n * h * w, 25, DEV)
    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):                      # warm-up on the capture stream (first-use attribute calls)
        ops.match_pairs_device(*static, hw_i, (h, w), (h, w), workspace=ws, fine_level=fl, fine_workspace=fws)
    torch.cuda.current_stream(DEV).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        res = ops.match_pairs_device(*static, hw_i, (h, w), (h, w), workspace=ws, fine_level=fl, fine_workspace=fws)
    assert res["fine_workspace"] is fws
    for which in (1, 0, 1):
        for dst, src in zip(static, sets[which]):
            dst.copy_(src)
        graph.replay()
        torch.cuda.synchronize()
        k, ref = want[which]
        assert res.total() == k and res.flags() == 0
        for key in KEYS:
            assert torch.equal(_bits(res[key][:k]), _bits(ref[key])), (which, key)


@pytest.mark.gpu
def test_batch_runner_with_fine_level_equals_sequential_steps_and_job_gather_stays_exact():
    from pope_b200 import driver
    n, h, w = 2, 20, 24
    m = _matcher(2)
    fl = m.fine_level(DEV)
    batches = [_inputs(seed, n, h, w) for seed in (91, 93, 95, 97)]
    runner = driver.DeviceBatchRunner(DEV, 2)
    job = driver.JobGather(len(batches), n * h * w, DEV)
    runner.fork()
    got = [runner.submit(*b, (h * 8, w * 8), (h, w), (h, w), after=lambda r, k=k: job.add(r, 10 * k), fine_level=fl)[0]
           for k, b in enumerate(batches)]
    assert all(ws is not None for ws in runner.fine_workspaces)
    runner.join()
    recs, sizes = job.finish()
    torch.cuda.synchronize()
    rec = driver.unpack_records(recs[0].cpu())
    off = 0
    for k, (b, res) in enumerate(zip(batches, got)):
        want = ops.match_pairs_device(*b, (h * 8, w * 8), (h, w), (h, w), fine_level=fl)
        c = want.total()
        assert res.total() == c and c > 100
        for key in KEYS:
            assert torch.equal(_bits(res[key][:c]), _bits(want[key][:c])), (k, key)
        assert torch.equal(rec["b_ids"][off:off + c], want["b_ids"][:c].cpu() + 10 * k)
        for key in ("i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f"):
            assert torch.equal(rec[key][off:off + c], want[key][:c].cpu()), (k, key)
        off += c
    assert sizes == [off]


@pytest.mark.gpu
def test_step_with_fine_level_and_zero_matches():
    n, h, w = 2, 20, 24
    m = _matcher(3)
    fl = m.fine_level(DEV)
    f0, f1, ff0, ff1 = _inputs(70, n, h, w)
    f1 = torch.zeros_like(f1)             # every similarity 0: uniform softmaxes, confidence 1 / (L S), no match
    res = ops.match_pairs_device(f0, f1, ff0, ff1, (h * 8, w * 8), (h, w), (h, w), fine_level=fl)
    assert res.total() == 0 and res.flags() == 0
    # the step's own count (0) bounds every fine-level launch: windows given to them keep every byte
    m_dev = res["counts"][n:n + 1]
    gen = torch.Generator().manual_seed(71)
    cap = res["b_ids"].shape[0]
    w0 = torch.randn(cap, 25, 128, generator=gen).to(DEV, torch.bfloat16)
    w1 = torch.randn(cap, 25, 128, generator=gen).to(DEV, torch.bfloat16)
    before0, before1 = w0.clone(), w1.clone()
    ops.fine_merge_coarse(w0, w1, f0, f1, res["b_ids"], res["i_ids"], res["j_ids"], fl["pre"], m_dev=m_dev)
    ops.fine_transformer(w0, w1, fl["layers"], fl["layer_names"], m_dev=m_dev)
    torch.cuda.synchronize()
    assert torch.equal(_bits(w0), _bits(before0)) and torch.equal(_bits(w1), _bits(before1))


@pytest.mark.gpu
def test_step_with_fine_level_rejects_what_it_cannot_run():
    n, h, w = 1, 20, 24
    m = _matcher(4)
    fl = m.fine_level(DEV)
    f0, f1, ff0, ff1 = _inputs(80, n, h, w)
    args = ((h * 8, w * 8), (h, w), (h, w))
    with pytest.raises(_lib.PopeError):                                        # fp32 coarse features
        ops.match_pairs_device(f0.float(), f1.float(), ff0, ff1, *args, fine_level=fl)
    with pytest.raises(_lib.PopeError):                                        # fp32 fine maps
        ops.match_pairs_device(f0, f1, ff0.float(), ff1.float(), *args, fine_level=fl)
    with pytest.raises(_lib.PopeError):                                        # CPU tensors
        ops.match_pairs_device(f0.cpu(), f1.cpu(), ff0.cpu(), ff1.cpu(), *args, fine_level=fl)
    with pytest.raises(_lib.PopeError):                                        # the fused route has no fine level
        ops.match_pairs_device(f0, f1, ff0, ff1, *args, fine_level=fl, fused_fine=True)
