"""The fp32-accuracy fine level (FinePreprocess Linears + fine transformer) inside the sync-free device step, bounded by
the match count kept on the device: `pope_fine_transformer_f32_ex` / `pope_fine_merge_coarse_f32_ex`,
`ops.match_pairs_device(fine_level=<fp32 bundle>)`, `Matcher.fine_level(device, dtype=torch.float32)`,
`DeviceBatchRunner.submit(fine_level=)`.

The bounded launches run the same kernels with the same per-row arithmetic as the unbounded ones (every Linear row, every
attention window and every LayerNorm row is computed from its own inputs only), so live rows are compared bit for bit,
and rows at or past the live count must keep what they held before (NaN sentinels)."""
import pytest
import torch

import pope_b200
from pope_b200 import _lib, driver, ops, synth

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
    return t.contiguous().view(torch.int32)


def _sentinel_windows(gen, dev, live, ww=25):
    """[CAP, ww, 128] fp32 windows: random rows below `live`, NaN from there on (a NaN that reached a live row through a
    shared tile would show in the comparison)."""
    w = torch.randn(CAP, ww, 128, generator=gen)
    w[live:] = float("nan")
    return w.to(dev)


# ---- CPU: argument checking and the weight bundle ------------------------------------------------------------------

def test_f32_ex_entry_points_reject_bad_arguments_before_touching_the_gpu():
    h = _lib.lib()
    kinds = (_lib.C.c_int * 2)(0, 1)
    ws = h.pope_fine_tf_f32_workspace_bytes(8, 25)
    # feat0, feat1, m_windows, m_dev, window_tokens, weights, n_layers, layer_kinds, workspace, workspace_bytes, stream
    ok = [16, 16, 8, None, 25, 16, 2, kinds, 16, ws, None]
    for i in (0, 1, 5, 8):                                         # null feature, weight and workspace pointers
        bad = list(ok); bad[i] = None
        assert h.pope_fine_transformer_f32_ex(*bad) == -1, i
    bad = list(ok); bad[2] = -1                                    # negative capacity
    assert h.pope_fine_transformer_f32_ex(*bad) == -1
    bad = list(ok); bad[4] = 0                                     # no tokens per window
    assert h.pope_fine_transformer_f32_ex(*bad) == -1
    bad = list(ok); bad[7] = (_lib.C.c_int * 2)(0, 2)              # layer kind other than 'self' / 'cross'
    assert h.pope_fine_transformer_f32_ex(*bad) == -1
    bad = list(ok); bad[9] = ws - 1                                # workspace too small
    assert h.pope_fine_transformer_f32_ex(*bad) == -3
    bad = list(ok); bad[0] = 24                                    # misaligned windows
    assert h.pope_fine_transformer_f32_ex(*bad) == -5
    bad = list(ok); bad[2] = 1 << 27                               # more rows than the kernels index
    assert h.pope_fine_transformer_f32_ex(*bad) == -4
    bad = list(ok); bad[2] = 0                                     # capacity 0 is a no-op
    assert h.pope_fine_transformer_f32_ex(*bad) == 0

    mw = h.pope_fine_merge_f32_workspace_bytes(8)
    # win0, win1, m_windows, m_dev, window_tokens, feat_c0, feat_c1, L, S, C, b_ids, i_ids, j_ids, weights, workspace, bytes, stream
    ok = [16, 16, 8, None, 25, 16, 16, 64, 64, 256, 16, 16, 16, 16, 16, mw, None]
    for i in (0, 1, 5, 6, 10, 11, 12, 13, 14):
        bad = list(ok); bad[i] = None
        assert h.pope_fine_merge_coarse_f32_ex(*bad) == -1, i
    bad = list(ok); bad[2] = -5
    assert h.pope_fine_merge_coarse_f32_ex(*bad) == -1
    bad = list(ok); bad[4] = 0
    assert h.pope_fine_merge_coarse_f32_ex(*bad) == -1
    bad = list(ok); bad[9] = 128                                   # coarse width other than 256
    assert h.pope_fine_merge_coarse_f32_ex(*bad) == -4
    bad = list(ok); bad[15] = mw - 1
    assert h.pope_fine_merge_coarse_f32_ex(*bad) == -3
    bad = list(ok); bad[0] = 24
    assert h.pope_fine_merge_coarse_f32_ex(*bad) == -5
    bad = list(ok); bad[2] = 1 << 27
    assert h.pope_fine_merge_coarse_f32_ex(*bad) == -4
    bad = list(ok); bad[2] = 0
    assert h.pope_fine_merge_coarse_f32_ex(*bad) == 0


def test_set_fine_level_ex_rejects_a_null_handle():
    kinds = (_lib.C.c_int * 2)(0, 1)
    for dtype in (_lib.POPE_BF16, _lib.POPE_F32):
        assert _lib.lib().pope_pipeline_set_fine_level_ex(None, dtype, 16, 16, 2, kinds) == -1
        assert _lib.lib().pope_pipeline_set_fine_level_ex(None, dtype, None, None, 0, None) == -1


def test_fine_level_fp32_packs_the_matcher_weights():
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    cpu = torch.device("cpu")
    fl = m.fine_level("cpu", dtype=torch.float32)
    assert fl["dtype"] == torch.float32 and fl["layer_names"] == m.loftr_fine.layer_names
    assert fl["layers"].numel() == len(fl["layer_names"]) * _lib.FINE_TF_F32_LAYER_BYTES
    assert fl["pre"].numel() == _lib.FINE_PRE_F32_BYTES
    assert fl["layers"] is m.loftr_fine._packed_weights(cpu, torch.float32)      # the modules' caches
    assert fl["pre"] is m.fine_preprocess._packed_weights(cpu, torch.float32)
    assert fl["layers"] is m.fine_level("cpu", dtype=torch.float32)["layers"]
    # the default call packs what it packed before, and says so
    dflt = m.fine_level("cpu")
    assert dflt["dtype"] == torch.bfloat16
    assert torch.equal(dflt["layers"], torch.cat([ops.pack_fine_layer(l.state_dict(), cpu) for l in m.loftr_fine.layers]))
    assert torch.equal(dflt["pre"], ops.pack_fine_pre(m.fine_preprocess.state_dict(), cpu))
    assert dflt["layers"] is m.loftr_fine._packed_weights(cpu)
    with pytest.raises(_lib.PopeError):
        m.fine_level("cpu", dtype=torch.float16)
    cfg = pope_b200.make_default_cfg()
    cfg["fine_concat_coarse_feat"] = False
    assert pope_b200.Matcher(cfg).fine_level("cpu", dtype=torch.float32)["pre"] is None


def test_pipeline_rejects_an_fp32_fine_level_it_cannot_run_before_touching_the_gpu():
    fl = pope_b200.Matcher(pope_b200.make_default_cfg()).eval().fine_level("cpu", dtype=torch.float32)
    args = (2, (160, 192), (20, 24), (20, 24))
    with pytest.raises(_lib.PopeError, match="float32"):                       # an fp32 bundle on a bf16 pipeline
        driver.Pipeline(torch.bfloat16, *args, fine_level=fl)
    with pytest.raises(_lib.PopeError, match="layer names"):                   # bf16-sized layers labelled fp32
        driver.Pipeline(torch.float32, *args, fine_level=dict(fl, layers=fl["layers"][:_lib.FINE_TF_LAYER_BYTES * 2]))
    with pytest.raises(_lib.PopeError, match="FinePreprocess"):
        driver.Pipeline(torch.float32, *args, fine_level=dict(fl, pre=fl["pre"][:_lib.FINE_PRE_BYTES]))
    with pytest.raises(_lib.PopeError, match="C_coarse"):
        driver.Pipeline(torch.float32, *args, C_coarse=128, fine_level=fl)
    with pytest.raises(_lib.PopeError, match="cuda"):                          # packed weights on the CPU
        driver.Pipeline(torch.float32, *args, fine_level=fl)


# ---- GPU -----------------------------------------------------------------------------------------------------------

DEV = torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("ww", [25, 9])
@pytest.mark.parametrize("names", [["self"], ["cross"]])
@pytest.mark.parametrize("live", LIVE)
def test_bounded_fp32_transformer_equals_unbounded_on_the_live_windows(names, live, ww):
    gen = torch.Generator().manual_seed(7 + live + ww)
    packed = torch.cat([ops.pack_fine_layer(_random_layer(gen), DEV, dtype=torch.float32) for _ in names])
    w0, w1 = _sentinel_windows(gen, DEV, live, ww), _sentinel_windows(gen, DEV, live, ww)
    before0, before1 = w0.clone(), w1.clone()
    want0, want1 = w0[:live].clone(), w1[:live].clone()
    ops.fine_transformer(want0, want1, packed, names)
    m_dev = torch.tensor([live], dtype=torch.int32, device=DEV)
    ws = ops.fine_level_workspace(CAP, ww, DEV, merge=False, dtype=torch.float32)
    ops._fine_transformer(w0, w1, packed, names, ws, m_dev)
    torch.cuda.synchronize()
    for got, want, before in ((w0, want0, before0), (w1, want1, before1)):
        assert torch.equal(_bits(got[:live]), _bits(want)), live
        assert torch.equal(_bits(got[live:]), _bits(before[live:])), live
        assert torch.isfinite(got[:live]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("ww", [25, 9])
@pytest.mark.parametrize("live", LIVE + (700,))
def test_bounded_fp32_merge_equals_unbounded_on_both_sides(live, ww):
    """The window part runs in chunks of 4 * CAP rows: 1003 and 700 windows end inside a chunk other than the first."""
    gen = torch.Generator().manual_seed(31 + live + ww)
    n, L, S = 3, 300, 280
    fc0 = torch.randn(n, L, 256, generator=gen).to(DEV)
    fc1 = torch.randn(n, S, 256, generator=gen).to(DEV)
    b = torch.randint(0, n, (CAP,), generator=gen).to(DEV)
    i = torch.randint(0, L, (CAP,), generator=gen).to(DEV)
    j = torch.randint(0, S, (CAP,), generator=gen).to(DEV)
    pre = ops.pack_fine_pre(_random_pre(gen), DEV, dtype=torch.float32)
    w0, w1 = _sentinel_windows(gen, DEV, live, ww), _sentinel_windows(gen, DEV, live, ww)
    before0, before1 = w0.clone(), w1.clone()
    want0, want1 = w0[:live].clone(), w1[:live].clone()
    ops.fine_merge_coarse(want0, want1, fc0, fc1, b[:live], i[:live], j[:live], pre)
    ws = ops.fine_level_workspace(CAP, ww, DEV, transformer=False, dtype=torch.float32)
    ops._fine_merge_coarse(w0, w1, fc0, fc1, b, i, j, pre, ws, torch.tensor([live], dtype=torch.int32, device=DEV))
    torch.cuda.synchronize()
    for side, (got, want, before) in enumerate(((w0, want0, before0), (w1, want1, before1))):
        assert torch.equal(_bits(got[:live]), _bits(want)), (live, side)
        assert torch.equal(_bits(got[live:]), _bits(before[live:])), (live, side)


def _shapes(h, w, n):
    return {"hw0_i": torch.Size([h * 8, w * 8]), "hw1_i": torch.Size([h * 8, w * 8]), "hw0_c": torch.Size([h, w]),
            "hw1_c": torch.Size([h, w]), "hw0_f": torch.Size([h * 4, w * 4]), "hw1_f": torch.Size([h * 4, w * 4]), "bs": n}


def _matcher(seed=0, **cfg_changes):
    torch.manual_seed(seed)
    cfg = pope_b200.make_default_cfg()
    cfg.update(cfg_changes)
    return pope_b200.Matcher(cfg, fine_cuda_fp32=True).eval().to(DEV)


def _inputs(seed, n, h, w, channels_last=True):
    f0, f1 = synth.coarse_features(seed, n, h * w, h * w, 256, sigma=0.9)
    ff0, ff1 = synth.fine_feature_maps(seed + 1, n, h * 4, w * 4, 128, channels_last=channels_last)
    return [t.to(DEV) for t in (f0, f1, ff0, ff1)]


KEYS = ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f", "expec_f")


@pytest.mark.gpu
@pytest.mark.parametrize("concat", [True, False])
@pytest.mark.parametrize("n,h,w", [(2, 20, 24), (8, 60, 80)])
def test_fp32_step_with_fine_level_equals_the_matcher(n, h, w, concat):
    m = _matcher(fine_concat_coarse_feat=concat)
    f0, f1, ff0, ff1 = _inputs(40 + n, n, h, w, channels_last=False)
    data = _shapes(h, w, n)
    with torch.no_grad():
        m.coarse_matching(f0, f1, data)
        w0, w1 = m.fine_preprocess(ff0, ff1, f0, f1, data)
        w0, w1 = m.loftr_fine(w0, w1)
        m.fine_matching(w0, w1, data)
    fl = m.fine_level(DEV, dtype=torch.float32)
    assert (fl["pre"] is None) == (not concat)
    res = ops.match_pairs_device(f0, f1, ff0, ff1, data["hw0_i"], (h, w), (h, w), fine_level=fl)
    assert res["win0"].dtype == torch.float32
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
def test_fp32_step_with_fine_level_is_graph_capturable():
    """With the fp32 level the step has no host sync either: it is captured into a CUDA graph, and replays on new feature
    contents equal eager calls bit for bit."""
    n, h, w = 24, 40, 48
    m = _matcher(1)
    fl = m.fine_level(DEV, dtype=torch.float32)
    sets = [_inputs(seed, n, h, w) for seed in (301, 302)]
    hw_i = (h * 8, w * 8)
    want = []
    for s in sets:
        r = ops.match_pairs_device(*s, hw_i, (h, w), (h, w), fine_level=fl)
        k = r.total()
        assert k > 5000 and r.flags() == 0
        want.append((k, {key: r[key][:k].clone() for key in KEYS}))
    static = [t.clone() for t in sets[0]]
    ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, h * w, h * w, 256, _lib.POPE_F32), dtype=torch.uint8,
                     device=DEV)
    fws = ops.fine_level_workspace(n * h * w, 25, DEV, dtype=torch.float32)
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
def test_batch_runner_with_fp32_fine_level_equals_sequential_steps_and_job_gather_stays_exact():
    n, h, w = 2, 20, 24
    m = _matcher(2)
    fl = m.fine_level(DEV, dtype=torch.float32)
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
def test_fp32_step_with_fine_level_and_zero_matches():
    n, h, w = 2, 20, 24
    m = _matcher(3)
    fl = m.fine_level(DEV, dtype=torch.float32)
    f0, f1, ff0, ff1 = _inputs(70, n, h, w)
    f1 = torch.zeros_like(f1)             # every similarity 0: uniform softmaxes, confidence 1 / (L S), no match
    res = ops.match_pairs_device(f0, f1, ff0, ff1, (h * 8, w * 8), (h, w), (h, w), fine_level=fl)
    assert res.total() == 0 and res.flags() == 0
    # the step's own count (0) bounds every fine-level launch: windows given to them keep every byte
    m_dev = res["counts"][n:n + 1]
    gen = torch.Generator().manual_seed(71)
    cap = res["b_ids"].shape[0]
    w0 = torch.randn(cap, 25, 128, generator=gen).to(DEV)
    w1 = torch.randn(cap, 25, 128, generator=gen).to(DEV)
    before0, before1 = w0.clone(), w1.clone()
    ws = ops.fine_level_workspace(cap, 25, DEV, dtype=torch.float32)
    ops._fine_merge_coarse(w0, w1, f0, f1, res["b_ids"], res["i_ids"], res["j_ids"], fl["pre"], ws, m_dev)
    ops._fine_transformer(w0, w1, fl["layers"], fl["layer_names"], ws, m_dev)
    torch.cuda.synchronize()
    assert torch.equal(_bits(w0), _bits(before0)) and torch.equal(_bits(w1), _bits(before1))


@pytest.mark.gpu
def test_fp32_step_with_fine_level_rejects_mixes():
    n, h, w = 1, 20, 24
    m = _matcher(4)
    fl = m.fine_level(DEV, dtype=torch.float32)
    f0, f1, ff0, ff1 = _inputs(80, n, h, w)
    args = ((h * 8, w * 8), (h, w), (h, w))
    bf = [t.bfloat16() for t in (f0, f1, ff0, ff1)]
    with pytest.raises(_lib.PopeError):                                        # fp32 bundle, bf16 features and maps
        ops.match_pairs_device(*bf, *args, fine_level=fl)
    with pytest.raises(_lib.PopeError):                                        # fp32 coarse features, bf16 maps
        ops.match_pairs_device(f0, f1, bf[2], bf[3], *args, fine_level=fl)
    with pytest.raises(_lib.PopeError):                                        # bf16 coarse features, fp32 maps
        ops.match_pairs_device(bf[0], bf[1], ff0, ff1, *args, fine_level=fl)
    with pytest.raises(_lib.PopeError):                                        # the fused route has no fine level
        ops.match_pairs_device(f0, f1, ff0, ff1, *args, fine_level=fl, fused_fine=True)
    with pytest.raises(_lib.PopeError):                                        # a bundle packed for another dtype
        ops.match_pairs_device(f0, f1, ff0, ff1, *args, fine_level=dict(fl, dtype=torch.float16))
