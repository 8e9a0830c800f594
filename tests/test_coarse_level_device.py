"""The coarse level (position encoding + coarse LoFTR transformer) inside the sync-free device step, so that the batched
forms start where the backbone stops: `pope_coarse_pos_encode_ex`, `ops.coarse_pos_encode(dtype=)`,
`Matcher.coarse_level(device, dtype)`, `ops.match_pairs_device(coarse_level=)`, `DeviceBatchRunner.submit(coarse_level=)`.

The reference is the real `Matcher.forward` with `coarse_cuda_X=True, fine_cuda_X=True`, its backbone replaced by a stub
that returns prepared coarse and fine maps.  The step runs the same kernels on the same values (every pair's transformer
output depends on that pair's inputs only), so ids, confidences and keypoints are compared bit for bit."""
import pytest
import torch
import torch.nn as nn

import pope_b200
from pope_b200 import _lib, driver, ops, synth

DTYPES = {"bf16": torch.bfloat16, "fp32": torch.float32}


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int32)


def _maps(seed, n, hw0, hw1, sigma=0.9):
    """CPU fp32 backbone outputs: coarse maps [n, 256, h, w] with planted correspondences, fine maps [n, 128, 4h, 4w]"""
    (h0, w0), (h1, w1) = hw0, hw1
    f0, f1 = synth.coarse_features(seed, n, h0 * w0, h1 * w1, 256, sigma=sigma)
    c0 = f0.transpose(1, 2).reshape(n, 256, h0, w0).contiguous()
    c1 = f1.transpose(1, 2).reshape(n, 256, h1, w1).contiguous()
    ff0, ff1 = synth.fine_feature_maps(seed + 1, n, 4 * max(h0, h1), 4 * max(w0, w1), 128, channels_last=False)
    return c0, c1, ff0[:, :, :4 * h0, :4 * w0].contiguous(), ff1[:, :, :4 * h1, :4 * w1].contiguous()


# ---- CPU: argument checking and the weight bundle ------------------------------------------------------------------

def test_coarse_level_returns_the_module_caches_and_rejects_bad_dtypes():
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    cpu = torch.device("cpu")
    for dt, per_layer in ((torch.bfloat16, _lib.COARSE_TF_LAYER_BYTES), (torch.float32, _lib.COARSE_TF_F32_LAYER_BYTES)):
        cl = m.coarse_level("cpu", dtype=dt)
        assert cl["dtype"] == dt and cl["layer_names"] == m.loftr_coarse.layer_names
        assert cl["pe"] is m.pos_encoding.pe
        assert cl["layers"] is m.loftr_coarse._packed_weights(cpu, dt)
        assert cl["layers"].numel() == len(cl["layer_names"]) * per_layer
        assert cl["layers"] is m.coarse_level("cpu", dtype=dt)["layers"]
        assert torch.equal(cl["layers"], torch.cat([ops.pack_coarse_layer(l.state_dict(), cpu, dt)
                                                    for l in m.loftr_coarse.layers]))
    assert m.coarse_level("cpu")["dtype"] == torch.bfloat16
    for bad in (torch.float16, torch.float64):
        with pytest.raises(_lib.PopeError):
            m.coarse_level("cpu", dtype=bad)
    cfg = pope_b200.make_default_cfg()
    cfg["coarse"]["attention"] = "full"
    with pytest.raises(NotImplementedError):
        pope_b200.Matcher(cfg).coarse_level("cpu")


def test_pos_encode_ex_rejects_bad_arguments_before_touching_the_gpu():
    h = _lib.lib()
    # feat, pe, n, C, H, W, pe_h, pe_w, out, out_dtype, stream
    for dt in (_lib.POPE_BF16, _lib.POPE_F32):
        ok = [16, 16, 2, 256, 60, 80, 256, 256, 16, dt, None]
        for i in (0, 1, 8):                                        # null map, encoding and output
            bad = list(ok); bad[i] = None
            assert h.pope_coarse_pos_encode_ex(*bad) == -1, i
        for i, v in ((2, -1), (4, 0), (5, 0), (6, 0)):             # negative / empty sizes
            bad = list(ok); bad[i] = v
            assert h.pope_coarse_pos_encode_ex(*bad) == -1, i
        for i, v in ((3, 128), (4, 257), (5, 300)):                # C != 256, map larger than the encoding
            bad = list(ok); bad[i] = v
            assert h.pope_coarse_pos_encode_ex(*bad) == -4, i
        for i, v in ((0, 18), (1, 6), (8, 24)):                    # misaligned map, encoding, output
            bad = list(ok); bad[i] = v
            assert h.pope_coarse_pos_encode_ex(*bad) == -5, i
        bad = list(ok); bad[2] = 0                                 # no maps: a no-op
        assert h.pope_coarse_pos_encode_ex(*bad) == 0
    for dt in (2, -1, 7):                                          # neither POPE_BF16 nor POPE_F32
        assert h.pope_coarse_pos_encode_ex(16, 16, 2, 256, 60, 80, 256, 256, 16, dt, None) == -2, dt


def test_set_coarse_level_rejects_a_null_handle():
    kinds = (_lib.C.c_int * 2)(0, 1)
    for dtype in (_lib.POPE_BF16, _lib.POPE_F32):
        assert _lib.lib().pope_pipeline_set_coarse_level(None, dtype, 16, 256, 256, 16, 2, kinds) == -1
        assert _lib.lib().pope_pipeline_set_coarse_level(None, dtype, None, 0, 0, None, 0, None) == -1


def test_pipeline_rejects_a_coarse_level_it_cannot_run_before_touching_the_gpu():
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    cl = m.coarse_level("cpu", dtype=torch.float32)
    args = (2, (160, 192), (20, 24), (20, 24))
    with pytest.raises(_lib.PopeError, match="float32"):                       # an fp32 bundle on a bf16 pipeline
        driver.Pipeline(torch.bfloat16, *args, coarse_level=cl)
    with pytest.raises(_lib.PopeError, match="bfloat16"):                      # a bf16 bundle on an fp32 pipeline
        driver.Pipeline(torch.float32, *args, coarse_level=m.coarse_level("cpu"))
    with pytest.raises(_lib.PopeError, match="layer names"):                   # bf16-sized layers labelled fp32
        driver.Pipeline(torch.float32, *args, coarse_level=dict(cl, layers=cl["layers"][:_lib.COARSE_TF_LAYER_BYTES * 8]))
    with pytest.raises(_lib.PopeError, match="layer names"):
        driver.Pipeline(torch.float32, *args, coarse_level=dict(cl, layer_names=["self"]))
    with pytest.raises(_lib.PopeError, match="C_coarse"):
        driver.Pipeline(torch.float32, *args, C_coarse=128, coarse_level=cl)
    with pytest.raises(_lib.PopeError, match="larger"):                         # a grid beyond the 256 x 256 encoding
        driver.Pipeline(torch.float32, 2, (160, 2400), (20, 300), (20, 24), coarse_level=cl)
    with pytest.raises(_lib.PopeError, match="cuda"):                          # the bundle on the CPU
        driver.Pipeline(torch.float32, *args, coarse_level=cl)
    with pytest.raises(_lib.PopeError):                                        # what match_pairs_host passes on
        driver.match_pairs_host(*_maps(1, 2, (20, 24), (20, 24)), (160, 192), (20, 24), (20, 24), coarse_level=cl)


def test_step_rejects_what_the_coarse_level_cannot_run_before_any_launch():
    m = pope_b200.Matcher(pope_b200.make_default_cfg()).eval()
    c0, c1, ff0, ff1 = _maps(2, 1, (20, 24), (20, 24))
    args = ((160, 192), (20, 24), (20, 24))
    cl32, cl16 = m.coarse_level("cpu", dtype=torch.float32), m.coarse_level("cpu")
    fl32, fl16 = m.fine_level("cpu", dtype=torch.float32), m.fine_level("cpu")
    step = ops.match_pairs_device
    with pytest.raises(_lib.PopeError, match="one dtype"):                     # bf16 coarse level, fp32 fine level
        step(c0, c1, ff0, ff1, *args, coarse_level=cl16, fine_level=fl32)
    with pytest.raises(_lib.PopeError, match="one dtype"):
        step(c0, c1, ff0, ff1, *args, coarse_level=cl32, fine_level=fl16)
    with pytest.raises(_lib.PopeError, match="fp32 maps"):                     # maps that are not fp32
        step(c0.bfloat16(), c1.bfloat16(), ff0, ff1, *args, coarse_level=cl32)
    with pytest.raises(_lib.PopeError, match="fp32 maps"):                     # token-major features, not maps
        step(c0.flatten(2).transpose(1, 2), c1.flatten(2).transpose(1, 2), ff0, ff1, *args, coarse_level=cl32)
    with pytest.raises(_lib.PopeError, match="C = 256"):
        step(c0[:, :128], c1[:, :128], ff0, ff1, *args, coarse_level=cl32)
    with pytest.raises(_lib.PopeError, match="hw_c"):                          # grid other than hw0_c
        step(c0, c1, ff0, ff1, (160, 192), (24, 20), (20, 24), coarse_level=cl32)
    big = torch.zeros(1, 256, 8, 260)
    with pytest.raises(_lib.PopeError, match="larger"):                        # grid beyond the encoding
        step(big, big, ff0, ff1, (64, 2080), (8, 260), (8, 260), coarse_level=cl32)
    with pytest.raises(_lib.PopeError):
        step(c0, c1, ff0, ff1, *args, coarse_level=dict(cl32, dtype=torch.float16))
    with pytest.raises(_lib.PopeError, match="CUDA"):                          # all of it well formed, on the CPU
        step(c0, c1, ff0, ff1, *args, coarse_level=cl32, fine_level=fl32)


# ---- GPU -----------------------------------------------------------------------------------------------------------

DEV = torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("temp_bug_fix", [True, False])
def test_fp32_pos_encode_is_bit_identical_to_torch(temp_bug_fix):
    pe = pope_b200.feature_net.PositionEncodingSine(256, temp_bug_fix=temp_bug_fix).to(DEV)
    gen = torch.Generator().manual_seed(5)
    for n, h, w in ((2, 60, 80), (1, 32, 32), (3, 7, 9), (1, 256, 256), (2, 33, 250)):
        x = (3 * torch.randn(n, 256, h, w, generator=gen)).to(DEV)
        want = pe(x).flatten(2).transpose(1, 2)
        got = ops.coarse_pos_encode(x, pe.pe, dtype=torch.float32)
        assert got.dtype == torch.float32 and got.is_contiguous() and got.shape == want.shape
        assert torch.equal(_bits(got), _bits(want)), (n, h, w)
        # the default is the bf16 encoding of before, and the bf16 output is the fp32 one rounded once
        b = ops.coarse_pos_encode(x, pe.pe)
        assert b.dtype == torch.bfloat16 and torch.equal(b.view(torch.int16), got.to(torch.bfloat16).view(torch.int16))


class _Backbone(nn.Module):
    """Stands in for the ResNet-FPN: returns prepared maps, so that the real Matcher.forward runs on them."""

    def __init__(self, c0, c1, ff0, ff1):
        super().__init__()
        self.maps = (c0, c1, ff0, ff1)

    def forward(self, x):
        c0, c1, ff0, ff1 = self.maps
        if x.shape[0] == 2 * c0.shape[0]:                # equal image sizes: one call on torch.cat([img0, img1])
            return torch.cat([c0, c1]), torch.cat([ff0, ff1])
        return (c0, ff0) if tuple(x.shape[2:]) == (8 * c0.shape[2], 8 * c0.shape[3]) else (c1, ff1)


def _matcher(dt, maps, seed=0, **cfg_changes):
    torch.manual_seed(seed)
    cfg = pope_b200.make_default_cfg()
    cfg.update(cfg_changes)
    f32 = dt == torch.float32
    m = pope_b200.Matcher(cfg, coarse_cuda_bf16=not f32, fine_cuda_bf16=not f32, coarse_cuda_fp32=f32,
                          fine_cuda_fp32=f32).eval().to(DEV)
    m.backbone = _Backbone(*maps)
    return m


def _images(maps):
    c0, c1 = maps[0], maps[1]
    return {"image0": torch.zeros(c0.shape[0], 1, 8 * c0.shape[2], 8 * c0.shape[3], device=DEV),
            "image1": torch.zeros(c1.shape[0], 1, 8 * c1.shape[2], 8 * c1.shape[3], device=DEV)}


def _step_args(maps, dt):
    """the step's inputs: the coarse maps as they are, the fine maps in the level's dtype (the Matcher's bf16 fine level
    rounds them once, the fp32 one takes them as they are)"""
    c0, c1, ff0, ff1 = maps
    return (c0, c1, ff0.to(dt), ff1.to(dt), (8 * c0.shape[2], 8 * c0.shape[3]), tuple(c0.shape[2:]), tuple(c1.shape[2:]))


CASES = [(2, (20, 24), (20, 24)), (8, (60, 80), (60, 80)), (2, (60, 80), (32, 32))]
KEYS = ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f", "expec_f")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("n,hw0,hw1", CASES)
def test_step_with_both_levels_equals_the_matcher(dt, n, hw0, hw1):
    dt = DTYPES[dt]
    maps = [t.to(DEV) for t in _maps(60 + n, n, hw0, hw1)]
    before = [t.clone() for t in maps]
    m = _matcher(dt, maps)
    data = _images(maps)
    with torch.no_grad():
        m(data)
        att0, att1 = m(_images(maps), only_att_fea=True)
    cl, fl = m.coarse_level(DEV, dt), m.fine_level(DEV, dt)
    res = ops.match_pairs_device(*_step_args(maps, dt), coarse_level=cl, fine_level=fl)
    k = res.total()
    assert k == data["b_ids"].numel() and k > 100 and res.flags() == 0
    for key in ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_f"):
        assert torch.equal(res[key][:k], data[key]), key
    for key in ("expec_f", "mkpts1_f"):
        assert torch.equal(_bits(res[key][:k]), _bits(data[key])), key
    assert res["feat_c0"].dtype == dt and res["feat_c0"].shape == (n, hw0[0] * hw0[1], 256)
    assert torch.equal(res["feat_c0"], att0) and torch.equal(res["feat_c1"], att1)
    assert res["coarse_workspace"].numel() >= ops.coarse_tf_workspace(n, hw0[0] * hw0[1], hw1[0] * hw1[1], DEV,
                                                                      dtype=dt).numel()
    # the maps are inputs, not scratch: neither the Matcher nor the step wrote to them
    assert all(torch.equal(_bits(t), _bits(b)) for t, b in zip(maps, before))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
def test_coarse_level_alone_gives_the_matchers_coarse_match(dt):
    dt = DTYPES[dt]
    n, hw0, hw1 = 3, (30, 40), (24, 32)
    maps = [t.to(DEV) for t in _maps(70, n, hw0, hw1)]
    m = _matcher(dt, maps, 1)
    data = _images(maps)
    with torch.no_grad():
        m(data)
    res = ops.match_pairs_device(*_step_args(maps, dt), coarse_level=m.coarse_level(DEV, dt))
    k = res.total()
    assert k == data["b_ids"].numel() and k > 100 and res.flags() == 0
    for key in ("b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c"):
        assert torch.equal(res[key][:k], data[key]), key


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
def test_step_with_both_levels_is_graph_capturable(dt):
    """No host sync with the coarse level either: the step is captured into a CUDA graph, and replays on new map contents
    equal eager calls bit for bit."""
    dt = DTYPES[dt]
    n, hw = 6, (40, 48)
    L = hw[0] * hw[1]
    sets = [[t.to(DEV) for t in _maps(seed, n, hw, hw)] for seed in (401, 402)]
    m = _matcher(dt, sets[0], 2)
    cl, fl = m.coarse_level(DEV, dt), m.fine_level(DEV, dt)
    want = []
    for s in sets:
        r = ops.match_pairs_device(*_step_args(s, dt), coarse_level=cl, fine_level=fl)
        k = r.total()
        assert k > 1000 and r.flags() == 0
        want.append((k, {key: r[key][:k].clone() for key in KEYS + ("feat_c0", "feat_c1")}))
    static = [t.clone() for t in _step_args(sets[0], dt)[:4]]
    tail = _step_args(sets[0], dt)[4:]
    ws = torch.empty(_lib.lib().pope_coarse_workspace_bytes_ex(n, L, L, 256, _lib.dtype_code(static[2])),
                     dtype=torch.uint8, device=DEV)
    fws = ops.fine_level_workspace(n * L, 25, DEV, dtype=dt)
    cws = ops.coarse_tf_workspace(n, L, L, DEV, dtype=dt)
    kw = dict(workspace=ws, fine_level=fl, fine_workspace=fws, coarse_level=cl, coarse_workspace=cws)
    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):                      # warm-up on the capture stream (first-use attribute calls)
        ops.match_pairs_device(*static, *tail, **kw)
    torch.cuda.current_stream(DEV).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        res = ops.match_pairs_device(*static, *tail, **kw)
    assert res["coarse_workspace"] is cws
    for which in (1, 0, 1):
        for dst, src in zip(static, _step_args(sets[which], dt)[:4]):
            dst.copy_(src)
        graph.replay()
        torch.cuda.synchronize()
        k, ref = want[which]
        assert res.total() == k and res.flags() == 0
        for key in KEYS:
            assert torch.equal(_bits(res[key][:k]), _bits(ref[key])), (which, key)
        assert torch.equal(res["feat_c0"], ref["feat_c0"]) and torch.equal(res["feat_c1"], ref["feat_c1"])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
def test_batch_runner_with_both_levels_equals_sequential_steps_and_job_gather_stays_exact(dt):
    dt = DTYPES[dt]
    n, hw = 2, (20, 24)
    batches = [[t.to(DEV) for t in _maps(seed, n, hw, hw)] for seed in (91, 93, 95, 97)]
    m = _matcher(dt, batches[0], 3)
    cl, fl = m.coarse_level(DEV, dt), m.fine_level(DEV, dt)
    runner = driver.DeviceBatchRunner(DEV, 2)
    job = driver.JobGather(len(batches), n * hw[0] * hw[1], DEV)
    steps = [_step_args(b, dt) for b in batches]       # (the bf16 fine maps are made here, before the fork)
    runner.fork()
    got = [runner.submit(*args, after=lambda r, k=k: job.add(r, 10 * k), fine_level=fl, coarse_level=cl)[0]
           for k, args in enumerate(steps)]
    assert all(ws is not None for ws in runner.coarse_workspaces)
    assert got[2]["coarse_workspace"] is got[0]["coarse_workspace"]          # one scratch per stream, reused
    runner.join()
    recs, sizes = job.finish()
    torch.cuda.synchronize()
    rec = driver.unpack_records(recs[0].cpu())
    off = 0
    for k, (args, res) in enumerate(zip(steps, got)):
        want = ops.match_pairs_device(*args, fine_level=fl, coarse_level=cl)
        c = want.total()
        assert res.total() == c and c > 100
        for key in KEYS:
            assert torch.equal(_bits(res[key][:c]), _bits(want[key][:c])), (k, key)
        assert torch.equal(res["feat_c0"], want["feat_c0"]) and torch.equal(res["feat_c1"], want["feat_c1"])
        assert torch.equal(rec["b_ids"][off:off + c], want["b_ids"][:c].cpu() + 10 * k)
        for key in ("i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f"):
            assert torch.equal(rec[key][off:off + c], want[key][:c].cpu()), (k, key)
        off += c
    assert sizes == [off]


@pytest.mark.gpu
def test_step_with_coarse_level_rejects_mixes_on_the_device():
    maps = [t.to(DEV) for t in _maps(80, 1, (20, 24), (20, 24))]
    m = _matcher(torch.float32, maps, 4)
    args = _step_args(maps, torch.float32)
    cl32, cl16 = m.coarse_level(DEV, torch.float32), m.coarse_level(DEV)
    fl32, fl16 = m.fine_level(DEV, torch.float32), m.fine_level(DEV)
    c0, c1 = maps[0], maps[1]
    for kw in (dict(coarse_level=cl16, fine_level=fl32), dict(coarse_level=cl32, fine_level=fl16)):
        with pytest.raises(_lib.PopeError, match="one dtype"):
            ops.match_pairs_device(*args, **kw)
    with pytest.raises(_lib.PopeError, match="fp32 maps"):
        ops.match_pairs_device(c0.bfloat16(), c1.bfloat16(), *args[2:], coarse_level=cl16)
    with pytest.raises(_lib.PopeError, match="C = 256"):
        ops.match_pairs_device(c0[:, :128].contiguous(), c1[:, :128].contiguous(), *args[2:], coarse_level=cl32)
    with pytest.raises(_lib.PopeError, match="layer names"):
        ops.match_pairs_device(*args, coarse_level=dict(cl32, layers=cl16["layers"]))
    with pytest.raises(_lib.PopeError):                # a bf16 fine level needs bf16 fine maps, coarse level or not
        ops.match_pairs_device(*args, coarse_level=cl16, fine_level=fl16)
