"""Pair-batching driver: batches of independent image pairs through the hot path, on one GPU (chunked stream
pipeline in libpope_b200.so) or sharded over the GPUs of one box with a single gather of the match lists.

Replaces the batch-1 loops of the eval drivers (eval_linemod_json.py:103-122, eval_onepose_json.py:103-124,
eval_ycb_json.py:86-105: three sequential `matcher(batch)` calls per test pair, `.cpu()` after each).
Pairs are independent, so ranks share nothing on the data path; the only cross-GPU step is `gather_matches`
(SURVEY.md section 8(e)).
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Callable, Dict, Optional, Sequence

import torch

from . import _lib
from ._lib import check, dtype_code, lib


def _pin(t: torch.Tensor) -> torch.Tensor:
    t = t.contiguous()
    if t.device.type != "cpu":
        raise _lib.PopeError("the host pipeline takes CPU (preferably pinned) tensors")
    return t


def _fine_to_nhwc(ff: torch.Tensor) -> torch.Tensor:
    """logical [N, Cf, H, W] (any strides) -> memory [N, H, W, Cf]; free for channels-last inputs."""
    return ff.permute(0, 2, 3, 1).contiguous()


def _check_fine_level(fine_level: dict, dtype: torch.dtype, C_coarse: int, device: int):
    """What `pope_pipeline_set_fine_level` needs, checked before any GPU call; returns its (pre, layers, kinds) arguments."""
    if dtype != torch.bfloat16 or C_coarse != 256:
        raise _lib.PopeError("the bf16 fine level needs a bfloat16 pipeline with C_coarse = 256")
    names, layers, pre = list(fine_level["layer_names"]), fine_level["layers"], fine_level["pre"]
    if not names or any(nm not in ("self", "cross") for nm in names) \
            or layers.numel() != len(names) * _lib.FINE_TF_LAYER_BYTES:
        raise _lib.PopeError("the fine level's layer names and packed layers do not agree")
    if pre is not None and pre.numel() != _lib.FINE_PRE_BYTES:
        raise _lib.PopeError("the fine level's packed FinePreprocess weights have the wrong size")
    dev = torch.device("cuda", device)
    for t in (layers, pre):
        if t is not None and (t.device != dev or t.dtype != torch.uint8 or not t.is_contiguous()):
            raise _lib.PopeError(f"the fine level's packed weights must be contiguous uint8 tensors on {dev} "
                                 f"(Matcher.fine_level({dev}))")
    return pre, layers, (C.c_int * len(names))(*[0 if nm == "self" else 1 for nm in names])


class Pipeline:
    """Owns one `pope_pipeline_t` (device slots + streams for one geometry).

    `fine_level` (`Matcher.fine_level(torch.device("cuda", device))`): every chunk also runs what Matcher.forward runs between
    window gather and fine matching -- FinePreprocess' two Linears and the fine transformer, in bf16 -- so that the results
    equal `ops.match_pairs_device(..., fine_level=...)` and thereby `Matcher(config, fine_cuda_bf16=True)`, bit for bit.
    Needs a bf16 pipeline with C_coarse = 256.  The pipeline keeps a reference to the dict, so the packed weights outlive
    the handle; it allocates windows and fine scratch for one chunk (0.98 GB + 2.5 GB at 16 pairs of 480x640)."""

    def __init__(self, dtype: torch.dtype, chunk_pairs: int, hw0_i: Sequence[int], hw0_c: Sequence[int],
                 hw1_c: Sequence[int], C_coarse: int = 256, C_fine: int = 128, fine_stride: int = 4, W: int = 5,
                 thr: float = 0.2, border_rm: int = 2, temperature: float = 0.1, impl: int = _lib.COARSE_AUTO,
                 device: int = 0, fine_level: Optional[dict] = None):
        self.dtype, self.chunk, self.device = dtype, chunk_pairs, device
        self.hw0_c, self.hw1_c = tuple(hw0_c), tuple(hw1_c)
        self.L, self.S = hw0_c[0] * hw0_c[1], hw1_c[0] * hw1_c[1]
        self.cap = min(self.L, self.S)
        self.C, self.Cf, self.fstride, self.W = C_coarse, C_fine, fine_stride, W
        self._h = C.c_void_p()
        code = _lib.POPE_BF16 if dtype == torch.bfloat16 else _lib.POPE_F32
        if dtype not in (torch.float32, torch.bfloat16):
            raise _lib.PopeError(f"unsupported dtype {dtype}")
        if fine_level is not None:
            _check_fine_level(fine_level, dtype, C_coarse, device)
        pixel_scale = hw0_i[0] / hw0_c[0]
        fine_scale = hw0_i[0] / (hw0_c[0] * fine_stride)
        st = lib().pope_pipeline_create(C.byref(self._h), device, code, chunk_pairs, C_coarse, C_fine,
                                        hw0_c[0], hw0_c[1], hw1_c[0], hw1_c[1], fine_stride, W,
                                        float(pixel_scale), float(fine_scale), float(temperature), float(thr),
                                        int(border_rm), int(impl))
        check(st, "pope_pipeline_create")
        self.fine_level = None
        if fine_level is not None:
            try:
                self.set_fine_level(fine_level)
            except BaseException:
                self.close()
                raise

    def set_fine_level(self, fine_level: Optional[dict]) -> None:
        """Attach a fine level (see the class docstring) or, with None, detach it: the pipeline then returns what a pipeline
        created without one returns."""
        if fine_level is None:
            check(lib().pope_pipeline_set_fine_level(self._h, None, None, 0, None), "pope_pipeline_set_fine_level")
            self.fine_level = None
            return
        pre, layers, kinds = _check_fine_level(fine_level, self.dtype, self.C, self.device)
        # the weights may have been packed just now on torch's stream, which the pipeline's own streams do not wait for
        torch.cuda.current_stream(layers.device).synchronize()
        check(lib().pope_pipeline_set_fine_level(self._h, None if pre is None else pre.data_ptr(), layers.data_ptr(),
                                                 len(kinds), kinds), "pope_pipeline_set_fine_level")
        self.fine_level = fine_level          # keeps the packed tensors alive while the handle may read them

    def alloc_outputs(self, n: int, pinned: bool = True) -> Dict[str, torch.Tensor]:
        kw = dict(pin_memory=pinned)
        return {"i_ids": torch.empty(n, self.cap, dtype=torch.int64, **kw),
                "j_ids": torch.empty(n, self.cap, dtype=torch.int64, **kw),
                "mconf": torch.empty(n, self.cap, dtype=torch.float32, **kw),
                "mkpts0_f": torch.empty(n, self.cap, 2, dtype=torch.float32, **kw),
                "mkpts1_f": torch.empty(n, self.cap, 2, dtype=torch.float32, **kw),
                "counts": torch.empty(n, dtype=torch.int32, **kw),
                "flags": torch.zeros(1, dtype=torch.int32, **kw)}

    def run(self, feat_c0, feat_c1, feat_f0_nhwc, feat_f1_nhwc, out: Optional[Dict[str, torch.Tensor]] = None):
        """Inputs: CPU tensors feat_c* [n,L|S,C], feat_f*_nhwc [n,Hf,Wf,Cf] (memory order), same dtype.  Outputs: per-pair
        slots (`flatten_slots` packs them) holding what `ops.match_pairs_device` returns on the same inputs -- with the fine
        level attached, what it returns with `fine_level=`."""
        n = feat_c0.shape[0]
        for t in (feat_c0, feat_c1, feat_f0_nhwc, feat_f1_nhwc):
            if t.dtype != self.dtype or not t.is_contiguous() or t.device.type != "cpu":
                raise _lib.PopeError("pipeline inputs must be contiguous CPU tensors of the pipeline dtype")
        if out is None:
            out = self.alloc_outputs(n)
        st = lib().pope_pipeline_run(self._h, feat_c0.data_ptr(), feat_c1.data_ptr(), feat_f0_nhwc.data_ptr(),
                                     feat_f1_nhwc.data_ptr(), n, out["i_ids"].data_ptr(), out["j_ids"].data_ptr(),
                                     out["mconf"].data_ptr(), out["mkpts0_f"].data_ptr(), out["mkpts1_f"].data_ptr(),
                                     out["counts"].data_ptr(), out["flags"].data_ptr())
        check(st, "pope_pipeline_run")
        self.last_h2d_bytes = int(lib().pope_pipeline_last_h2d_bytes(self._h))
        self.last_f1_mode = ("bulk", "windows", "union")[int(lib().pope_pipeline_last_f1_mode(self._h))]
        return out

    def close(self):
        if self._h:
            lib().pope_pipeline_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def match_pairs_host(feat_c0, feat_c1, feat_f0, feat_f1, hw0_i, hw0_c, hw1_c, chunk_pairs: int = 16, device: int = 0,
                     fine_level: Optional[dict] = None, **kw) -> Dict[str, torch.Tensor]:
    """One-shot host-buffer entry: feat_f* are logical [N, Cf, Hf, Wf] CPU tensors (channels-last is free).  With
    `fine_level` (`Matcher.fine_level(torch.device("cuda", device))`) the results equal what
    `Matcher(config, fine_cuda_bf16=True)` computes from these features (see `Pipeline`)."""
    n = feat_c0.shape[0]
    pl = Pipeline(feat_c0.dtype, min(chunk_pairs, n), hw0_i, hw0_c, hw1_c, feat_c0.shape[2], feat_f0.shape[1],
                  feat_f0.shape[2] // hw0_c[0], device=device, fine_level=fine_level, **kw)
    try:
        return pl.run(_pin(feat_c0), _pin(feat_c1), _fine_to_nhwc(feat_f0), _fine_to_nhwc(feat_f1))
    finally:
        pl.close()


def flatten_slots(out: Dict[str, torch.Tensor], pair_offset: int = 0) -> Dict[str, torch.Tensor]:
    """Per-pair slots [n, cap] -> the reference's packed lists sorted by (b, i)."""
    counts = out["counts"].to(torch.int64)
    n, cap = out["i_ids"].shape
    live = torch.arange(cap)[None, :] < counts[:, None]
    b = torch.arange(n)[:, None].expand(n, cap)[live] + pair_offset
    return {"b_ids": b, "i_ids": out["i_ids"][live], "j_ids": out["j_ids"][live], "mconf": out["mconf"][live],
            "mkpts0_f": out["mkpts0_f"][live], "mkpts1_f": out["mkpts1_f"][live], "counts": out["counts"]}


# ---- batches of device-resident pairs -------------------------------------------------------------------------------

class DeviceBatchRunner:
    """Runs the hot path (`ops.match_pairs_device`) on a sequence of device-resident batches, consecutive batches on
    alternating CUDA streams with their own coarse scratch.  A batch ends with a few latency-bound kernels (column-sum
    reduction, list evaluation, compaction) that need a fraction of an SM each; on alternating streams they run beside
    the next batch's sweep (B200, 64 pairs at 480x640: 0.97 -> 0.91 ms per batch).  No host synchronisation anywhere:
    results are capacity-sized `CoarseResult`s whose match count stays on the device; call `join()` before reading them
    on another stream.  With `submit(..., fine_level=Matcher.fine_level(device))` each batch also runs the bf16
    FinePreprocess Linears and fine transformer (see `ops.match_pairs_device`), in a fine scratch kept per stream."""

    def __init__(self, device, n_streams: int = 2):
        self.device = torch.device(device)
        self.streams = ([torch.cuda.Stream(device=self.device) for _ in range(n_streams)] if n_streams > 1
                        else [torch.cuda.current_stream(self.device)])
        self.workspaces = [None] * len(self.streams)
        self.fine_workspaces = [None] * len(self.streams)
        self._k = 0
        self._pending = []          # weak references to the results submitted since the last join()

    def fork(self) -> None:
        """the runner's streams wait for everything queued so far on the current stream (inputs being produced there)"""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            if st != cur:
                st.wait_stream(cur)

    def join(self) -> None:
        """the current stream waits for every batch submitted so far; results that are still alive are marked as in use
        on the current stream (`Tensor.record_stream`), so that dropping one while a consumer queued here is still reading
        it cannot hand its memory back to the batch stream's allocator pool early"""
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            if st != cur:
                cur.wait_stream(st)
        for ref, st in self._pending:
            res = ref()
            if res is not None and st != cur:
                for key, v in res.items():
                    if key not in ("workspace", "fine_workspace") and isinstance(v, torch.Tensor) and v.is_cuda:   # (the scratch stays with its stream)
                        v.record_stream(cur)
        self._pending.clear()

    def submit(self, feat_c0, feat_c1, feat_f0, feat_f1, hw0_i, hw0_c, hw1_c, after=None, fine_level=None, **kw):
        """Queues one batch; returns (result, stream it was queued on).  `after(result)` runs inside the batch's stream
        context (e.g. to append the batch's records to a job buffer)."""
        from . import ops
        k = self._k % len(self.streams)
        self._k += 1
        with torch.cuda.stream(self.streams[k]):
            if fine_level is not None:
                kw.update(fine_level=fine_level, fine_workspace=self.fine_workspaces[k])
            res = ops.match_pairs_device(feat_c0, feat_c1, feat_f0, feat_f1, hw0_i, hw0_c, hw1_c,
                                         workspace=self.workspaces[k], **kw)
            self.workspaces[k] = res["workspace"]
            if fine_level is not None:
                self.fine_workspaces[k] = res["fine_workspace"]
            if after is not None:
                after(res)
        if len(self._pending) >= 64:         # callers that never join(): forget the results that are gone
            self._pending = [(r, st) for r, st in self._pending if r() is not None]
        self._pending.append((weakref.ref(res), self.streams[k]))
        return res, self.streams[k]


# ---- multi-GPU sharding -----------------------------------------------------------------------------------------

def shard_range(n_pairs: int, rank: int, world: int):
    """Contiguous block partition of pair indices: rank r owns [lo, hi)."""
    base, rem = divmod(n_pairs, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_matches(local: Dict[str, torch.Tensor], n_pairs: int, rank: int, world: int, group=None,
                   device: Optional[torch.device] = None) -> Optional[Dict[str, torch.Tensor]]:
    """THE one collective of a sharded run: every rank contributes the packed match lists of its pairs
    (`flatten_slots(..., pair_offset=lo)`), rank 0 receives the concatenation, which is sorted by (b, i) because the
    partition is contiguous.  One all_gather of the per-rank totals sizes a single padded all_gather of one packed
    [max_M, 8] fp64-free record tensor (ids as int64, values as float32 bit patterns)."""
    import torch.distributed as dist
    dev = device or local["i_ids"].device
    m = torch.tensor([local["i_ids"].numel()], dtype=torch.int64, device=dev)
    totals = [torch.zeros_like(m) for _ in range(world)]
    dist.all_gather(totals, m, group=group)
    totals = [int(t.item()) for t in totals]
    mx = max(max(totals), 1)
    rec = torch.zeros(mx, 8, dtype=torch.int64, device=dev)
    k = local["i_ids"].numel()
    if k:
        rec[:k, 0] = local["b_ids"].to(dev)
        rec[:k, 1] = local["i_ids"].to(dev)
        rec[:k, 2] = local["j_ids"].to(dev)
        f = torch.cat([local["mconf"][:, None], local["mkpts0_f"], local["mkpts1_f"]], 1).to(dev).contiguous()
        rec[:k, 3:8] = f.view(torch.int32).to(torch.int64)
    bufs = [torch.zeros_like(rec) for _ in range(world)]
    dist.all_gather(bufs, rec, group=group)
    if rank != 0:
        return None
    allrec = torch.cat([b[:t] for b, t in zip(bufs, totals)], 0)
    fl = allrec[:, 3:8].to(torch.int32).view(torch.float32)
    return {"b_ids": allrec[:, 0], "i_ids": allrec[:, 1], "j_ids": allrec[:, 2], "mconf": fl[:, 0],
            "mkpts0_f": fl[:, 1:3], "mkpts1_f": fl[:, 3:5], "per_rank_matches": totals}


def pack_records(res, pair_offset: int, out: Optional[torch.Tensor] = None, base: Optional[torch.Tensor] = None,
                 compact: bool = False) -> torch.Tensor:
    """Capacity-sized result -> packed int32 records; rows past the live count are not written.  One kernel, no host sync.
      compact=False: [cap, 8] = (b_global, i, j, mconf, x0, y0, x1, y1; floats as bit patterns)   (`pope_pack_records`)
      compact=True : [cap, 5] = (b_global, i | j << 16, mconf, x1, y1) -- 20 instead of 32 bytes per match: the keypoint of
                     image 0 is implied by i (`unpack_records` restores it); needs L, S <= 65536  (`pope_pack_records_compact`)
    `base` (device int64[1]): the batch is appended to `out` behind the `base` records already there."""
    cap = res["i_ids"].shape[0]
    dev = res["i_ids"].device
    words = 5 if compact else 8
    if dev.type != "cuda":
        # host-side bookkeeping of already-computed results (the world_size-2 gloo tests of the sharding logic); the
        # records themselves are produced on the GPU in every real run
        head = [(res["b_ids"] + pair_offset).to(torch.int32)[:, None]]
        if compact:
            ij = (res["i_ids"] | (res["j_ids"] << 16)).to(torch.int64)
            ij = torch.where(ij >= 2 ** 31, ij - 2 ** 32, ij).to(torch.int32)
            rec = torch.cat(head + [ij[:, None], res["mconf"].view(torch.int32)[:, None], res["mkpts1_f"].view(torch.int32)], 1)
        else:
            rec = torch.cat(head + [res["i_ids"].to(torch.int32)[:, None], res["j_ids"].to(torch.int32)[:, None],
                                    res["mconf"].view(torch.int32)[:, None], res["mkpts0_f"].view(torch.int32),
                                    res["mkpts1_f"].view(torch.int32)], 1)
        if out is None:
            return rec
        m, b = int(res["counts"][res["n_pairs"]]), (int(base) if base is not None else 0)
        out[b:b + m] = rec[:m]
        return out
    if out is None:
        out = torch.empty(cap, words, dtype=torch.int32, device=dev)
    n = res["n_pairs"]
    base_ptr = None if base is None else base.data_ptr()
    with torch.cuda.device(dev):
        if compact:
            st = _lib.lib().pope_pack_records_compact(res["b_ids"].data_ptr(), res["i_ids"].data_ptr(), res["j_ids"].data_ptr(),
                                                      res["mconf"].data_ptr(), res["mkpts1_f"].contiguous().data_ptr(),
                                                      res["counts"][n:n + 1].data_ptr(), cap, int(pair_offset), out.data_ptr(),
                                                      base_ptr, _lib.stream_ptr(dev))
        else:
            st = _lib.lib().pope_pack_records(res["b_ids"].data_ptr(), res["i_ids"].data_ptr(), res["j_ids"].data_ptr(),
                                              res["mconf"].data_ptr(), res["mkpts0_f"].contiguous().data_ptr(),
                                              res["mkpts1_f"].contiguous().data_ptr(), res["counts"][n:n + 1].data_ptr(), cap,
                                              int(pair_offset), out.data_ptr(), base_ptr, _lib.stream_ptr(dev))
    _lib.check(st, "pope_pack_records")
    return out


def unpack_records(rec: torch.Tensor, w0c: Optional[int] = None, pixel_scale: Optional[float] = None) -> Dict[str, torch.Tensor]:
    """Packed int32 records [M, 8] or [M, 5] (`pack_records`) -> the reference's match-list tensors (ids int64, the rest fp32).
    The compact form needs the width of image 0's coarse grid and hw0_i[0] / hw0_c[0] to restore mkpts0_f from i."""
    if rec.shape[1] == 8:
        fl = rec[:, 3:8].contiguous().view(torch.float32)
        return {"b_ids": rec[:, 0].long(), "i_ids": rec[:, 1].long(), "j_ids": rec[:, 2].long(), "mconf": fl[:, 0],
                "mkpts0_f": fl[:, 1:3], "mkpts1_f": fl[:, 3:5]}
    if w0c is None or pixel_scale is None:
        raise _lib.PopeError("compact records need w0c and pixel_scale to restore mkpts0_f")
    ij = rec[:, 1].long() & 0xFFFFFFFF
    i, j = ij & 0xFFFF, ij >> 16
    fl = rec[:, 2:5].contiguous().view(torch.float32)
    mk0 = torch.stack([(i % w0c).float() * pixel_scale, (i // w0c).float() * pixel_scale], 1)
    return {"b_ids": rec[:, 0].long(), "i_ids": i, "j_ids": j, "mconf": fl[:, 0], "mkpts0_f": mk0, "mkpts1_f": fl[:, 1:3]}


class JobGather:
    """The single cross-GPU step of a sharded job (SURVEY.md section 8(e)): every rank appends the packed records of each
    of its steps behind the previous ones in one device buffer (no sync, no collective, no compaction: the running count
    stays on the device); `finish()` runs once at the end of the job -- one all-gather of the totals (with the job's one
    host read) and ONE collective on the records: a gather to rank 0 (default) or an all-gather (`to_all=True`).

    Nothing is allocated after the constructor: rank 0's receive buffer [world, steps * cap, words] exists from the start
    and the gather lands in views of it (a job's first `finish()` is as fast as any later one).
    `add()` is stream-safe by itself: appends may be issued from different streams (e.g. `DeviceBatchRunner.submit(after=)`
    on alternating streams); each one waits for the previous append's event before it reads the running count, and
    `finish()` waits for the last."""

    def __init__(self, steps: int, cap: int, device, rank: int = 0, world: int = 1, compact: bool = False, to_all: bool = False):
        self.words = 5 if compact else 8
        self.compact, self.rank, self.world, self.to_all = compact, rank, world, to_all
        self.rec = torch.empty(steps * cap, self.words, dtype=torch.int32, device=device)
        self.total = torch.zeros(1, dtype=torch.int64, device=device)
        self.sizes = torch.zeros(max(world, 1), dtype=torch.int64, device=device)
        self.recv = (torch.empty(world, steps * cap, self.words, dtype=torch.int32, device=device)
                     if world > 1 and (rank == 0 or to_all) else None)
        self._last = None                    # event after the most recent append (cuda only)

    def add(self, res, pair_offset: int):
        n = res["n_pairs"]
        cuda = self.rec.device.type == "cuda"
        if cuda:
            cur = torch.cuda.current_stream(self.rec.device)
            if self._last is not None:
                cur.wait_event(self._last)          # the previous append has advanced the count
        pack_records(res, pair_offset, out=self.rec, base=self.total, compact=self.compact)
        self.total += res["counts"][n:n + 1]
        if cuda:
            self._last = torch.cuda.Event()
            self._last.record(cur)

    def finish(self, group=None):
        """Returns (records [world, max_total, words], totals): rank r's records are records[r, :totals[r]], sorted by (b, i)
        within each step.  With the default gather only rank 0 receives the records (the others get None)."""
        import torch.distributed as dist
        if self.rec.device.type == "cuda" and self._last is not None:
            torch.cuda.current_stream(self.rec.device).wait_event(self._last)
            self._last = None
        if self.world == 1:
            mine = int(self.total.item())                       # the job's one host read
            self.total.zero_()
            return self.rec[:mine].unsqueeze(0), [mine]
        dist.all_gather_into_tensor(self.sizes, self.total, group=group)
        sizes = self.sizes.tolist()                             # the job's one host read (every rank's total)
        mx = max(max(sizes), 1)
        send = self.rec[:mx]                                    # rows past the rank's own total are never read
        out = None
        if self.to_all:
            out = self.recv.view(-1, self.words)[:self.world * mx]
            dist.all_gather_into_tensor(out, send, group=group)
            out = out.view(self.world, mx, self.words)
        else:
            parts = [self.recv[r, :mx] for r in range(self.world)] if self.rank == 0 else None
            dist.gather(send, parts, dst=0, group=group)
            if self.rank == 0:
                out = self.recv[:, :mx]
        self.total.zero_()
        return out, sizes

    def checksum(self, records: Optional[torch.Tensor] = None, totals=None) -> torch.Tensor:
        """int64 word sum of the live records: of this rank's own buffer (no arguments; call before `finish()` clears the
        count, or pass the count), or per rank of a gathered [world, max_total, words] tensor -> [world]."""
        if records is None:
            m = int(self.total.item()) if totals is None else int(totals)
            return self.rec[:m].to(torch.int64).sum().reshape(1)
        return torch.stack([records[r, :int(t)].to(torch.int64).sum() for r, t in enumerate(totals)])


def bind_host_to_gpu(device_index: int):
    """Pin this process to the CPUs next to its GPU while it allocates page-locked staging buffers, so that they land
    on the GPU's NUMA node (with 4-8 ranks the host link otherwise saturates on one socket).  Returns the previous
    affinity (restore with os.sched_setaffinity(0, prev)) or None if NVML is unavailable."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {c for c in range(ncpu) if (words[c // 64] >> (c % 64)) & 1}
        prev = os.sched_getaffinity(0)
        cpus &= prev
        if cpus:
            os.sched_setaffinity(0, cpus)
            return prev
    except Exception:
        pass
    return None


def gather_matches_padded(res, n_local: int, rank: int, world: int, group=None):
    """Sync-free form of the single gather for a steady-state loop: every rank contributes its capacity-sized result
    as one packed int32 record tensor [cap, 8] = (b_global, i, j, mconf, x0, y0, x1, y1; floats as bit patterns) plus
    its per-pair counts; two NCCL all-gathers, no host read.  Returns (records [world, cap, 8], counts [world, n+2]);
    rank r's live records are records[r, :counts[r, n]] and are sorted by (b, i)."""
    import torch.distributed as dist
    cap = res["i_ids"].shape[0]
    rec = pack_records(res, rank * n_local)
    out = torch.empty(world * cap, 8, dtype=torch.int32, device=rec.device)
    cnt = torch.empty(world * res["counts"].numel(), dtype=torch.int32, device=rec.device)
    dist.all_gather_into_tensor(out, rec, group=group)
    dist.all_gather_into_tensor(cnt, res["counts"], group=group)
    return out.view(world, cap, 8), cnt.view(world, -1)


def run_sharded(n_pairs: int, rank: int, world: int, local_fn: Callable[[int, int], Dict[str, torch.Tensor]],
                group=None, device: Optional[torch.device] = None):
    """Shard `n_pairs` over `world` ranks, run `local_fn(lo, hi)` (returns packed lists with *global* b_ids) on each,
    gather on rank 0.  No collective runs inside `local_fn`."""
    lo, hi = shard_range(n_pairs, rank, world)
    local = local_fn(lo, hi)
    return gather_matches(local, n_pairs, rank, world, group, device)


# ---- the pair loop of the evaluation scripts (eval_linemod_json.py:103-122, :146-149) ---------------------------------------

def bgr_to_gray(img: torch.Tensor) -> torch.Tensor:
    """cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) for a uint8 [..., H, W, 3] tensor, on the tensor's device: OpenCV's 8-bit
    path (4.x) is the fixed-point sum (B * 3735 + G * 19235 + R * 9798 + 16384) >> 15, reproduced exactly (checked over all
    2^24 colours in tests/test_driver_sharding.py)."""
    if img.dtype != torch.uint8 or img.shape[-1] != 3:
        raise _lib.PopeError("bgr_to_gray takes uint8 images with three channels last")
    x = img.to(torch.int32)
    return ((x[..., 0] * 3735 + x[..., 1] * 19235 + x[..., 2] * 9798 + 16384) >> 15).to(torch.uint8)


def match_crops(matcher, image0: torch.Tensor, crops: Sequence[torch.Tensor], conf_thr: float = 0.9):
    """The reference's per-query loop (eval_linemod_json.py:103-122, :146-149): the query image against each of the
    retrieved crops -- grey conversion, / 255, one Matcher call per crop, `matching_score` = number of matches with
    mconf > 0.9, best crop = first arg-max.  Here crops of equal size go through ONE Matcher call (image0 repeated), and the
    scores and the arg-max are computed on the device (`pope_match_scores`); the only host reads are the ones the Matcher
    itself needs.  image0 / crops: uint8 BGR [H, W, 3] tensors on the matcher's device.
    Returns (per-crop list of dicts with mkpts0_f / mkpts1_f / mconf, scores int32 [n_crops] (device), best int)."""
    from . import ops
    dev = image0.device
    g0 = (bgr_to_gray(image0).float() / 255.0)[None, None]
    results = [None] * len(crops)
    scores = torch.zeros(len(crops), dtype=torch.int32, device=dev)
    by_size = {}
    for k, c in enumerate(crops):
        by_size.setdefault(tuple(c.shape[:2]), []).append(k)
    for size, ks in by_size.items():
        g1 = torch.stack([bgr_to_gray(crops[k]).float() / 255.0 for k in ks])[:, None]
        batch = {"image0": g0.expand(len(ks), -1, -1, -1).contiguous(), "image1": g1}
        with torch.no_grad():
            matcher(batch)
        counts = torch.bincount(batch["b_ids"], minlength=len(ks)).to(torch.int32)
        if batch["mconf"].numel():
            sc, _ = ops.match_scores(batch["mconf"].contiguous(), counts, len(ks), group=len(ks), thr=conf_thr)
        else:
            sc = torch.zeros(len(ks), dtype=torch.int32, device=dev)
        for slot, k in enumerate(ks):
            sel = batch["b_ids"] == slot
            results[k] = {"mkpts0_f": batch["mkpts0_f"][sel], "mkpts1_f": batch["mkpts1_f"][sel], "mconf": batch["mconf"][sel]}
            scores[k] = sc[slot]
    best = int(torch.argmax(scores).item()) if len(crops) else -1        # torch.argmax returns the first maximum, like np.argmax
    return results, scores, best
