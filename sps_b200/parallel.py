"""Scan-sharded multi-GPU inference (BASELINE.json configs[3], SURVEY.md §8e).

Scans are independent units (a fresh coordinate manager per forward, src/sps/models/models.py:24),
so rank r takes scan ids ``r::world`` with the weights (and the base-map hash) replicated; the
only collective is the gather of predictions and metric partials at the end -- no collective
inside the forward.  Works with the ``nccl`` backend (CUDA tensors, NVLink/NVSwitch) and with
``gloo`` (CPU tensors; used by the CPU-side tests of this host logic).
"""
from __future__ import annotations

from typing import Callable, Iterable, NamedTuple, Sequence

import numpy as np
import torch
import torch.distributed as dist

from ._cabi import SPS_ERR_CAPACITY, SpsError


def shard_ids(n_items: int, rank: int, world: int) -> list[int]:
    """Scan ids owned by ``rank``: r, r+W, r+2W, ..."""
    return list(range(rank, n_items, world))


def _world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def gather_scores(local_scores: Sequence[torch.Tensor], ids: Sequence[int], n_items: int, max_points: int):
    """All-gather per-scan score vectors, padded to ``max_points`` (fp32 [B, max_points] + int32
    lengths): ~0.26 MB per 65k-point scan, far below NVLink time.  Returns on every rank a list of
    ``n_items`` 1-D tensors in scan-id order."""
    rank, world = _world()
    device = local_scores[0].device if len(local_scores) else torch.device("cpu")
    per_rank = (n_items + world - 1) // world
    buf = torch.zeros((per_rank, max_points), dtype=torch.float32, device=device)
    lens = torch.zeros(per_rank, dtype=torch.int32, device=device)
    for j, s in enumerate(local_scores):
        buf[j, : len(s)] = s
        lens[j] = len(s)
    if world > 1:
        all_buf = [torch.empty_like(buf) for _ in range(world)]
        all_len = [torch.empty_like(lens) for _ in range(world)]
        dist.all_gather(all_buf, buf)
        dist.all_gather(all_len, lens)
    else:
        all_buf, all_len = [buf], [lens]
    out = [None] * n_items
    for r in range(world):
        for j, i in enumerate(shard_ids(n_items, r, world)):
            out[i] = all_buf[r][j, : int(all_len[r][j])]
    return out


def gather_partials(counts: torch.Tensor, sums: torch.Tensor, n_items: int):
    """counts int64 [B_local,4] (TP,TN,FP,FN), sums float64 [B_local,5] per local scan ->
    (counts [n_items,4], sums [n_items,5]) in scan-id order on every rank."""
    rank, world = _world()
    per_rank = (n_items + world - 1) // world
    c = torch.zeros((per_rank, 4), dtype=torch.int64, device=counts.device)
    s = torch.zeros((per_rank, 5), dtype=torch.float64, device=sums.device)
    c[: len(counts)] = counts
    s[: len(sums)] = sums
    if world > 1:
        ac = [torch.empty_like(c) for _ in range(world)]
        as_ = [torch.empty_like(s) for _ in range(world)]
        dist.all_gather(ac, c)
        dist.all_gather(as_, s)
    else:
        ac, as_ = [c], [s]
    oc = torch.zeros((n_items, 4), dtype=torch.int64)
    os_ = torch.zeros((n_items, 5), dtype=torch.float64)
    for r in range(world):
        for j, i in enumerate(shard_ids(n_items, r, world)):
            oc[i] = ac[r][j].cpu()
            os_[i] = as_[r][j].cpu()
    return oc, os_


def per_scan_metrics(counts: torch.Tensor, sums: torch.Tensor) -> dict:
    """The values ``SPSNet.predict_step`` appends for each scan (models.py:84-104, util.py:285-299), from its partials:
    {metric: [value per scan]}; scans without points are skipped."""
    out = {"Loss": [], "R2": [], "dIoU": [], "Precision": [], "Recall": [], "F1": []}
    for (tp, tn, fp, fn), (n, sse, sl, sll, _ss) in zip(counts.tolist(), sums.tolist()):
        if n == 0:
            continue
        precision = tp / (tp + fp) if (tp + fp) != 0 else 0
        recall = tp / (tp + fn) if (tp + fn) != 0 else 0
        f1 = 2 * (precision * recall) / (precision + recall) if (precision + recall) != 0 else 0
        diou = tp / (tp + fn + fp) if (tp + fn + fp) != 0 else float("nan")
        ss_tot = sll - sl * sl / n
        out["Loss"].append(sse / n)
        out["R2"].append(1.0 - sse / ss_tot if ss_tot > 0 else 0.0)
        out["dIoU"].append(diou)
        out["Precision"].append(precision)
        out["Recall"].append(recall)
        out["F1"].append(f1)
    return out


def metrics_from_partials(counts: torch.Tensor, sums: torch.Tensor) -> dict:
    """scripts/predict.py:70-83 semantics: every metric is the MEAN over per-scan values (not pooled
    counts); per-scan formulas from util.py:285-299 and models.py:91-92."""
    return {k: float(np.mean(v)) for k, v in per_scan_metrics(counts, sums).items() if len(v)}


def device_partials(scores: torch.Tensor, rows: torch.Tensor, eps: float):
    """Metric partials of one scan on the GPU (library kernel, no torch arithmetic)."""
    import ctypes as C
    from . import _cabi
    from .engine import _ptr, _stream
    lib = _cabi.load()
    counts = torch.empty(4, dtype=torch.int64, device=scores.device)
    sums = torch.empty(5, dtype=torch.float64, device=scores.device)
    _cabi.check(lib.sps_confusion_counts(_ptr(scores), _ptr(rows), rows.stride(0), rows.shape[0], -1.0, float(eps),
                                         _ptr(counts), _ptr(sums), _stream()), "sps_confusion_counts")
    return counts, sums


class ShardedPredictor:
    """``predict.py`` over a list of scans, sharded by scan id across the ranks of the default
    process group.  ``score_fn(rows[N,6]) -> scores[N]`` is ``SPSNet.forward`` on a GPU rank;
    ``partials_fn(scores, rows, eps) -> (counts[4], sums[5])`` defaults to the library kernel."""

    def __init__(self, score_fn: Callable, eps: float, partials_fn: Callable | None = None):
        self.score_fn, self.eps = score_fn, float(eps)
        self.partials_fn = partials_fn or device_partials

    def predict(self, scans: Sequence, max_points: int | None = None, gather_predictions=True):
        rank, world = _world()
        ids = shard_ids(len(scans), rank, world)
        scores, counts, sums = [], [], []
        for i in ids:
            rows = scans[i]() if callable(scans[i]) else scans[i]
            s = self.score_fn(rows)
            c, q = self.partials_fn(s, rows, self.eps)
            scan_mask = rows[:, 4] == 1
            scores.append(s[scan_mask])
            counts.append(c)
            sums.append(q)
        dev = scores[0].device if scores else torch.device("cpu")
        counts = torch.stack(counts) if counts else torch.zeros((0, 4), dtype=torch.int64, device=dev)
        sums = torch.stack(sums) if sums else torch.zeros((0, 5), dtype=torch.float64, device=dev)
        all_counts, all_sums = gather_partials(counts, sums, len(scans))
        result = {"metrics": metrics_from_partials(all_counts, all_sums), "counts": all_counts, "sums": all_sums}
        if gather_predictions:
            if max_points is None:
                m = torch.tensor([max([len(s) for s in scores] + [1])], device=dev)
                if world > 1:
                    dist.all_reduce(m, op=dist.ReduceOp.MAX)
                max_points = int(m.item())
            result["scores"] = gather_scores(scores, ids, len(scans), max_points)
        return result


# ---------------------------------------------------------------------------------------------------------------------
# Sharding the batched calls (SPSModel.predict_radius_async / filter_scans_async) over the ranks, by batch.
# ---------------------------------------------------------------------------------------------------------------------
class ShardPlan:
    """Which rank runs which batch of a sequence and where its results go, from the scan lengths alone: every rank
    computes the same plan without communicating.  Batch k holds scans ``[kB, min((k+1)B, S))`` and runs on rank
    ``k mod W``.  A rank keeps its batches' scan rows back to back (``row_start``: where batch k's first row goes, in its
    rank's buffer) and their scans back to back (``slot_start``); ``cap`` and ``slots`` are the largest such row and
    scan count over the ranks, i.e. the per-rank block of the gathered buffers."""

    def __init__(self, sizes: Sequence[int], batch: int, world: int):
        S, B = len(sizes), int(batch)
        self.world = world
        self.bounds = [(a, min(a + B, S)) for a in range(0, S, B)]
        self.owner = [k % world for k in range(len(self.bounds))]
        self.rows = [int(sum(sizes[a:b])) for a, b in self.bounds]
        self.row_start, self.slot_start = [], []
        rows_of, slots_of = [0] * world, [0] * world
        for k, (a, b) in enumerate(self.bounds):
            r = self.owner[k]
            self.row_start.append(rows_of[r])
            self.slot_start.append(slots_of[r])
            rows_of[r] += self.rows[k]
            slots_of[r] += b - a
        self.cap, self.slots = max(rows_of), max(slots_of)
        # scan i of the sequence -> its row in the gathered [W * slots] per-scan arrays
        self.scan_index = [self.owner[k] * self.slots + self.slot_start[k] + i - a
                           for k, (a, b) in enumerate(self.bounds) for i in range(a, b)]

    def batches(self, rank: int) -> list[int]:
        return [k for k in range(len(self.bounds)) if self.owner[k] == rank]


class ShardedResult(NamedTuple):
    """Results of :class:`ShardedScans`' calls.  The per-scan arrays reach every rank; ``scan_scores``, ``kept`` and
    ``kept_offsets`` reach rank 0 only (None on the other ranks).  ``kept``, ``kept_offsets`` and ``counts`` are None
    for ``evaluate``."""
    scan_scores: torch.Tensor | None    # fp32 [sum n]: the scan points' scores, in sequence order
    kept: torch.Tensor | None           # fp32 [K, 4]: the published rows of every scan, end to end
    kept_offsets: torch.Tensor | None   # int32 [S + 1]: scan i's published rows are kept[kept_offsets[i]:kept_offsets[i+1]]
    counts: torch.Tensor | None         # int32 [S, 2]: MapHash.crop_voxel's (len(submap), n_unique_scan_voxels) per scan
    metric_counts: torch.Tensor         # int64 [S, 4]: per-scan confusion counts (device_partials' layout)
    metric_sums: torch.Tensor           # float64 [S, 5]: per-scan sums (device_partials' layout)
    metrics: dict                       # metrics_from_partials(metric_counts, metric_sums)


def _scan_sizes(scans, what):
    if isinstance(scans, torch.Tensor) or len(scans) == 0:
        raise ValueError(f"{what} takes a non-empty list of per-scan tensors")
    if any(not isinstance(t, torch.Tensor) or t.dim() != 2 or t.shape[1] < 4 for t in scans):
        raise ValueError(f"{what}: every scan must be a 2-D tensor with at least 4 columns")
    return [int(t.shape[0]) for t in scans]


def _read_on(stream, *tensors):
    """The lane buffers a copy on ``stream`` reads: the lane's next call may replace a buffer that is too small
    (``models._lane_buffers``) before that copy has run, so the caching allocator must not hand the old block out again
    until ``stream`` has passed this point."""
    for t in tensors:
        t.record_stream(stream)


def gather_segments(src: torch.Tensor, ranks, starts, max_rows, lengths: torch.Tensor, out: torch.Tensor,
                    out_offsets: torch.Tensor):
    """``sps_gather_segments`` on the current stream: ``src`` fp32 ``[W, cap, w]`` (or ``[W, cap]``), segment s = rows
    ``starts[s] .. starts[s] + lengths[s]`` of block ``ranks[s]`` (host ints; ``lengths`` a device int32 tensor, clamped
    to ``0 .. max_rows[s]``), concatenated into ``out`` (fp32 ``[>= sum max_rows, w]``) in segment order;
    ``out_offsets`` int32 ``[len(ranks) + 1]`` receives where each segment starts.  All four tensors are contiguous and
    live on one CUDA device."""
    import ctypes as C
    from . import _cabi
    from .engine import _ptr, _stream
    n = len(ranks)
    if not len(starts) == len(max_rows) == n:
        raise ValueError("ranks, starts and max_rows need one entry per segment")
    if src.dim() not in (2, 3) or out.dim() != src.dim() - 1 or (src.dim() == 3 and out.shape[1:] != src.shape[2:]):
        raise ValueError(f"src [W, cap] or [W, cap, w] with out [rows] or [rows, w], got {tuple(src.shape)} and "
                         f"{tuple(out.shape)}")
    for name, t, dtype, numel in (("src", src, torch.float32, None), ("out", out, torch.float32, None),
                                  ("lengths", lengths, torch.int32, n), ("out_offsets", out_offsets, torch.int32, n + 1)):
        if t.dtype != dtype or not t.is_contiguous() or not t.is_cuda or t.device != src.device:
            raise ValueError(f"{name} must be a contiguous {dtype} tensor on the device of src ({src.device}), got "
                             f"{t.dtype} on {t.device}{'' if t.is_contiguous() else ', not contiguous'}")
        if numel is not None and t.numel() < numel:
            raise ValueError(f"{name} needs {numel} entries, got {t.numel()}")
    lib = _cabi.load()
    width = src.shape[2] if src.dim() == 3 else 1
    h_rank = (C.c_int32 * max(n, 1))(*ranks)
    h_start, h_rows = (C.c_int64 * max(n, 1))(*starts), (C.c_int64 * max(n, 1))(*max_rows)
    _cabi.check(lib.sps_gather_segments(_ptr(src), src.shape[0], src.shape[1], width, n, h_rank, h_start, h_rows,
                                        _ptr(lengths), _ptr(out), out.shape[0], _ptr(out_offsets), _stream(src.device)),
                "sps_gather_segments")


class ShardedScans:
    """A whole sequence of scans through ``model``'s batched calls, sharded across the ranks of the default process
    group (or one process without one).  Every rank passes the same full list of scans and runs only its own batches:
    batch k (scans ``[kB, min((k+1)B, S))``) on rank ``k mod W`` (:class:`ShardPlan`).  Each call is the call a single
    process makes on that batch, so the results are bit-identical to the single-GPU loop over the batches (the float64
    metric sums, which each call accumulates with atomics, to their rounding).  ``replay`` is so for any world size.
    ``evaluate`` is so for any world size with the shape sort always on (``engine.set_defaults(pattern_sort=2)`` before
    the model's lanes exist): in the default mode a radius call sorts when its lane holds >= 400 000 rows, and how large
    a lane has grown depends on the calls it served before, which differ between world sizes.  Up to ``model.lanes``
    calls are in flight; each call's results are copied into rank-local buffers on its lane's stream, with no host
    synchronisation per call.  After the last call, one collective per kind of output: the per-scan partials (and
    counts) to every rank, the scan scores (and the published rows) to rank 0.  An error of one rank's calls (a
    coordinate outside the voxel-key range) travels with the partials and raises :class:`SpsError` on every rank before
    the gathers to rank 0.  ``gather_events`` holds
    the CUDA events around that last phase of the latest call; on rank 0 ``batch_offsets`` (int32 ``[n_batches + 1]``)
    holds where each batch's rows start in its last reassembled output (the published rows of ``replay``, the scan
    scores of ``evaluate``)."""

    def __init__(self, model, eps: float, batch: int):
        if not 1 <= int(batch) <= 255:
            raise ValueError(f"a batch holds 1..255 scans, got {batch}")
        self.model, self.eps, self.batch = model, float(eps), int(batch)
        self.gather_events = self.batch_offsets = None

    def _device(self):
        device = next(self.model.MinkUNet.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("move the model to a CUDA device first: sps_b200 has no CPU path")
        return device

    def evaluate(self, scans, submap) -> ShardedResult:
        """``SPSModel.predict_radius_async`` over the sequence: ``scans`` per-scan fp32 ``[n_b, >=4]`` (x, y, z, label in
        the map frame; host or device), ``submap`` a :class:`sps_b200.datasets.RadiusSubmap` each rank builds from the
        same map points.  A batch whose rows did not fit its lane runs again at the end with lanes of its true row count,
        as ``result()`` of the single call does."""
        plan = ShardPlan(_scan_sizes(scans, "evaluate"), self.batch, _world()[1])
        return self._run(plan, lambda a, b: self.model.predict_radius_async(scans[a:b], submap, self.eps), 9,
                         self._keep_radius, rerun=lambda a, b: self.model.predict_radius_async(scans[a:b], submap,
                                                                                               self.eps).result())

    def replay(self, scans, poses, map_hash) -> ShardedResult:
        """``SPSModel.filter_scans_async`` over the sequence: ``scans`` per-scan fp32 ``[n_b, >=4]`` (sensor-frame x, y,
        z, intensity; host or device), ``poses`` float64 ``[S, 4, 4]`` (numpy or tensor, host or device), ``map_hash`` a
        :class:`sps_b200.engine.MapHash` each rank builds from the same map points."""
        sizes = _scan_sizes(scans, "replay")
        poses = poses if isinstance(poses, torch.Tensor) else torch.as_tensor(np.asarray(poses))
        if poses.dtype != torch.float64 or tuple(poses.shape) != (len(sizes), 4, 4):
            raise ValueError(f"poses must be float64 [{len(sizes)}, 4, 4] (one matrix per scan), got {poses.dtype} "
                             f"{tuple(poses.shape)}")
        plan = ShardPlan(sizes, self.batch, _world()[1])
        return self._run(plan, lambda a, b: self.model.filter_scans_async(scans[a:b], poses[a:b], map_hash, self.eps), 12,
                         self._keep_filter)

    # per-scan int64 columns of the rank-local partials: metric counts (4), metric sums (5, float64 bits), and for
    # replay the crop counts (2) and the published row count (1); then one column of this rank's error code
    @staticmethod
    def _keep_radius(h, k, plan, bufs):
        scores, counts, sums = h.device_out
        r0, s0, nb = plan.row_start[k], plan.slot_start[k], counts.shape[0]
        bufs["scores"][r0:r0 + scores.shape[0]].copy_(scores)
        bufs["small"][s0:s0 + nb, :4].copy_(counts)
        bufs["small"][s0:s0 + nb, 4:9].copy_(sums.view(torch.int64))
        bufs["n_rows"][k:k + 1].copy_(h.device_n_rows)
        _read_on(h.stream, scores, counts, sums, h.device_n_rows)

    @staticmethod
    def _keep_filter(h, k, plan, bufs):
        out = h.device_out
        r0, s0, n, nb = plan.row_start[k], plan.slot_start[k], out.scan_scores.shape[0], out.counts.shape[0]
        bufs["scores"][r0:r0 + n].copy_(out.scan_scores)
        bufs["rows"][r0:r0 + n].copy_(out.kept)          # all n rows: how many are published is known on the device only
        small = bufs["small"][s0:s0 + nb]
        small[:, :4].copy_(out.metric_counts)
        small[:, 4:9].copy_(out.metric_sums.view(torch.int64))
        small[:, 9:11].copy_(out.counts)
        small[:, 11].copy_(out.kept_offsets[1:] - out.kept_offsets[:-1])
        _read_on(h.stream, *out)

    def _run(self, plan, call, width, keep, rerun=None) -> ShardedResult:
        rank, world = _world()
        device = self._device()
        replay = width == 12
        S, cap = len(plan.scan_index), max(plan.cap, 1)
        with torch.cuda.device(device):
            bufs = {"scores": torch.empty(cap, dtype=torch.float32, device=device),
                    "small": torch.zeros((max(plan.slots, 1), width + 1), dtype=torch.int64, device=device),
                    "n_rows": torch.zeros(len(plan.bounds), dtype=torch.int32, device=device)}
            if replay:
                bufs["rows"] = torch.empty((cap, 4), dtype=torch.float32, device=device)
            # the host-known index arrays of the last phase, on the device before the first call
            scan_index = torch.as_tensor(plan.scan_index, dtype=torch.int64).to(device)
            batch_rows = torch.as_tensor(plan.rows, dtype=torch.int32).to(device)
            firsts, ends = (torch.as_tensor([ab[j] for ab in plan.bounds], dtype=torch.int64).to(device) for j in (0, 1))
            mine, caps, streams = plan.batches(rank), {}, []
            for k in mine:
                h = call(*plan.bounds[k])
                with torch.cuda.stream(h.stream):
                    keep(h, k, plan, bufs)
                caps[k] = getattr(h, "row_capacity", 0)
                if all(h.stream is not s for s in streams):
                    streams.append(h.stream)
            current = torch.cuda.current_stream(device)
            for s in streams:
                current.wait_stream(s)
            error = None
            try:
                if rerun is not None and mine:
                    self._rerun_overflows(plan, mine, caps, bufs, rerun)
                self.model.check()                  # a coordinate outside the voxel-key range raises here
            except SpsError as e:
                error = e
            if world == 1 and error is not None:
                raise error
            start = torch.cuda.Event(enable_timing=True)
            start.record(current)
            small = bufs["small"]
            if world > 1:
                # the error code travels with the partials, so that every rank raises instead of the others waiting in
                # the gathers to rank 0 for a rank that left
                small[:, width].fill_(error.code if error is not None else 0)
                all_small = torch.empty((world * small.shape[0], width + 1), dtype=torch.int64, device=device)
                dist.all_gather_into_tensor(all_small, small)
                small = all_small
                code = int(small[:, width].max())
                if error is not None:
                    raise error
                if code:
                    raise SpsError(code, "ShardedScans (a batch of another rank)")
            seq = small.index_select(0, scan_index)
            metric_counts = seq[:, :4].contiguous()
            metric_sums = seq[:, 4:9].contiguous().view(torch.float64)
            counts = seq[:, 9:11].to(torch.int32) if replay else None
            scores = self._to_rank0(bufs["scores"], rank, world)
            rows = self._to_rank0(bufs["rows"], rank, world) if replay else None
            scan_scores = kept = kept_offsets = None
            if rank == 0:
                n_total = sum(plan.rows)
                segments = (plan.owner, plan.row_start, plan.rows)
                self.batch_offsets = torch.empty(len(plan.bounds) + 1, dtype=torch.int32, device=device)
                scan_scores = torch.empty(max(n_total, 1), dtype=torch.float32, device=device)
                gather_segments(scores, *segments, batch_rows, scan_scores, self.batch_offsets)
                scan_scores = scan_scores[:n_total]
                if replay:
                    kept_offsets = torch.zeros(S + 1, dtype=torch.int32, device=device)
                    kept_offsets[1:] = torch.cumsum(seq[:, 11], 0)
                    kept = torch.empty((max(n_total, 1), 4), dtype=torch.float32, device=device)
                    gather_segments(rows, *segments, kept_offsets[ends] - kept_offsets[firsts], kept, self.batch_offsets)
            end = torch.cuda.Event(enable_timing=True)
            end.record(current)
            self.gather_events = (start, end)
            if kept is not None:
                kept = kept[:int(kept_offsets[-1])]
        return ShardedResult(scan_scores, kept, kept_offsets, counts, metric_counts, metric_sums,
                             metrics_from_partials(metric_counts.cpu(), metric_sums.cpu()))

    def _rerun_overflows(self, plan, mine, caps, bufs, rerun):
        """Batches whose rows did not fit their lane's context (nothing of them was scored): run each once more, as
        ``_PendingRadius.result()`` does, and put its results in place.  One host synchronisation for all calls."""
        n_rows = bufs["n_rows"].cpu().tolist()
        over = [k for k in mine if n_rows[k] > caps[k]]
        if not over:
            return
        for eng in self.model._engines():
            try:
                eng.status()
            except SpsError as e:
                if e.code != SPS_ERR_CAPACITY:
                    raise
        for k in over:
            scores, counts, sums = rerun(*plan.bounds[k])
            r0, s0, nb = plan.row_start[k], plan.slot_start[k], counts.shape[0]
            bufs["scores"][r0:r0 + scores.shape[0]].copy_(scores)
            bufs["small"][s0:s0 + nb, :4].copy_(counts)
            bufs["small"][s0:s0 + nb, 4:9].copy_(sums.view(torch.int64))

    @staticmethod
    def _to_rank0(buf, rank, world):
        """``dist.gather`` of every rank's ``buf`` into one ``[W, *buf.shape]`` tensor on rank 0 (None elsewhere)."""
        if world == 1:
            return buf[None]
        out = torch.empty((world,) + tuple(buf.shape), dtype=buf.dtype, device=buf.device) if rank == 0 else None
        dist.gather(buf, list(out.unbind(0)) if rank == 0 else None, dst=0)
        return out
