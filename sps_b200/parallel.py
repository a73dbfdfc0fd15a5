"""Scan-sharded multi-GPU inference (BASELINE.json configs[3], SURVEY.md §8e).

Scans are independent units (a fresh coordinate manager per forward, src/sps/models/models.py:24),
so rank r takes scan ids ``r::world`` with the weights (and the base-map hash) replicated; the
only collective is the gather of predictions and metric partials at the end -- no collective
inside the forward.  Works with the ``nccl`` backend (CUDA tensors, NVLink/NVSwitch) and with
``gloo`` (CPU tensors; used by the CPU-side tests of this host logic).
"""
from __future__ import annotations

from typing import Callable, Iterable, Sequence

import numpy as np
import torch
import torch.distributed as dist


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
