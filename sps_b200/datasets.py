"""Host mirror of the offline loader's submap selection (src/sps/datasets/blt_dataset.py).

``BLTDataset.__getitem__`` (blt_dataset.py:209-243) builds one item as::

    kd_tree_scan = cKDTree(scan[:, :3])
    submap_idx   = select_closest_points(kd_tree_scan, kd_tree_target)     # query_ball_tree, r = VOXEL_SIZE
    rows         = vstack([scan xyz | t=1 | label], [map[submap_idx] xyz | t=0 | 1])

Here the map is indexed once on the GPU (a uniform grid of edge r instead of ``kd_tree_target``) and every scan is a
27-cell ball query through the C ABI (``sps_ballmap_build`` / ``sps_submap_ball_query``).  The selection runs in the
library; stacking the selected rows under the scan rows is torch plumbing as in the reference.  ``make_batch`` does
the selection, the stacking and the collation of a whole batch of scans in the library (``sps_radius_batch``).
No CPU fallback."""
from __future__ import annotations

import ctypes as C

import torch

from . import _cabi
from ._cabi import check
from .engine import _ptr, _stream

SCAN_TIMESTAMP, MAP_TIMESTAMP = 1.0, 0.0     # src/sps/datasets/util.py:20-21
MAX_BATCH = 255                               # scans per batch: the batch index is the voxel key's 8-bit b field


def batch_parts(scans, offsets=None, min_width=4):
    """A batch of scans as the library takes it: ``scans`` is a list of per-scan fp32 ``[n_b, >=min_width]`` tensors
    (x, y, z, label, in the map frame; the deployment path has no label and passes ``min_width=3``), or one
    ``[sum n_b, >=min_width]`` tensor with ``offsets`` (``B + 1`` ints, scan b = rows ``offsets[b]:offsets[b+1]``).
    Returns ``(parts, offsets, ld)``: ``parts`` = [(contiguous fp32 tensor, first row)], ``offsets`` a list of B + 1
    ints, ``ld`` the common row width."""
    if isinstance(scans, torch.Tensor):
        if offsets is None:
            raise ValueError("one scan tensor needs the per-scan offsets")
        offsets = [int(o) for o in (offsets.tolist() if isinstance(offsets, torch.Tensor) else offsets)]
        scans = [scans]
        starts = [0]
        if offsets[-1] != scans[0].shape[0]:
            raise ValueError(f"offsets end at {offsets[-1]}, the scan tensor has {scans[0].shape[0]} rows")
    else:
        if offsets is not None:
            raise ValueError("offsets go with one concatenated scan tensor, not with a list of scans")
        offsets = [0]
        for t in scans:
            offsets.append(offsets[-1] + t.shape[0])
        starts = offsets[:-1]
    if not 1 <= len(offsets) - 1 <= MAX_BATCH:
        raise ValueError(f"a batch holds 1..{MAX_BATCH} scans, got {len(offsets) - 1}")
    if offsets[0] != 0 or any(b < a for a, b in zip(offsets, offsets[1:])):
        raise ValueError("offsets must start at 0 and never decrease")
    widths = {t.shape[1] for t in scans if t.dim() == 2}
    if len(widths) != 1 or any(t.dim() != 2 for t in scans) or min(widths) < min_width:
        cols = "x, y, z, label" if min_width >= 4 else "x, y, z"
        raise ValueError(f"scans must be 2-D with one common width >= {min_width} ({cols})")
    parts = [(t.contiguous().float(), s) for t, s in zip(scans, starts)]
    return parts, offsets, widths.pop()


def device_scans(parts, n, ld, device):
    """The scans of :func:`batch_parts` as one device tensor ``[max(n, 1), ld]``: the single part itself when it already
    lives on ``device``, else a new tensor the parts are copied into (on the current stream)."""
    if len(parts) == 1 and parts[0][0].device == device:
        return parts[0][0]
    src = torch.empty((max(n, 1), ld), dtype=torch.float32, device=device)
    for t, start in parts:
        src[start:start + t.shape[0]].copy_(t)
    return src


class RadiusSubmap:
    """The role of ``kd_tree_target`` + ``select_closest_points`` (blt_dataset.py:193,258-271) for one base map.

    ``map_xyz``: CUDA fp32 ``[M, >=3]`` (xyz in the first three columns); ``radius``: ``cfg["MODEL"]["VOXEL_SIZE"]``."""

    def __init__(self, map_xyz: torch.Tensor, radius: float):
        if not map_xyz.is_cuda:
            raise RuntimeError("RadiusSubmap needs the map on a CUDA device (no CPU fallback)")
        self.lib = _cabi.load()
        self.map_xyz = map_xyz[:, :3].contiguous().float()
        self.radius = float(radius)
        n = len(self.map_xyz)
        self._storage = torch.empty(self.lib.sps_ballmap_bytes(n) + 256, dtype=torch.uint8, device=map_xyz.device)
        base = (self._storage.data_ptr() + 255) & ~255
        self.handle = C.c_void_p()
        check(self.lib.sps_ballmap_build(C.byref(self.handle), C.c_void_p(base), self.lib.sps_ballmap_bytes(n),
                                         _ptr(self.map_xyz), n, self.radius, _stream()), "sps_ballmap_build")

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            self.lib.sps_ballmap_destroy(h)

    def select_closest_points(self, scan_xyz: torch.Tensor, return_offsets: bool = False):
        """Indices into the map, scan point by scan point, duplicates kept (``merged_indexes``, blt_dataset.py:262-267).
        One host synchronisation (the number of hits sizes the result, as ``np.concatenate`` does in the reference)."""
        if not scan_xyz.is_cuda:
            raise RuntimeError("select_closest_points needs the scan on a CUDA device (no CPU fallback)")
        scan = scan_xyz[:, :3].contiguous().float()
        n = len(scan)
        dev = scan.device
        scratch = torch.empty(self.lib.sps_ball_query_scratch_bytes(n) + 256, dtype=torch.uint8, device=dev)
        sbase = (scratch.data_ptr() + 255) & ~255
        offsets = torch.empty(n + 1, dtype=torch.int32, device=dev)
        total = torch.zeros(1, dtype=torch.int32, device=dev)
        cap = max(4 * n, 1024)
        while True:
            out = torch.empty(cap, dtype=torch.int32, device=dev)
            check(self.lib.sps_submap_ball_query(self.handle, _ptr(scan), n, _ptr(offsets), _ptr(out), cap, _ptr(total),
                                                 C.c_void_p(sbase), self.lib.sps_ball_query_scratch_bytes(n), _stream()),
                  "sps_submap_ball_query")
            m = int(total.item())
            if m <= cap:
                break
            cap = m                                     # second pass with the exact size
        idx = out[:m].long()
        return (idx, offsets) if return_offsets else idx

    def make_item(self, scan: torch.Tensor) -> torch.Tensor:
        """``BLTDataset.__getitem__`` without augmentation: ``scan`` ``[N, 4]`` = x, y, z, label ->
        rows ``[N + M, 5]`` = x, y, z, t, label (scan rows t = 1 first, submap rows t = 0, label 1)."""
        idx = self.select_closest_points(scan)
        sub = self.map_xyz[idx]
        ones = torch.ones(len(sub), 1, dtype=torch.float32, device=scan.device)
        scan_rows = torch.hstack([scan[:, :3].float(), torch.full((len(scan), 1), SCAN_TIMESTAMP, device=scan.device),
                                  scan[:, 3:4].float()])
        sub_rows = torch.hstack([sub, ones * MAP_TIMESTAMP, ones])
        return torch.vstack([scan_rows, sub_rows])

    def make_batch(self, scans, offsets=None, return_offsets: bool = False):
        """``BLTDataset.__getitem__`` (no augmentation) for every scan of a batch + ``collate_fn`` (blt_dataset.py:173-182)
        in the library: device rows ``[N, 6]`` = b, x, y, z, t, label; for each scan its rows (t = 1, its label), then
        its submap rows (t = 0, label 1) -- bit-identical to ``vstack([hstack([b, make_item(scan_b)]) for b])``.
        ``scans``/``offsets`` as in :func:`batch_parts`.  One host synchronisation (the number of rows sizes the
        result).  ``return_offsets``: also the int32 ``[B + 1]`` row offsets of the scans."""
        parts, offs, ld = batch_parts(scans, offsets)
        dev = self.map_xyz.device
        n, batch = offs[-1], len(offs) - 1
        src = device_scans(parts, n, ld, dev)
        nbytes = self.lib.sps_radius_batch_scratch_bytes(n, batch)
        scratch = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
        sbase = (scratch.data_ptr() + 255) & ~255
        row_offsets = torch.empty(batch + 1, dtype=torch.int32, device=dev)
        n_rows = torch.zeros(1, dtype=torch.int32, device=dev)
        h_off = (C.c_int64 * (batch + 1))(*offs)
        cap = 6 * n + 1024
        with torch.cuda.device(dev):
            while True:
                rows = torch.empty((cap, 6), dtype=torch.float32, device=dev)
                check(self.lib.sps_radius_batch(self.handle, _ptr(src), ld, h_off, batch, _ptr(rows), cap, _ptr(row_offsets),
                                                _ptr(n_rows), C.c_void_p(sbase), nbytes, _stream()), "sps_radius_batch")
                m = int(n_rows.item())
                if m <= cap:
                    break
                cap = m                                     # second pass with the exact size
        return (rows[:m], row_offsets) if return_offsets else rows[:m]
