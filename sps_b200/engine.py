"""Host-side engine: owns the device workspace (a torch tensor), the coordinate-manager context
and the packed network, and forwards everything to the C ABI.  PyTorch is used for device
memory and streams only -- no arithmetic of the hot path happens in torch."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _cabi
from ._cabi import check


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream(device=None) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


# Host-side defaults for NEW engines (the C library itself keeps no process-wide state: every setting lives in a
# context, see include/sps_b200.h).  conv_backend: 0 auto / 1 exact fp32 / 2 TF32 on fp32 rows / 3 fp16 rows.
DEFAULTS = {"conv_backend": 0, "pattern_sort": 1}


def set_defaults(conv_backend=None, pattern_sort=None):
    """Arithmetic / processing-order mode that engines created from now on start with."""
    if conv_backend is not None:
        if conv_backend not in (0, 1, 2, 3):
            raise ValueError("conv_backend must be 0 (auto), 1 (fp32), 2 (tf32) or 3 (fp16)")
        DEFAULTS["conv_backend"] = int(conv_backend)
    if pattern_sort is not None:
        if pattern_sort not in (0, 1, 2):
            raise ValueError("pattern_sort must be 0, 1 or 2")
        DEFAULTS["pattern_sort"] = int(pattern_sort)


def _on_device(fn):
    """Run a method with ``self.device`` current: the C calls enqueue on that device's current stream."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapper


def norm_device(device) -> torch.device:
    d = torch.device(device)
    if d.type == "cuda" and d.index is None:
        d = torch.device("cuda", torch.cuda.current_device())
    return d


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: sps_b200 has no CPU path")


class Net:
    """BN-folded, packed ``CustomMinkUNet(1,1,D=4)`` weights on the device (sps_net)."""

    def __init__(self, state_dict, device="cuda", output_channel=0, apply_sigmoid=True):
        """``output_channel`` / ``apply_sigmoid``: which column of ``final`` the forward returns and whether
        the sigmoid is applied (SPSModel: 0, True; MOS4DNet: 2, False)."""
        self.lib = _cabi.load()
        self.device = norm_device(device)
        h = C.c_void_p()
        check(self.lib.sps_net_create(C.byref(h)), "sps_net_create")
        self.handle = h
        self._keep = []
        for name, value in state_dict.items():
            if name.endswith("num_batches_tracked"):
                continue
            arr = value.detach().cpu().numpy() if isinstance(value, torch.Tensor) else np.asarray(value)
            arr = np.ascontiguousarray(arr, dtype=np.float32)
            check(self.lib.sps_net_set_tensor(h, name.encode(), arr.ctypes.data_as(C.c_void_p), arr.size),
                  f"sps_net_set_tensor({name})")
        check(self.lib.sps_net_set_output(h, int(output_channel), int(bool(apply_sigmoid))), "sps_net_set_output")
        nbytes = self.lib.sps_net_device_bytes()
        with torch.cuda.device(self.device):
            self.storage = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            check(self.lib.sps_net_finalize(h, _ptr(self.storage), nbytes, _stream()), "sps_net_finalize")

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.sps_net_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Engine:
    """One coordinate-manager context (sps_ctx) sized for ``max_points`` input rows."""

    def __init__(self, max_points: int, device="cuda"):
        self.lib = _cabi.load()
        if torch.device(device).type != "cuda":
            raise RuntimeError("sps_b200.Engine needs a CUDA device (no CPU fallback exists)")
        self.device = norm_device(device)
        self.max_points = int(max_points)
        nbytes = self.lib.sps_workspace_bytes(self.max_points)
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            h = C.c_void_p()
            check(self.lib.sps_ctx_create(C.byref(h), _ptr(self.workspace), nbytes, self.max_points), "sps_ctx_create")
        self.handle = h
        self.n = 0
        self.conv_backend = self.pattern_sort = None
        self.set_conv_backend(DEFAULTS["conv_backend"])
        self.set_pattern_sort(DEFAULTS["pattern_sort"])

    def set_conv_backend(self, backend: int):
        """0 auto (tcgen05 on fp16 rows + fp32 FMA kernels for the 8-channel layers), 1 exact fp32 CUDA cores,
        2 TF32 operands on fp32 rows, 3 = 0 (sps_ctx_set_conv_backend)."""
        check(self.lib.sps_ctx_set_conv_backend(self.handle, int(backend)), "sps_ctx_set_conv_backend")
        self.conv_backend = int(backend)

    def set_pattern_sort(self, mode: int):
        check(self.lib.sps_ctx_set_pattern_sort(self.handle, int(mode)), "sps_ctx_set_pattern_sort")
        self.pattern_sort = int(mode)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.sps_ctx_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # ---- coordinate maps -------------------------------------------------------------
    @_on_device
    def voxelize(self, points: torch.Tensor, voxel_size: float):
        _require_cuda(points, "points")
        assert points.dtype == torch.float32 and points.dim() == 2 and points.stride(1) == 1
        self._points = points  # keep alive until the stream is done with it
        self.n = points.shape[0]
        check(self.lib.sps_voxelize(self.handle, _ptr(points), self.n, points.stride(0), float(voxel_size), _stream()),
              "sps_voxelize")

    @_on_device
    def build_maps(self):
        check(self.lib.sps_build_maps(self.handle, _stream()), "sps_build_maps")

    @_on_device
    def status(self):
        check(self.lib.sps_ctx_status(self.handle, _stream()), "sps_ctx_status")

    def level(self, L: int) -> _cabi.LevelView:
        v = _cabi.LevelView()
        check(self.lib.sps_ctx_level(self.handle, L, C.byref(v)), "sps_ctx_level")
        return v

    @_on_device
    def _read(self, ptr, count, dtype):
        out = np.empty(count, dtype=dtype)
        if count:
            check(self.lib.sps_memcpy_d2h(out.ctypes.data_as(C.c_void_p), C.c_void_p(ptr), out.nbytes, _stream()),
                  "sps_memcpy_d2h")
        return out

    def count(self, L: int) -> int:
        return int(self._read(self.level(L).count, 1, np.int32)[0])

    @_on_device
    def coords(self, L: int) -> np.ndarray:
        """int32 [V_L, 5] rows (b, x, y, z, t) == ME ``SparseTensor.C`` at tensor stride 2**L."""
        n = self.count(L)
        out = torch.empty((max(n, 1), 5), dtype=torch.int32, device=self.device)
        check(self.lib.sps_unpack_coords(self.handle, L, _ptr(out), _stream()), "sps_unpack_coords")
        return out[:n].cpu().numpy()

    def inverse_map(self) -> np.ndarray:
        return self._read(self.lib.sps_ctx_inverse_map(self.handle), self.n, np.int32)

    def kernel_map(self, L: int, kind: str) -> np.ndarray:
        """Dense kernel map ``nbr[K, V]``: kind '3' (3x3x3x3), '5' (5x5x5x1, level 0) or
        'child' (2x2x2x1 children of level-L voxels)."""
        v = self.level(L)
        ptr, K = {"3": (v.nbr3, 81), "5": (v.nbr5, 125), "child": (v.child, 8)}[kind]
        if not ptr:
            raise ValueError(f"no '{kind}' map at level {L}")
        n = self.count(L)
        out = np.empty((K, n), np.int32)
        for k in range(K):      # row by row: the padding columns [n, ld) of the table are never written
            out[k] = self._read(ptr + 4 * k * v.ld, n, np.int32)
        return out

    def parent(self, L: int) -> np.ndarray:
        v = self.level(L)
        return self._read(v.parent, self.count(L), np.int32)

    # ---- network ---------------------------------------------------------------------
    @_on_device
    def forward(self, net: Net, points: torch.Tensor, voxel_size: float, out: torch.Tensor | None = None):
        """SPSModel.forward on device tensors; asynchronous (no host sync)."""
        _require_cuda(points, "points")
        assert points.dtype == torch.float32 and points.dim() == 2 and points.stride(1) == 1
        n = points.shape[0]
        if out is None:
            out = torch.empty(n, dtype=torch.float32, device=points.device)
        self._points = points
        self.n = n
        check(self.lib.sps_forward(self.handle, net.handle, _ptr(points), n, points.stride(0), float(voxel_size),
                                   _ptr(out), _stream()), "sps_forward")
        return out

    @_on_device
    def forward_features(self, net: Net, points: torch.Tensor, features: torch.Tensor, voxel_size: float,
                         out: torch.Tensor | None = None):
        """As :meth:`forward` with one input feature per point (voxel feature = mean of its points' features):
        MapMOSNet.forward (c_ws/src/mapmos/scripts/mapmos.py:59-83).  Asynchronous."""
        _require_cuda(points, "points")
        _require_cuda(features, "features")
        assert points.dtype == torch.float32 and points.dim() == 2 and points.stride(1) == 1
        features = features.reshape(-1).to(torch.float32).contiguous()
        n = points.shape[0]
        assert features.numel() == n
        if out is None:
            out = torch.empty(n, dtype=torch.float32, device=points.device)
        self._points, self._features = points, features
        self.n = n
        check(self.lib.sps_forward_features(self.handle, net.handle, _ptr(points), n, points.stride(0), _ptr(features),
                                            float(voxel_size), _ptr(out), _stream()), "sps_forward_features")
        return out

    def forward_host(self, net: Net, points: torch.Tensor, voxel_size: float, out: torch.Tensor | None = None):
        """Same through HOST tensors (H2D + forward + D2H + sync + status check)."""
        assert not points.is_cuda and points.dtype == torch.float32 and points.is_contiguous()
        n, ld = points.shape
        if out is None:
            out = torch.empty(n, dtype=torch.float32)
        self.n = n
        with torch.cuda.device(self.device):
            check(self.lib.sps_forward_host(self.handle, net.handle, _ptr(points), n, ld, float(voxel_size), _ptr(out),
                                            _stream()), "sps_forward_host")
        return out

    @_on_device
    def unet_forward(self, net: Net, feat0: torch.Tensor) -> torch.Tensor:
        logits = torch.empty(feat0.shape[0], dtype=torch.float32, device=self.device)
        check(self.lib.sps_unet_forward(self.handle, net.handle, _ptr(feat0), _ptr(logits), _stream()),
              "sps_unet_forward")
        return logits

    def launch_count(self) -> int:
        """Kernels the last fused forward of this engine enqueued."""
        return int(self.lib.sps_ctx_launch_count(self.handle))

    def profile(self, on: bool):
        check(self.lib.sps_profile_enable(self.handle, int(bool(on))), "sps_profile_enable")

    def profile_read(self, max_segments: int = 160) -> dict:
        """Synchronises; {stage name: milliseconds} of the last profiled forward (names repeat -> summed)."""
        names = C.create_string_buffer(32 * max_segments)
        ms = (C.c_float * max_segments)()
        cnt = C.c_int()
        check(self.lib.sps_profile_read(self.handle, names, ms, max_segments, C.byref(cnt)), "sps_profile_read")
        out = {}
        for i in range(cnt.value):
            nm = names.raw[32 * i:32 * i + 32].split(b"\0")[0].decode()
            out[nm] = out.get(nm, 0.0) + ms[i]
        return out


class MapHash:
    """Replicated base-map voxel hash (built once per process / rank) + submap crops."""

    def __init__(self, map_xyz: torch.Tensor, ds: float):
        _require_cuda(map_xyz, "map_xyz")
        self.lib = _cabi.load()
        self.device = map_xyz.device
        self.ds = float(ds)
        self.map_xyz = map_xyz[:, :3].contiguous().to(torch.float32)
        n = self.map_xyz.shape[0]
        nbytes = self.lib.sps_map_bytes(n)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            self.storage = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            check(self.lib.sps_map_build(C.byref(h), _ptr(self.storage), nbytes, _ptr(self.map_xyz), n, self.ds, _stream()),
                  "sps_map_build")
        self.handle = h
        self._scratch = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.sps_map_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def _scratch_for(self, nbytes):
        if self._scratch is None or self._scratch.numel() < nbytes:
            self._scratch = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self._scratch

    @_on_device
    def crop_voxel(self, scan_xyz: torch.Tensor):
        """``util.prune`` semantics -> (submap_points fp32 [M,3] on device, n_unique_scan_voxels)."""
        _require_cuda(scan_xyz, "scan_xyz")
        scan = scan_xyz[:, :3].contiguous().to(torch.float32)
        n = scan.shape[0]
        nbytes = self.lib.sps_map_bytes(max(n, 1))
        scratch = self._scratch_for(nbytes)
        out = torch.empty((max(n, 1), 3), dtype=torch.float32, device=self.device)
        counts = torch.zeros(2, dtype=torch.int32, device=self.device)
        check(self.lib.sps_submap_crop_voxel(self.handle, _ptr(scan), n, _ptr(scratch), nbytes, _ptr(out), _ptr(counts),
                                             _stream()), "sps_submap_crop_voxel")
        m, nuniq = counts.cpu().tolist()
        return out[:m], nuniq

    @_on_device
    def prune_batch(self, scans, offsets=None):
        """:meth:`crop_voxel` + ``util.infer``'s assembly for every scan of a batch, collated, in the library
        (``sps_prune_batch``).  ``scans``: a list of per-scan fp32 ``[n_b, >=3]`` tensors (x, y, z in the map frame;
        further columns are ignored) or one ``[sum n_b, >=3]`` tensor plus ``offsets`` (``B + 1`` ints), on the device
        or on the host.  Returns device tensors ``(rows [R, 5], row_offsets int32 [B + 1], counts int32 [B, 2])``: per
        scan its rows ``[b, x, y, z, 1]``, then its submap rows ``[b, corner, 0]`` (bit-identical to stacking the
        per-scan rows built from ``crop_voxel``), and ``crop_voxel``'s ``(len(submap), n_unique_scan_voxels)``.  One
        host synchronisation (the row count sizes the result)."""
        from .datasets import batch_parts, device_scans
        parts, offs, ld = batch_parts(scans, offsets, min_width=3)
        n, batch = offs[-1], len(offs) - 1
        src = device_scans(parts, n, ld, self.device)
        nbytes = self.lib.sps_prune_batch_scratch_bytes(n, batch)
        scratch = self._scratch_for(nbytes)
        rows = torch.empty((max(2 * n, 1), 5), dtype=torch.float32, device=self.device)
        row_offsets = torch.empty(batch + 1, dtype=torch.int32, device=self.device)
        n_rows = torch.empty(1, dtype=torch.int32, device=self.device)
        counts = torch.empty((batch, 2), dtype=torch.int32, device=self.device)
        h_off = (C.c_int64 * (batch + 1))(*offs)
        check(self.lib.sps_prune_batch(self.handle, _ptr(src), ld, h_off, batch, _ptr(rows), _ptr(row_offsets), _ptr(n_rows),
                                       _ptr(counts), _ptr(scratch), nbytes, _stream()), "sps_prune_batch")
        return rows[:int(n_rows.item())], row_offsets, counts

    @_on_device
    def crop_radius(self, center, radius: float) -> torch.Tensor:
        """MapMOS-style radius crop: indices (int32, map order) of map points within ``radius``."""
        n = self.map_xyz.shape[0]
        nbytes = self.lib.sps_map_bytes(max(n, 1))
        scratch = self._scratch_for(nbytes)
        idx = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        count = torch.zeros(1, dtype=torch.int32, device=self.device)
        c = (C.c_double * 3)(*[float(x) for x in center])
        check(self.lib.sps_submap_crop_radius(_ptr(self.map_xyz), n, c, float(radius), _ptr(idx), _ptr(count),
                                              _ptr(scratch), nbytes, _stream()), "sps_submap_crop_radius")
        return idx[: int(count.item())]

    @_on_device
    def infer_scan(self, engine: Engine, net: Net, scan_xyz: torch.Tensor, voxel_size: float,
                   out: torch.Tensor | None = None, counts: torch.Tensor | None = None):
        """prune -> assemble -> forward for one scan, fully asynchronous (no host sync)."""
        _require_cuda(scan_xyz, "scan_xyz")
        assert scan_xyz.dtype == torch.float32 and scan_xyz.is_contiguous() and scan_xyz.shape[1] == 3
        n = scan_xyz.shape[0]
        nbytes = self.lib.sps_infer_scan_scratch_bytes(n)
        scratch = self._scratch_for(nbytes)
        if out is None:
            out = torch.empty(n, dtype=torch.float32, device=self.device)
        if counts is None:
            counts = torch.empty(2, dtype=torch.int32, device=self.device)
        engine.n = n
        check(self.lib.sps_infer_scan(engine.handle, net.handle, self.handle, _ptr(scan_xyz), n, float(voxel_size),
                                      _ptr(out), _ptr(scratch), nbytes, _ptr(counts), _stream()), "sps_infer_scan")
        return out, counts


class ScanStreamer:
    """The ROS node's per-scan loop (c_ws/src/sps_filter/scripts/sps_node.py:111-120) as ONE CUDA graph:
    prune against the replicated map hash -> assemble -> SPSModel.forward, ~95 kernels captured once for a
    fixed scan size and replayed per scan, so the loop is no longer bound by launch overhead
    (measured: 1.07 ms -> see profiles/).  Scans with fewer points are padded with a copy of their
    first point (same voxel set, same scores for the real points)."""

    def __init__(self, map_hash: MapHash, engine: Engine, net: Net, n_scan: int, voxel_size: float):
        self.map_hash, self.engine, self.net = map_hash, engine, net
        self.n_scan, self.voxel_size = int(n_scan), float(voxel_size)
        dev = map_hash.device
        self.scan = torch.zeros((self.n_scan, 3), dtype=torch.float32, device=dev)
        self.scores = torch.empty(self.n_scan, dtype=torch.float32, device=dev)
        self.counts = torch.zeros(2, dtype=torch.int32, device=dev)
        self.graph = None

    def _capture(self):
        side = torch.cuda.Stream(device=self.scan.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):          # warm-up outside capture: kernel attributes, scratch allocation
            for _ in range(2):
                self.map_hash.infer_scan(self.engine, self.net, self.scan, self.voxel_size, out=self.scores,
                                         counts=self.counts)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.map_hash.infer_scan(self.engine, self.net, self.scan, self.voxel_size, out=self.scores,
                                     counts=self.counts)

    def infer(self, scan_xyz: torch.Tensor) -> torch.Tensor:
        """scan_xyz fp32 [n <= n_scan, 3] in the map frame, on the device or in (pinned) host memory -> scores [n]
        (a view of a static device buffer that the next call overwrites).  Asynchronous."""
        n = scan_xyz.shape[0]
        if n > self.n_scan or n == 0:
            raise ValueError(f"scan has {n} points, streamer was built for 1..{self.n_scan}")
        self.scan[:n].copy_(scan_xyz[:, :3], non_blocking=True)     # device tensor, or (pinned) host tensor: H2D on this stream
        if n < self.n_scan:
            self.scan[n:] = self.scan[0]
        if self.graph is None:
            self._capture()
        self.graph.replay()
        return self.scores[:n]
