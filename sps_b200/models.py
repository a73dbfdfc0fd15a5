"""Host-side mirror of ``sps.models.models`` (reference: src/sps/models/models.py) on top of the
B200 engine.  Same class names, constructor arguments, forward signatures and state_dict
layout, so reference checkpoints (Lightning prefix ``model.MinkUNet.``) load unchanged:

    SPSModel(voxel_size).forward(coordinates[N,5] fp32 (b,x,y,z,t)) -> scores[N] fp32   (models.py:13-30)
    SPSNet(hparams).forward(batch[N,>=5]) / .predict_step(batch, idx)                   (models.py:33-111)

Lightning and torchmetrics are not dependencies: SPSNet is a plain ``nn.Module`` and R2 is
computed inline.  Training (models.py:62-82,154-160) is out of scope (inference-only north star).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import NamedTuple

import numpy as np
import torch
import torch.nn as nn

from . import util
from ._cabi import SPS_ERR_CAPACITY, SpsError, check
from .datasets import MAX_BATCH, batch_parts
from .engine import Engine, Net, _ptr, _stream, norm_device
from .parallel import per_scan_metrics

PLANES = (8, 16, 32, 64, 64, 32, 16, 8)   # customminkunet.py:11
INIT_DIM = 8                              # customminkunet.py:12


class _Kernel(nn.Module):
    """Parameter holder with ME's ``MinkowskiConvolution`` state_dict layout:
    ``kernel`` fp32 [K_vol, Cin, Cout] (2-D [Cin, Cout] for 1x1), optional ``bias`` [1, Cout]."""

    def __init__(self, kernel_volume, cin, cout, bias=False, transpose=False):
        super().__init__()
        self.kernel_volume, self.in_channels, self.out_channels, self.transpose = kernel_volume, cin, cout, transpose
        shape = (cin, cout) if kernel_volume == 1 else (kernel_volume, cin, cout)
        self.kernel = nn.Parameter(torch.empty(shape))
        self.bias = nn.Parameter(torch.empty(1, cout)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        # ME default init (MinkowskiConvolutionBase.reset_parameters): U(-s, s)
        with torch.no_grad():
            s = 1.0 / math.sqrt((self.out_channels if self.transpose else self.in_channels) * self.kernel_volume)
            self.kernel.uniform_(-s, s)
            if self.bias is not None:
                self.bias.uniform_(-s, s)


class _BatchNorm(nn.Module):
    """ME.MinkowskiBatchNorm wraps ``nn.BatchNorm1d`` as attribute ``bn`` (resnet.py:92-94)."""

    def __init__(self, channels):
        super().__init__()
        self.bn = nn.BatchNorm1d(channels, eps=1e-5, momentum=0.1)


class _BasicBlock(nn.Module):
    """ME ``modules.resnet_block.BasicBlock`` parameters (c_ws/src/mapmos/scripts/minkunet.py:31-64)."""

    def __init__(self, inplanes, planes, downsample=None):
        super().__init__()
        self.conv1 = _Kernel(81, inplanes, planes)
        self.norm1 = _BatchNorm(planes)
        self.conv2 = _Kernel(81, planes, planes)
        self.norm2 = _BatchNorm(planes)
        self.downsample = downsample


def kaiming_normal_(tensor, mode="fan_out", nonlinearity="relu"):
    """ME.utils.kaiming_normal_ on a ``[K_vol, Cin, Cout]`` (or ``[Cin, Cout]``) kernel
    (resnet.py:88-90): fan_out = K_vol * Cout, fan_in = K_vol * Cin, std = sqrt(2 / fan)."""
    k = tensor.shape[0] if tensor.dim() == 3 else 1
    cin, cout = tensor.shape[-2], tensor.shape[-1]
    fan = k * (cout if mode == "fan_out" else cin)
    gain = nn.init.calculate_gain(nonlinearity)
    with torch.no_grad():
        return tensor.normal_(0, gain / math.sqrt(fan))


class CustomMinkUNet(nn.Module):
    """Parameters of ``CustomMinkUNet(in_channels=1, out_channels=1, D=4)`` = MinkUNet14 with
    PLANES=(8,16,32,64,64,32,16,8), INIT_DIM=8 (customminkunet.py:10-12; graph
    minkunet.py:52-159; init resnet.py:87-94).  The forward lives in the CUDA library
    (csrc/net.cu) -- this module only owns the tensors under the reference's key names."""

    def __init__(self, in_channels=1, out_channels=1, D=4):
        super().__init__()
        if (in_channels, D) != (1, 4) or out_channels < 1:
            raise NotImplementedError("the B200 engine implements CustomMinkUNet(1, out_channels, D=4) (models.py:17, mos4d.py:15)")
        P, self.inplanes = PLANES, INIT_DIM
        self.conv0p1s1 = _Kernel(125, in_channels, self.inplanes)
        self.bn0 = _BatchNorm(self.inplanes)
        for i, name in enumerate(["conv1p1s2", "conv2p2s2", "conv3p4s2", "conv4p8s2"]):
            setattr(self, name, _Kernel(8, self.inplanes, self.inplanes))
            setattr(self, f"bn{i + 1}", _BatchNorm(self.inplanes))
            setattr(self, f"block{i + 1}", self._make_layer(P[i]))
        skips = [P[2], P[1], P[0], INIT_DIM]
        for i, name in enumerate(["convtr4p16s2", "convtr5p8s2", "convtr6p4s2", "convtr7p2s2"]):
            setattr(self, name, _Kernel(8, self.inplanes, P[4 + i], transpose=True))
            setattr(self, f"bntr{4 + i}", _BatchNorm(P[4 + i]))
            self.inplanes = P[4 + i] + skips[i]
            setattr(self, f"block{5 + i}", self._make_layer(P[4 + i]))
        self.final = _Kernel(1, P[7], out_channels, bias=True)
        self.weight_initialization()
        self.weights_version = 0   # bumped whenever tensors are (re)loaded or moved
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.touch())

    def touch(self):
        self.weights_version += 1

    def _apply(self, fn, *args, **kwargs):
        self.weights_version += 1
        return super()._apply(fn, *args, **kwargs)

    def _make_layer(self, planes):  # resnet.py:96-126 with blocks=1, stride=1, expansion=1
        downsample = None
        if self.inplanes != planes:
            downsample = nn.Sequential(_Kernel(1, self.inplanes, planes), _BatchNorm(planes))
        layer = nn.Sequential(_BasicBlock(self.inplanes, planes, downsample))
        self.inplanes = planes
        return layer

    def weight_initialization(self):  # resnet.py:87-94
        for m in self.modules():
            if isinstance(m, _Kernel) and not m.transpose:
                kaiming_normal_(m.kernel, mode="fan_out", nonlinearity="relu")
            if isinstance(m, _BatchNorm):
                nn.init.constant_(m.bn.weight, 1)
                nn.init.constant_(m.bn.bias, 0)


class _Pending:
    """Handle of an in-flight ``SPSModel.forward_async`` or ``SPSModel.infer_scans_async`` call."""

    def __init__(self, event, out, engine, device_scores=None):
        self._event, self._out, self._engine = event, out, engine
        # the scores on the device (valid once the call is done; the lane reuses the buffer `lanes` calls later)
        self.device_scores = device_scores if device_scores is not None else out

    def result(self, check: bool = True):
        """Wait for the call and return its results (forward_async: the scores).  ``check`` (default) also reads the
        engine's sticky status word, so a coordinate outside the voxel-key range raises here instead of leaving NaN
        scores behind."""
        self._event.synchronize()
        if check:
            self._engine.status()
        return self._out


class _PendingRadius:
    """Handle of an in-flight ``SPSModel.predict_radius_async`` call.  ``device_out`` (scan scores, counts, sums),
    ``device_n_rows`` and ``row_capacity`` are the call's device results, its true row count and the rows its lane
    held; they are valid on the lane's ``stream`` after the call and until the lane's next call."""

    def __init__(self, event, out, engine, n_rows, retry, device_out=None, device_n_rows=None, row_capacity=0,
                 stream=None):
        self._event, self._out, self._engine, self._n_rows, self._retry = event, out, engine, n_rows, retry
        self.device_out, self.device_n_rows, self.row_capacity, self.stream = device_out, device_n_rows, row_capacity, stream

    def result(self, check: bool = True):
        """Wait for the call and return ``(scan_scores, counts, sums)``.  ``check`` (default) also reads the engine's
        sticky status word: a coordinate outside the voxel-key range raises here; rows that did not fit the lane's
        context make the call run once more with contexts of the true row count."""
        self._event.synchronize()
        if check:
            try:
                self._engine.status()
            except SpsError as e:
                if e.code != SPS_ERR_CAPACITY:
                    raise
                return self._retry(int(self._n_rows[0])).result(check)
        return self._out


class FilteredScans(NamedTuple):
    """Results of ``SPSModel.filter_scans_async`` for a batch of B scans of n_total points."""
    scan_scores: torch.Tensor    # fp32 [n_total]: the scan points' scores, in input order
    kept: torch.Tensor           # fp32 [K, 4]: the published rows (sensor-frame x, y, z, column 3), scan after scan
    kept_offsets: torch.Tensor   # int32 [B + 1]: scan b's published rows are kept[kept_offsets[b]:kept_offsets[b+1]]
    counts: torch.Tensor         # int32 [B, 2]: MapHash.crop_voxel's (len(submap), n_unique_scan_voxels) per scan
    metric_counts: torch.Tensor  # int64 [B, 4]: per-scan confusion counts (parallel.device_partials' layout)
    metric_sums: torch.Tensor    # float64 [B, 5]: per-scan sums (parallel.device_partials' layout)


class _PendingFilter(_Pending):
    """Handle of an in-flight ``SPSModel.filter_scans_async`` call.  ``device_out`` is the call's :class:`FilteredScans`
    on the device, ``kept`` with all ``sum n_b`` rows of the lane's buffer (the first ``kept_offsets[B]`` are the
    published ones); it is valid on the lane's ``stream`` after the call and until the lane's next call."""

    def __init__(self, event, out, engine, kept_end, device_out=None, stream=None):
        super().__init__(event, out, engine)
        self._kept_end = kept_end     # pinned host int32 [1]: K, once the call is done
        self.device_out, self.stream = device_out, stream

    def result(self, check: bool = True) -> FilteredScans:
        """Wait for the call and return its :class:`FilteredScans` (``check``: as ``_Pending.result``)."""
        out = super().result(check)
        return out._replace(kept=out.kept[:int(self._kept_end[0])])


def _lane_buffers(buf, device):
    """``grow(name, shape, dtype, pinned=False)``: the lane buffer ``buf[name]``, (re)allocated when it is missing or
    has fewer than ``shape[0]`` rows -- on ``device``, or in pinned host memory."""
    def grow(name, shape, dtype, pinned=False):
        t = buf.get(name)
        if t is None or t.shape[0] < shape[0]:
            t = torch.empty(shape, dtype=dtype, device="cpu" if pinned else device)
            buf[name] = t.pin_memory() if pinned else t
        return buf[name]
    return grow


class SPSModel(nn.Module):
    def __init__(self, voxel_size: float, max_points: int = 0):
        super().__init__()
        self.voxel_size = float(voxel_size)
        self.quantization = torch.Tensor([1.0, voxel_size, voxel_size, voxel_size, 1.0])  # models.py:16
        self.MinkUNet = CustomMinkUNet(in_channels=1, out_channels=1, D=4)
        self.sigmoid = nn.Sigmoid()
        self._engine = None
        self._net = None
        self._min_points = int(max_points)
        self._net_version = -1
        self._host_out = None
        self._pipe = None
        self.lanes = 3            # engine contexts / streams that forward_async alternates between
        self.output_channel, self.apply_sigmoid = 0, True   # models.py:28-29: sigmoid of the single output channel
        self.conv_backend = None  # None: the host default of sps_b200.engine.DEFAULTS at engine creation
        # forward_async replays the whole forward (~56 kernels) as ONE CUDA graph per (lane, input buffer, row count):
        # the first call with a given input runs eagerly, the second is captured, later ones are replays.  Only for
        # inputs of at most `graph_max_rows` rows, whose forward is bound by launch overhead; measured on the batch-8
        # workload (2.47 M rows, GPU-bound) replay was 2 % SLOWER than enqueueing kernel by kernel.
        self.use_graphs = os.environ.get("SPS_NO_GRAPHS", "0") != "1"
        self.graph_max_rows = 400_000

    def set_conv_backend(self, backend: int):
        """Arithmetic mode of every engine this model owns (0 auto, 1 exact fp32, 2 TF32 on fp32 rows, 3 fp16 rows)."""
        self.conv_backend = int(backend)
        for eng in self._engines():
            eng.set_conv_backend(self.conv_backend)

    def _engines(self):
        out = [self._engine] if self._engine is not None else []
        if self._pipe is not None:
            out += [e for e in self._pipe["engine"] if e is not self._engine]
        return out

    def _new_engine(self, cap, device):
        eng = Engine(cap, device)
        if self.conv_backend is not None:
            eng.set_conv_backend(self.conv_backend)
        return eng

    def invalidate(self):
        """Weights changed in place: re-fold and re-upload them at the next forward."""
        self.MinkUNet.touch()

    def _prepare(self, n, device):
        device = norm_device(device)
        if self._net is None or self._net.device != device or self._net_version != self.MinkUNet.weights_version:
            self._net = Net(self.MinkUNet.state_dict(), device, self.output_channel, self.apply_sigmoid)
            self._net_version = self.MinkUNet.weights_version
        if self._engine is None or self._engine.max_points < n or self._engine.device != device:
            cap = max(self._min_points, 1 << max(10, int(math.ceil(math.log2(max(n, 1))))))
            self._engine = None  # release the old workspace before growing
            self._engine = self._new_engine(cap, device)
        return self._engine, self._net

    def forward(self, coordinates: torch.Tensor):
        """coordinates fp32 [N,5] = (b, x, y, z, t) in metres, t in {0,1} -> scores fp32 [N]
        (models.py:20-30).  CUDA tensors run asynchronously on the current stream (no host synchronisation: a
        coordinate outside the voxel-key range -- INTEGRATION.md "Coordinate limits" -- leaves NaN scores and a
        sticky status word that ``check()`` / ``predict_step`` / ``util.infer`` raise on); CPU tensors go
        through the host entry point (H2D + forward + D2H, synchronising, status checked)."""
        if self.training:
            raise RuntimeError("sps_b200 is inference-only (call .eval()); training is out of scope")
        coordinates = coordinates.reshape(-1, coordinates.shape[-1]).to(torch.float32)
        if coordinates.stride(-1) != 1:
            coordinates = coordinates.contiguous()
        if coordinates.is_cuda:
            engine, net = self._prepare(coordinates.shape[0], coordinates.device)
            return engine.forward(net, coordinates, self.voxel_size)
        device = next(self.MinkUNet.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("move the model to a CUDA device first: sps_b200 has no CPU path")
        engine, net = self._prepare(coordinates.shape[0], device)
        n = coordinates.shape[0]
        if self._host_out is None or self._host_out.numel() < n:
            # pinned landing buffer for the D2H of the scores, reused across calls: the returned
            # tensor is a view that the NEXT host-side forward overwrites (clone it to keep it)
            self._host_out = torch.empty(max(n, 1), dtype=torch.float32).pin_memory()
        return engine.forward_host(net, coordinates.contiguous(), self.voxel_size, out=self._host_out[:n])

    def forward_async(self, coordinates: torch.Tensor):
        """Pipelined entry point.  ``coordinates`` may live on the device (no copies at all) or be a
        (preferably pinned) HOST tensor; in the latter case the H2D
        copy runs on a side stream into one of two device staging buffers, the forward and the D2H of
        the scores are queued behind it, and a handle is returned immediately -- so the copies of
        call k+1 overlap the kernels of call k.  ``handle.result()`` waits for and returns the scores
        (a pinned host tensor that the call after next reuses)."""
        if self.training:
            raise RuntimeError("sps_b200 is inference-only (call .eval()); training is out of scope")
        assert coordinates.dtype == torch.float32 and coordinates.dim() == 2
        on_device = coordinates.is_cuda
        device = next(self.MinkUNet.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("move the model to a CUDA device first: sps_b200 has no CPU path")
        n, ld = coordinates.shape
        p, net = self._lanes(n, ld, device)
        slot = self._next_lane(p)
        lane_engine, compute = p["engine"][slot], p["stream"][slot]
        d_in, d_out, h_out = p["d_in"][slot][:n], p["d_out"][slot][:n], p["h_out"][slot][:n]
        compute.wait_stream(torch.cuda.current_stream(device))
        if on_device:
            # inputs already resident in HBM: no copies, the scores stay on the device
            with torch.cuda.stream(compute):
                self._lane_forward(p, slot, lane_engine, net, coordinates, d_out, compute)
                done = torch.cuda.Event()
                done.record(compute)
            p["busy"][slot] = done
            return _Pending(done, d_out, lane_engine)
        with torch.cuda.stream(p["copy"]):
            d_in.copy_(coordinates, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(p["copy"])
        with torch.cuda.stream(compute):
            compute.wait_event(ready)
            self._lane_forward(p, slot, lane_engine, net, d_in, d_out, compute)
            h_out.copy_(d_out, non_blocking=True)
            done = torch.cuda.Event()
            done.record(compute)
        p["busy"][slot] = done
        engine = lane_engine
        return _Pending(done, h_out, engine, device_scores=d_out)

    def _lanes(self, n, ld, device):
        """The lanes of the pipelined entry points, (re)made for inputs of up to ``n`` rows of width ``ld`` (None: any
        width; a new set of lanes then takes 5)."""
        engine, net = self._prepare(n, device)
        p = self._pipe
        if p is None or p["cap"] < n or (ld is not None and p["ld"] != ld):
            cap = max(n, engine.max_points)
            ld = ld or 5
            # two complete lanes (engine context + stream + staging buffers): consecutive calls alternate,
            # so the hash/kernel-map phase of one call overlaps the convolution phase of the other
            p = self._pipe = {"cap": cap, "ld": ld, "k": 0, "copy": torch.cuda.Stream(device=device),
                              "engine": [engine] + [self._new_engine(engine.max_points, device) for _ in range(self.lanes - 1)],
                              "stream": [torch.cuda.Stream(device=device) for _ in range(self.lanes)],
                              "d_in": [torch.empty((cap, ld), dtype=torch.float32, device=device) for _ in range(self.lanes)],
                              "d_out": [torch.empty(cap, dtype=torch.float32, device=device) for _ in range(self.lanes)],
                              "h_out": [torch.empty(cap, dtype=torch.float32).pin_memory() for _ in range(self.lanes)],
                              "busy": [None] * self.lanes, "graphs": [dict() for _ in range(self.lanes)],
                              "radius": [dict() for _ in range(self.lanes)], "prune": [dict() for _ in range(self.lanes)],
                              "filter": [dict() for _ in range(self.lanes)]}
        return p, net

    def _next_lane(self, p):
        """The lane of the next call, once the call that used it before is done with its buffers."""
        slot = p["k"] % self.lanes
        p["k"] += 1
        if p["busy"][slot] is not None:
            p["busy"][slot].synchronize()          # the buffers of this lane are free again
        return slot

    def predict_radius_async(self, scans, submap, eps: float, offsets=None):
        """``scripts/predict.py``'s loop body for a whole batch in one asynchronous library call: for every scan its
        radius submap from ``submap`` (a :class:`sps_b200.datasets.RadiusSubmap` of the base map, radius =
        VOXEL_SIZE), the collated rows (``RadiusSubmap.make_batch``), ``forward`` on them and ``predict_step``'s metric
        partials per scan (threshold ``eps``).  ``scans``: a list of per-scan fp32 ``[n_b, >=4]`` tensors (x, y, z,
        label in the map frame) or one ``[sum n_b, >=4]`` tensor plus ``offsets`` (``B + 1`` ints).

        Returns a handle whose ``result()`` gives ``(scan_scores [sum n_b], counts int64 [B, 4], sums float64 [B, 5])``
        (layouts of ``parallel.device_partials``; ``parallel.per_scan_metrics`` turns them into predict.py's values).
        Host scans go to the device on a copy stream into the staging buffer of one of the model's lanes (the copies of
        call k+1 overlap the kernels of call k) and the results come back to pinned host memory; device scans are read
        in place and the results stay on the device.  Either way the buffers belong to the lane: the call ``lanes``
        calls later reuses them.  The row capacity is the lane context's size; rows that do not fit are never scored:
        ``result()`` then grows the contexts to the true row count and runs the batch once more (the only extra host
        synchronisation, on that path only)."""
        if self.training:
            raise RuntimeError("sps_b200 is inference-only (call .eval()); training is out of scope")
        parts, offs, ld = batch_parts(scans, offsets)
        return self._predict_radius(parts, offs, ld, submap, float(eps), 6 * offs[-1])

    def _predict_radius(self, parts, offs, ld, submap, eps, rows_guess):
        device = next(self.MinkUNet.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("move the model to a CUDA device first: sps_b200 has no CPU path")
        if submap.map_xyz.device != device:
            raise RuntimeError("the submap's base map must live on the model's device")
        n, batch = offs[-1], len(offs) - 1
        p, net = self._lanes(max(rows_guess, 1), None, device)
        slot = self._next_lane(p)
        lane_engine, compute = p["engine"][slot], p["stream"][slot]
        cap = lane_engine.max_points
        on_device = all(t.is_cuda for t, _ in parts)
        buf = p["radius"][slot]
        lib = lane_engine.lib
        grow = _lane_buffers(buf, device)
        nbytes = lib.sps_radius_batch_scratch_bytes(n, batch)
        rows = grow("rows", (cap, 6), torch.float32)
        scratch = grow("scratch", (nbytes,), torch.uint8)    # the caching allocator hands out 512-byte aligned blocks
        row_offsets = grow("row_offsets", (MAX_BATCH + 1,), torch.int32)
        n_rows = grow("n_rows", (1,), torch.int32)
        scores = grow("scores", (max(n, 1),), torch.float32)
        counts = grow("counts", (MAX_BATCH, 4), torch.int64)
        sums = grow("sums", (MAX_BATCH, 5), torch.float64)
        compute.wait_stream(torch.cuda.current_stream(device))
        src = self._lane_scans(p, buf, grow, parts, n, ld, on_device, compute, device)
        h_off = (C.c_int64 * (batch + 1))(*offs)
        with torch.cuda.device(device), torch.cuda.stream(compute):
            check(lib.sps_predict_radius_batch(lane_engine.handle, net.handle, submap.handle, _ptr(src), ld, h_off, batch,
                                               _ptr(rows), cap, _ptr(row_offsets), _ptr(n_rows), _ptr(scratch), nbytes,
                                               self.voxel_size, eps, _ptr(scores), _ptr(counts), _ptr(sums),
                                               _stream(device)), "sps_predict_radius_batch")
            out = dev_out = (scores[:n], counts[:batch], sums[:batch])
            if not on_device:
                h = (grow("h_scores", (max(n, 1),), torch.float32, True), grow("h_counts", (MAX_BATCH, 4), torch.int64, True),
                     grow("h_sums", (MAX_BATCH, 5), torch.float64, True))
                out = (h[0][:n], h[1][:batch], h[2][:batch])
                for dst, s in zip(out, (scores[:n], counts[:batch], sums[:batch])):
                    dst.copy_(s, non_blocking=True)
            h_rows = grow("h_n_rows", (1,), torch.int32, True)
            h_rows.copy_(n_rows, non_blocking=True)
            done = torch.cuda.Event()
            done.record(compute)
        p["busy"][slot] = done

        def retry(true_rows):
            return self._predict_radius(parts, offs, ld, submap, eps, true_rows)
        return _PendingRadius(done, out, lane_engine, h_rows, retry, dev_out, n_rows, cap, compute)

    @staticmethod
    def _lane_scans(p, buf, grow, parts, n, ld, on_device, compute, device):
        """The scans of a batched call on the device, ready on the lane's stream ``compute``: a single device part is
        read in place; otherwise the parts are copied into the lane's staging buffer, host parts on the copy stream (the
        copies of call k+1 overlap the kernels of call k).  The sources stay alive until the lane's next call."""
        if len(parts) == 1 and on_device and parts[0][0].device == device:
            src = parts[0][0]
        else:
            src = grow(("scans", ld), (max(n, 1), ld), torch.float32)
            copy = compute if on_device else p["copy"]
            with torch.cuda.stream(copy):
                for t, start in parts:
                    src[start:start + t.shape[0]].copy_(t, non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(copy)
            compute.wait_event(ready)
        buf["keep"] = (parts, src)
        return src

    def infer_scans_async(self, scans, map_hash, offsets=None):
        """The ROS node's per-scan loop body (``sps_node.py:111-120``: ``util.prune`` against the base map, then
        ``util.infer``) for a whole batch of scans in one asynchronous library call (``sps_infer_prune_batch``): every
        scan's voxel-pruned submap from ``map_hash`` (a :class:`sps_b200.engine.MapHash`; its ``ds`` is the crop
        lattice, this model's voxel size the forward's), the collated rows, one ``forward`` on them.  ``scans``: a list
        of per-scan fp32 ``[n_b, >=3]`` tensors (x, y, z in the map frame; further columns are ignored) or one
        ``[sum n_b, >=3]`` tensor plus ``offsets`` (``B + 1`` ints); 1..255 scans, empty ones allowed.

        Returns a handle whose ``result()`` gives ``(scan_scores [sum n_b], counts int32 [B, 2])``: the scores of the
        scan points in input order (those of ``util.infer`` on each scan's rows) and per scan ``MapHash.crop_voxel``'s
        ``(len(submap), n_unique_scan_voxels)``; it raises :class:`SpsError` when a point lay outside the voxel-key
        range.  Device scans are read in place and the results stay on the device; host (preferably pinned) scans go
        to the device on the copy stream and the results come back to pinned host memory.  Either way the buffers
        belong to one of the model's lanes, whose contexts hold ``2 * sum n_b`` rows: the call ``lanes`` calls later
        reuses them.  The forward is sized by ``2 * sum n_b`` rows, which, like a row count, decides the default shape
        sort (``sps_ctx_set_pattern_sort`` mode 1)."""
        if self.training:
            raise RuntimeError("sps_b200 is inference-only (call .eval()); training is out of scope")
        parts, offs, ld = batch_parts(scans, offsets, min_width=3)
        device = next(self.MinkUNet.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("move the model to a CUDA device first: sps_b200 has no CPU path")
        if norm_device(map_hash.device) != norm_device(device):
            raise RuntimeError("the map hash must live on the model's device")
        n, batch = offs[-1], len(offs) - 1
        p, net = self._lanes(max(2 * n, 1), None, device)
        slot = self._next_lane(p)
        lane_engine, compute = p["engine"][slot], p["stream"][slot]
        on_device = all(t.is_cuda for t, _ in parts)
        buf = p["prune"][slot]
        lib = lane_engine.lib
        grow = _lane_buffers(buf, device)
        nbytes = lib.sps_prune_batch_scratch_bytes(n, batch)
        rows = grow("rows", (max(2 * n, 1), 5), torch.float32)
        scratch = grow("scratch", (nbytes,), torch.uint8)    # the caching allocator hands out 512-byte aligned blocks
        row_offsets = grow("row_offsets", (MAX_BATCH + 1,), torch.int32)
        n_rows = grow("n_rows", (1,), torch.int32)
        scores = grow("scores", (max(n, 1),), torch.float32)
        counts = grow("counts", (MAX_BATCH, 2), torch.int32)
        compute.wait_stream(torch.cuda.current_stream(device))
        src = self._lane_scans(p, buf, grow, parts, n, ld, on_device, compute, device)
        h_off = (C.c_int64 * (batch + 1))(*offs)
        with torch.cuda.device(device), torch.cuda.stream(compute):
            check(lib.sps_infer_prune_batch(lane_engine.handle, net.handle, map_hash.handle, _ptr(src), ld, h_off, batch,
                                            _ptr(rows), _ptr(row_offsets), _ptr(n_rows), _ptr(counts), _ptr(scratch), nbytes,
                                            self.voxel_size, _ptr(scores), _stream(device)), "sps_infer_prune_batch")
            out = (scores[:n], counts[:batch])
            if not on_device:
                h = (grow("h_scores", (max(n, 1),), torch.float32, True), grow("h_counts", (MAX_BATCH, 2), torch.int32, True))
                out = (h[0][:n], h[1][:batch])
                for dst, s in zip(out, (scores[:n], counts[:batch])):
                    dst.copy_(s, non_blocking=True)
            done = torch.cuda.Event()
            done.record(compute)
        p["busy"][slot] = done
        return _Pending(done, out, lane_engine)

    def filter_scans_async(self, scans, poses, map_hash, eps: float, offsets=None):
        """The ROS node's whole callback (``sps_node.py:88-176``) for a batch of sensor-frame scans in one asynchronous
        library call (``sps_filter_scans_batch``): every scan moved into the map frame with its pose
        (``util.transform_point_cloud``), ``infer_scans_async`` on the moved scans, the node's metrics against the
        scan's column 3 (``pred = score < eps``, ``gt = label < eps``) and the rows the node publishes
        (``util.filter_scan``: sensor-frame x, y, z, column 3 of the points whose score is ``<= eps``).  ``scans``: a
        list of per-scan fp32 ``[n_b, >=4]`` tensors (x, y, z, intensity in the sensor frame; the intensity is also
        the label) or one ``[sum n_b, >=4]`` tensor plus ``offsets``; ``poses``: float64 ``[B, 4, 4]`` (numpy array or
        tensor, on the host or the device), scan b's row-major matrix (``util.to_tr_matrix``).

        Returns a handle whose ``result()`` gives a :class:`FilteredScans`; it raises :class:`SpsError` when a
        map-frame point lay outside the voxel-key range.  ``parallel.per_scan_metrics(metric_counts, metric_sums)``
        gives the node's per-scan values, ``util.to_rosmsg(kept[o[b]:o[b+1]], header)`` scan b's message.  Device
        scans give device results; host (preferably pinned) scans go to the device on the copy stream and the results
        come back to pinned host memory (the whole ``[sum n_b, 4]`` buffer of published rows, which ``result()``
        slices).  Host poses go through a pinned buffer of the lane on the copy stream.  Either way the buffers belong
        to one of the model's lanes: the call ``lanes`` calls later reuses them."""
        if self.training:
            raise RuntimeError("sps_b200 is inference-only (call .eval()); training is out of scope")
        parts, offs, ld = batch_parts(scans, offsets, min_width=4)
        n, batch = offs[-1], len(offs) - 1
        poses = poses if isinstance(poses, torch.Tensor) else torch.as_tensor(np.asarray(poses))
        if poses.dtype != torch.float64 or tuple(poses.shape) != (batch, 4, 4):
            raise ValueError(f"poses must be float64 [{batch}, 4, 4] (one matrix per scan), got {poses.dtype} "
                             f"{tuple(poses.shape)}")
        device = next(self.MinkUNet.parameters()).device
        if device.type != "cuda":
            raise RuntimeError("move the model to a CUDA device first: sps_b200 has no CPU path")
        if norm_device(map_hash.device) != norm_device(device):
            raise RuntimeError("the map hash must live on the model's device")
        if poses.is_cuda and poses.device != device:
            raise RuntimeError("device poses must live on the model's device")
        p, net = self._lanes(max(2 * n, 1), None, device)
        slot = self._next_lane(p)
        lane_engine, compute = p["engine"][slot], p["stream"][slot]
        on_device = all(t.is_cuda for t, _ in parts)
        buf = p["filter"][slot]
        lib = lane_engine.lib
        grow = _lane_buffers(buf, device)
        nbytes = lib.sps_filter_scans_batch_scratch_bytes(n, batch)
        rows = grow("rows", (max(2 * n, 1), 5), torch.float32)
        scratch = grow("scratch", (nbytes,), torch.uint8)    # the caching allocator hands out 512-byte aligned blocks
        row_offsets = grow("row_offsets", (MAX_BATCH + 1,), torch.int32)
        n_rows = grow("n_rows", (1,), torch.int32)
        scores = grow("scores", (max(n, 1),), torch.float32)
        counts = grow("counts", (MAX_BATCH, 2), torch.int32)
        metric_counts = grow("metric_counts", (MAX_BATCH, 4), torch.int64)
        metric_sums = grow("metric_sums", (MAX_BATCH, 5), torch.float64)
        kept = grow("kept", (max(n, 1), 4), torch.float32)
        kept_offsets = grow("kept_offsets", (MAX_BATCH + 1,), torch.int32)
        if poses.is_cuda:
            d_poses = poses.contiguous()                   # (on the current stream, which the lane's stream waits for)
            buf["keep_poses"] = d_poses                     # alive until the lane's next call
        compute.wait_stream(torch.cuda.current_stream(device))
        src = self._lane_scans(p, buf, grow, parts, n, ld, on_device, compute, device)
        if not poses.is_cuda:
            h_poses = grow("h_poses", (MAX_BATCH, 4, 4), torch.float64, True)
            h_poses[:batch].copy_(poses)
            d_poses = grow("poses", (MAX_BATCH, 4, 4), torch.float64)
            with torch.cuda.stream(p["copy"]):
                d_poses[:batch].copy_(h_poses[:batch], non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(p["copy"])
            compute.wait_event(ready)
        h_off = (C.c_int64 * (batch + 1))(*offs)
        with torch.cuda.device(device), torch.cuda.stream(compute):
            check(lib.sps_filter_scans_batch(lane_engine.handle, net.handle, map_hash.handle, _ptr(src), ld, h_off, batch,
                                             _ptr(d_poses), float(eps), self.voxel_size, _ptr(rows), _ptr(row_offsets),
                                             _ptr(n_rows), _ptr(counts), _ptr(scores), _ptr(metric_counts),
                                             _ptr(metric_sums), _ptr(kept), _ptr(kept_offsets), _ptr(scratch), nbytes,
                                             _stream(device)), "sps_filter_scans_batch")
            out = dev_out = FilteredScans(scores[:n], kept[:n], kept_offsets[:batch + 1], counts[:batch],
                                          metric_counts[:batch], metric_sums[:batch])
            if on_device:
                kept_end = grow("h_kept_end", (1,), torch.int32, True)
                kept_end.copy_(kept_offsets[batch:batch + 1], non_blocking=True)
            else:                                       # every result to pinned host memory, K not known yet
                dev, out = out, FilteredScans(*(grow("h_" + name, (max(t.shape[0], 1),) + t.shape[1:], t.dtype, True)
                                                [:t.shape[0]] for name, t in zip(FilteredScans._fields, out)))
                for dst, t in zip(out, dev):
                    dst.copy_(t, non_blocking=True)
                kept_end = out.kept_offsets[batch:batch + 1]
            done = torch.cuda.Event()
            done.record(compute)
        p["busy"][slot] = done
        return _PendingFilter(done, out, lane_engine, kept_end, dev_out, compute)

    def _lane_forward(self, p, slot, lane_engine, net, src, d_out, compute):
        """One forward on a lane's stream (current), eagerly or as a CUDA-graph replay.  Every size that only exists on
        the device stays there, so the captured launch sequence is valid for any content of the same buffers."""
        if not self.use_graphs or src.shape[0] > self.graph_max_rows:
            lane_engine.forward(net, src, self.voxel_size, out=d_out)
            return
        graphs = p["graphs"][slot]
        key = (src.data_ptr(), src.shape[0], src.stride(0), d_out.data_ptr(), lane_engine.conv_backend, id(net))
        entry = graphs.get(key)
        if entry is None:                      # first sight: eager (also sets one-time kernel attributes)
            if len(graphs) >= 8:
                graphs.clear()
            graphs[key] = "warm"
            lane_engine.forward(net, src, self.voxel_size, out=d_out)
        elif entry == "warm":                  # second sight: capture, then replay
            compute.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=compute):
                lane_engine.forward(net, src, self.voxel_size, out=d_out)
            graphs[key] = (g, src, d_out, net)   # the graph holds raw pointers: keep the tensors alive with it
            g.replay()
        else:
            entry[0].replay()

    def check(self):
        """Synchronise and raise if a forward since the last check met an out-of-range coordinate."""
        for eng in self._engines():
            eng.status()


class MOS4DNet(SPSModel):
    """The 4DMOS baseline the reference ships (c_ws/src/mos4d/scripts/mos4d.py:10-32): the same network with
    ``CustomMinkUNet(in_channels=1, out_channels=3, D=4)``; ``forward`` returns the raw logit of class 2 (moving)
    for every point.  The time column is the scan index of a sliding window (mos4d_node.py:98-117); only time
    DIFFERENCES matter to the sparse convolutions, so the window is shifted to start at t = 0 (the voxel key holds
    16 time planes: windows of up to 16 scans, the node uses 10)."""

    def __init__(self, voxel_size: float, max_points: int = 0):
        super().__init__(voxel_size, max_points)
        self.MinkUNet = CustomMinkUNet(in_channels=1, out_channels=3, D=4)
        self.output_channel, self.apply_sigmoid = 2, False     # mos4d.py:32 `out.features[:, 2]`

    def forward(self, coordinates: torch.Tensor):
        coordinates = coordinates.reshape(-1, coordinates.shape[-1]).to(torch.float32)
        if coordinates.shape[0]:
            coordinates = coordinates.clone()
            coordinates[:, 4] -= torch.floor(coordinates[:, 4].min())
        return super().forward(coordinates)


class MapMOSNet(SPSModel):
    """The MapMOS baseline the reference ships (c_ws/src/mapmos/scripts/mapmos.py:32-90): the same network
    (``CustomMinkUNet14(1, 1, D=4)``), input features = index-normalised scan/map indices averaged per voxel, t = 0 for
    the scan and -1 for the map (shifted to 1 / 0 here: only time differences matter), raw logits out."""

    def __init__(self, voxel_size: float, max_points: int = 0):
        super().__init__(voxel_size, max_points)
        self.output_channel, self.apply_sigmoid = 0, False

    def forward(self, coordinates: torch.Tensor, indices: torch.Tensor):
        if self.training:
            raise RuntimeError("sps_b200 is inference-only (call .eval()); training is out of scope")
        coordinates = coordinates.reshape(-1, 5).to(torch.float32)
        if not coordinates.is_cuda:
            raise RuntimeError("MapMOSNet.forward needs CUDA tensors: sps_b200 has no CPU path")
        indices = indices.reshape(-1).to(coordinates)
        i_max, i_min = torch.max(indices), torch.min(indices)                     # mapmos.py:66-71
        features = torch.ones_like(indices) if bool(i_min == i_max) else 1 + (i_max - indices) / (i_max - i_min)
        coordinates = coordinates.clone()
        coordinates[:, 4] -= torch.floor(coordinates[:, 4].min())
        engine, net = self._prepare(coordinates.shape[0], coordinates.device)
        return engine.forward_features(net, coordinates, features, self.voxel_size)

    def predict(self, scan_input, map_input, scan_indices, map_indices):          # mapmos.py:39-57
        def extend(tensor, batch_idx, time_idx):
            ones = torch.ones(len(tensor), 1).type_as(tensor)
            return torch.hstack([batch_idx * ones, tensor, time_idx * ones])
        coordinates = torch.vstack([extend(scan_input, 0, 0).reshape(-1, 5), extend(map_input, 0, -1).reshape(-1, 5)])
        indices = torch.vstack([scan_indices.reshape(-1, 1), map_indices.reshape(-1, 1)])
        logits = self.forward(coordinates, indices)
        mask_scan = coordinates[:, 4] == 0.0
        return logits[mask_scan], logits[~mask_scan]


class SPSNet(nn.Module):
    """Inference surface of the reference's LightningModule (models.py:33-111)."""

    def __init__(self, hparams: dict, data_size=0, save_vis=False):
        super().__init__()
        self.hparams = hparams
        self.model = SPSModel(hparams["MODEL"]["VOXEL_SIZE"])
        self.save_vis = save_vis
        self.test_seq = hparams.get("DATA", {}).get("SPLIT", {}).get("TEST")
        self.epsilon = hparams["FILTER"]["THRESHOLD"]
        self.loss = nn.MSELoss()
        self.predict_loss, self.predict_r2 = [], []
        self.dIoU, self.precision, self.recall, self.F1 = [], [], [], []
        self.data_size = data_size
        self.eval()

    def freeze(self):  # Lightning API used by the reference (scripts/predict.py:61, util.py:41)
        for p in self.parameters():
            p.requires_grad_(False)
        self.eval()

    def forward(self, batch):
        coordinates = batch[:, :5].reshape(-1, 5)   # models.py:57
        return self.model(coordinates)

    @staticmethod
    def r2score(pred, target):
        """torchmetrics.R2Score semantics: 1 - SS_res / SS_tot."""
        ss_res = torch.sum((target - pred) ** 2)
        ss_tot = torch.sum((target - target.mean()) ** 2)
        return 1 - ss_res / ss_tot

    @torch.no_grad()
    def predict_step(self, batch, batch_idx=0, dataloader_idx=0):
        coordinates = batch[:, :5].reshape(-1, 5)
        gt_labels = batch[:, 5].reshape(-1)
        scan_mask = coordinates[:, 4] == 1                 # models.py:87
        scores = self.model(coordinates)
        self.model.check()                                 # raises on out-of-range coordinates instead of scoring NaN
        if not scores.is_cuda:
            scores = scores.clone()                        # the host path returns a view of a reused pinned buffer
        scan_scores, scan_gt = scores[scan_mask.to(scores.device)], gt_labels[scan_mask].to(scores.device)
        loss = self.loss(scan_scores, scan_gt)
        r2 = self.r2score(scan_scores, scan_gt)
        self.predict_loss.append(loss)
        self.predict_r2.append(r2)
        pred = np.where(scan_scores.cpu().view(-1) < self.epsilon, 0, 1)   # models.py:97-98
        gt = np.where(scan_gt.cpu().view(-1) < self.epsilon, 0, 1)
        precision, recall, f1, accuracy, dIoU = util.calculate_metrics(gt, pred)
        self.dIoU.append(dIoU)
        self.precision.append(precision)
        self.recall.append(recall)
        self.F1.append(f1)
        return scores

    @torch.no_grad()
    def predict_scans(self, scans, submap, offsets=None):
        """``predict_step`` for a batch of raw scans (``SPSModel.predict_radius_async``: radius submaps, collation,
        forward and metric partials in the library): appends each scan's Loss / R2 / dIoU / Precision / Recall / F1 to
        the lists ``predict_step`` fills -- the values predict.py gets with ``batch_size=1`` -- and returns the scan
        rows' scores.  Scans without points add nothing."""
        scan_scores, counts, sums = self.model.predict_radius_async(scans, submap, self.epsilon, offsets=offsets).result()
        m = per_scan_metrics(counts, sums)
        self.predict_loss += m["Loss"]
        self.predict_r2 += m["R2"]
        self.dIoU += m["dIoU"]
        self.precision += m["Precision"]
        self.recall += m["Recall"]
        self.F1 += m["F1"]
        return scan_scores

    def summary(self):
        """scripts/predict.py:70-83: mean over per-batch values (not pooled counts)."""
        metrics = {"Loss": self.predict_loss, "R2": self.predict_r2, "dIoU": self.dIoU,
                   "Precision": self.precision, "Recall": self.recall, "F1": self.F1}
        return {k: float(sum(float(x) for x in v) / len(v)) for k, v in metrics.items() if len(v)}
