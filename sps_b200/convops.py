"""Python entry to the layer-level C-ABI call ``sps_conv_fwd`` (used by the ME-shaped layer
shim and by the layer-wise parity tests).  All tensors are CUDA fp32/int32; nothing is computed
in torch."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _cabi
from ._cabi import check
from .engine import _ptr, _stream


def pack_kmajor(weight: torch.Tensor, weight2: torch.Tensor | None = None) -> torch.Tensor:
    """ME-layout ``[K,Cin,Cout]`` (+ fused 1x1 ``[Cin2,Cout]``) -> K-major TF32 matrix for the
    tcgen05 kernel (host-side packing in the library, result on the weights' device)."""
    lib = _cabi.load()
    w = np.ascontiguousarray(weight.detach().cpu().numpy(), np.float32)
    K, cin, cout = w.shape
    w2 = None if weight2 is None else np.ascontiguousarray(weight2.detach().cpu().numpy(), np.float32)
    cin2 = 0 if w2 is None else w2.shape[0]
    ld = lib.sps_conv_kmajor_ld(K, cin, cin2)
    out = np.empty((cout, ld), np.float32)
    check(lib.sps_conv_pack_kmajor(w.ctypes.data_as(C.c_void_p), K, cin, cout,
                                   None if w2 is None else w2.ctypes.data_as(C.c_void_p), cin2,
                                   out.ctypes.data_as(C.c_void_p)), "sps_conv_pack_kmajor")
    return torch.as_tensor(out).to(weight.device)


def pack_kmajor_f16(weight: torch.Tensor, weight2: torch.Tensor | None = None) -> torch.Tensor:
    """fp16 twin of :func:`pack_kmajor` (``sps_conv_pack_kmajor_f16``): the weight matrix of the fp16-row path."""
    lib = _cabi.load()
    w = np.ascontiguousarray(weight.detach().cpu().numpy(), np.float32)
    K, cin, cout = w.shape
    w2 = None if weight2 is None else np.ascontiguousarray(weight2.detach().cpu().numpy(), np.float32)
    cin2 = 0 if w2 is None else w2.shape[0]
    ld = lib.sps_conv_kmajor_ld_f16(K, cin, cin2)
    out = np.empty((cout, ld), np.float16)
    check(lib.sps_conv_pack_kmajor_f16(w.ctypes.data_as(C.c_void_p), K, cin, cout,
                                       None if w2 is None else w2.ctypes.data_as(C.c_void_p), cin2,
                                       out.ctypes.data_as(C.c_void_p)), "sps_conv_pack_kmajor_f16")
    return torch.as_tensor(out).to(weight.device)


def pack_kmajor_f16x(weight: torch.Tensor, weight2: torch.Tensor | None = None, in_split=False, in2_split=False,
                     fold_lo=False, cin_split=0) -> torch.Tensor:
    """``sps_conv_pack_kmajor_f16x``: the fp16 weight matrix with the precision options of the fused forward --
    ``in_split`` / ``in2_split``: the rows of ``in`` / ``in2`` are hi|lo pairs (weights duplicated along K);
    ``fold_lo`` (cout == 8): rows 8..15 hold the low parts of the weights (SPS_CONV_FOLD_LO); ``cin_split``: the rows are two
    channel segments (``sps_conv_args.cin_split``, ``sps_conv_pack_kmajor_f16s``)."""
    lib = _cabi.load()
    w = np.ascontiguousarray(weight.detach().cpu().numpy(), np.float32)
    K, cin, cout = w.shape
    w2 = None if weight2 is None else np.ascontiguousarray(weight2.detach().cpu().numpy(), np.float32)
    cin2 = 0 if w2 is None else w2.shape[0]
    flags = (1 if in_split else 0) | (2 if in2_split else 0) | (4 if fold_lo else 0)
    ld = lib.sps_conv_kmajor_ld_f16s(K, cin, cin2, flags, int(cin_split))
    out = np.zeros((16 if fold_lo else cout, ld), np.float16)
    check(lib.sps_conv_pack_kmajor_f16s(w.ctypes.data_as(C.c_void_p), K, cin, cout,
                                        None if w2 is None else w2.ctypes.data_as(C.c_void_p), cin2, flags, int(cin_split),
                                        out.ctypes.data_as(C.c_void_p)), "sps_conv_pack_kmajor_f16s")
    return torch.as_tensor(out).to(weight.device)


def split_rows(x: torch.Tensor) -> torch.Tensor:
    """fp32 [V, C] (C multiple of 8) -> the hi|lo row format of SPS_CONV_OUT_SPLIT: fp16 [V, 2C], per 8 channels
    [fp16(v) x 8 | fp16(v - hi) x 8] (test helper: the kernels produce this format themselves)."""
    V, Cc = x.shape
    hi = x.to(torch.float16)
    lo = (x - hi.float()).to(torch.float16)
    return torch.stack([hi.reshape(V, Cc // 8, 8), lo.reshape(V, Cc // 8, 8)], dim=2).reshape(V, 2 * Cc).contiguous()


def merge_rows(x2: torch.Tensor) -> torch.Tensor:
    """Inverse of :func:`split_rows`: fp16 hi|lo rows [V, 2C] -> fp32 [V, C]."""
    V, C2 = x2.shape
    g = x2.float().reshape(V, C2 // 16, 2, 8)
    return (g[:, :, 0] + g[:, :, 1]).reshape(V, C2 // 2)


def _addr(x):
    """Device address of a CUDA tensor, or a raw device pointer (an ``Engine.level`` view field) as it is; None -> NULL."""
    if x is None or isinstance(x, int):
        return x
    return x.data_ptr()


def kernel_map_tile_masks(map, map_ld, K, n_out, n_out_max):
    """Present-offset bitmask per 128-row tile of a dense kernel map (tensor-core path input).  ``map``: a CUDA tensor
    or a device pointer."""
    lib = _cabi.load()
    masks = torch.zeros(((n_out_max + 127) // 128 + 1, 4), dtype=torch.int32, device=n_out.device)
    check(lib.sps_kernel_map_tile_masks(C.c_void_p(_addr(map)), int(map_ld), int(K), _ptr(n_out), int(n_out_max), _ptr(masks),
                                        _stream()), "sps_kernel_map_tile_masks")
    return masks


def conv_fwd(inp, weight, n_out, *, map=None, map_ld=0, mode=_cabi.SPS_CONV_NBR, shift=None, in2=None, weight2=None,
             res=None, relu=False, out=None, head_w=None, head_b=0.0, head_out=None, weight_kmajor=None,
             round_out=False, n_out_max=None, backend=None, tile_mask=None, io_f16=False, flags=0, cin_rows=None, cin2_rows=None, cin_split=0,
             perm=None, tile_slices=None):
    """out[o] = act(sum_k in[map[k][o]] @ W[k] (+ in2[o] @ W2) + shift (+ res[o])); ``n_out`` is a
    1-element int32 CUDA tensor (device-side count).  ``inp``/``out``/``in2``/``res`` may be
    channel slices (stride(0) is the leading dimension).  ``io_f16``: ``inp``/``in2``/``res``/``out`` are fp16
    rows and ``weight_kmajor`` comes from :func:`pack_kmajor_f16` (SPS_IO_F16, the fused forward's format).
    ``flags``: SPS_CONV_FOLD_LO / SPS_CONV_OUT_SPLIT; ``cin_rows`` / ``cin2_rows``: channel counts the kernel sees when the rows are
    hi|lo pairs (2 x the weight's).  ``backend``: SPS_BACKEND_* of this one call (default AUTO) -- the library has no
    process-wide switch.  ``perm`` / ``tile_mask`` / ``tile_slices``: a processing order of the output rows, the tile
    masks in that order and, optionally, the kernel map gathered per tile (``map`` may then be None) -- what
    ``Engine.level`` hands out after a shape-sorted pass.  ``map``, ``tile_mask``, ``perm`` and ``tile_slices`` take CUDA
    tensors or raw device pointers."""
    lib = _cabi.load()
    K = weight.shape[0] if weight.dim() == 3 else 1
    cin, cout = weight.shape[-2], weight.shape[-1]
    if n_out_max is None:
        n_out_max = int(n_out.item())
    if out is None and head_out is None:
        width = 2 * cout if (flags & _cabi.SPS_CONV_OUT_SPLIT) else cout
        out = torch.empty((max(n_out_max, 1), width), dtype=torch.float16 if io_f16 else torch.float32, device=inp.device)
    a = _cabi.ConvArgs()
    a.mode, a.K, a.cin, a.cout = mode, K, cin, cout
    a.map, a.map_ld = _addr(map), int(map_ld)
    a.n_out, a.n_out_max = n_out.data_ptr(), int(n_out_max)
    a.in_, a.in_ld = inp.data_ptr(), inp.stride(0)
    a.weight = weight.data_ptr()
    a.shift = shift.data_ptr() if shift is not None else None
    if in2 is not None:
        a.in2, a.in2_ld, a.cin2, a.weight2 = in2.data_ptr(), in2.stride(0), weight2.shape[0], weight2.data_ptr()
    if res is not None:
        a.res, a.res_ld = res.data_ptr(), res.stride(0)
    a.relu = int(relu)
    if out is not None:
        a.out, a.out_ld = out.data_ptr(), out.stride(0)
    if head_out is not None:
        a.head_w, a.head_b, a.head_out = head_w.data_ptr(), float(head_b), head_out.data_ptr()
    if weight_kmajor is not None:
        a.weight_kmajor, a.kmajor_ld = weight_kmajor.data_ptr(), weight_kmajor.stride(0)
    a.round_out = int(round_out)
    a.io_dtype = _cabi.SPS_IO_F16 if io_f16 else _cabi.SPS_IO_F32
    a.backend = int(backend) if backend is not None else _cabi.SPS_BACKEND_AUTO
    a.flags = int(flags)
    a.cin_split = int(cin_split)
    if cin_rows is not None:   # hi|lo input rows: the kernel sees the doubled channel count
        a.cin = int(cin_rows)
    if cin2_rows is not None:
        a.cin2 = int(cin2_rows)
    if weight_kmajor is not None and map is not None and tile_mask is None and perm is None and K <= 81:
        tile_mask = kernel_map_tile_masks(map, map_ld, K, n_out, n_out_max)
    a.tile_mask, a.perm, a.tile_slices = _addr(tile_mask), _addr(perm), _addr(tile_slices)
    with torch.cuda.device(inp.device):
        check(lib.sps_conv_fwd(C.byref(a), _stream()), "sps_conv_fwd")
    return out if out is not None else head_out
