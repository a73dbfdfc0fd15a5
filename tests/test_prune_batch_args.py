"""CPU-side checks of the batched voxel-prune entry points: bad arguments are rejected before any CUDA call."""
import ctypes as C

import pytest
import torch


def offsets(*v):
    return (C.c_int64 * len(v))(*v)


def test_prune_batch_argument_validation_without_gpu():
    from sps_b200 import _cabi
    lib = _cabi.load()
    BAD, CAP = _cabi.SPS_ERR_BAD_ARG, _cabi.SPS_ERR_CAPACITY
    assert lib.sps_prune_batch_scratch_bytes(524288, 8) > lib.sps_prune_batch_scratch_bytes(1000, 8) >= 4 * 1000
    assert lib.sps_prune_batch_scratch_bytes(0, 1) == lib.sps_prune_batch_scratch_bytes(1, 1) > 0
    nbytes = lib.sps_prune_batch_scratch_bytes(30, 2)
    fake = C.c_void_p(0x10000)         # never dereferenced: every call below fails validation first
    m, scans, rows, roff, nrows, counts, scratch = fake, fake, fake, fake, fake, fake, fake

    def call(m=m, scans=scans, ld=3, offs=offsets(0, 10, 30), batch=2, rows=rows, roff=roff, nrows=nrows, counts=counts,
             scratch=scratch, nbytes=nbytes):
        return lib.sps_prune_batch(m, scans, ld, offs, batch, rows, roff, nrows, counts, scratch, nbytes, None)

    assert call(m=None) == BAD
    assert call(scans=None) == BAD
    assert call(rows=None) == BAD and call(roff=None) == BAD and call(nrows=None) == BAD
    assert call(counts=None) == BAD and call(scratch=None) == BAD
    assert call(offs=None) == BAD
    assert call(ld=2) == BAD
    assert call(batch=0) == BAD and call(batch=256, offs=offsets(*range(257))) == BAD
    assert call(offs=offsets(1, 10, 30)) == BAD                    # must start at 0
    assert call(offs=offsets(0, 20, 10)) == BAD                    # must not decrease
    assert call(offs=offsets(0, 10, 0x40000000)) == BAD            # row indices are int32: 2 n_total must fit
    assert call(scratch=C.c_void_p(0x10010)) == BAD                # 256-byte alignment
    assert call(nbytes=nbytes - 1) == CAP
    # an empty batch needs no scan pointer; a bad one still fails on its other arguments
    assert call(scans=None, offs=offsets(0, 0, 0), nbytes=0) == CAP

    def fused(ctx=fake, net=fake, scores=fake, voxel=0.1, **kw):
        a = dict(m=m, scans=scans, ld=3, offs=offsets(0, 10, 30), batch=2, rows=rows, roff=roff, nrows=nrows,
                 counts=counts, scratch=scratch, nbytes=nbytes)
        a.update(kw)
        return lib.sps_infer_prune_batch(ctx, net, a["m"], a["scans"], a["ld"], a["offs"], a["batch"], a["rows"],
                                         a["roff"], a["nrows"], a["counts"], a["scratch"], a["nbytes"], voxel, scores, None)

    assert fused(ctx=None) == BAD and fused(net=None) == BAD and fused(scores=None) == BAD
    assert fused(voxel=0.0) == BAD and fused(voxel=-0.1) == BAD
    assert fused(m=None) == BAD and fused(scans=None) == BAD and fused(rows=None) == BAD and fused(roff=None) == BAD
    assert fused(nrows=None) == BAD and fused(counts=None) == BAD and fused(scratch=None) == BAD
    assert fused(ld=2) == BAD and fused(batch=0) == BAD and fused(batch=256, offs=offsets(*range(257))) == BAD
    assert fused(offs=offsets(1, 10, 30)) == BAD and fused(offs=offsets(0, 20, 10)) == BAD
    assert fused(offs=offsets(0, 10, 0x40000000)) == BAD
    assert fused(scratch=C.c_void_p(0x10010)) == BAD
    assert fused(nbytes=nbytes - 1) == CAP
    # (2 n_total above the context's max_points -> SPS_ERR_CAPACITY needs a real context: tests/test_gpu_prune_batch.py)


def test_batch_parts_min_width():
    from sps_b200.datasets import batch_parts
    parts, offs, ld = batch_parts([torch.zeros(3, 3), torch.zeros(0, 3)], min_width=3)
    assert offs == [0, 3, 3] and ld == 3 and len(parts) == 2
    parts, offs, ld = batch_parts(torch.zeros(8, 5), [0, 3, 8], min_width=3)
    assert offs == [0, 3, 8] and ld == 5
    with pytest.raises(ValueError):
        batch_parts([torch.zeros(3, 3)])                           # the default still needs the label column
    with pytest.raises(ValueError):
        batch_parts([torch.zeros(3, 2)], min_width=3)
    with pytest.raises(ValueError):
        batch_parts([torch.zeros(1, 3)] * 256, min_width=3)
