"""CPU-side checks of the batched radius-submap entry points: bad arguments are rejected before any CUDA call."""
import ctypes as C

import pytest
import torch


def offsets(*v):
    return (C.c_int64 * len(v))(*v)


def test_radius_batch_argument_validation_without_gpu():
    from sps_b200 import _cabi
    lib = _cabi.load()
    BAD, CAP = _cabi.SPS_ERR_BAD_ARG, _cabi.SPS_ERR_CAPACITY
    assert lib.sps_radius_batch_scratch_bytes(524288, 8) > lib.sps_radius_batch_scratch_bytes(1000, 8) >= 4 * 1000
    nbytes = lib.sps_radius_batch_scratch_bytes(30, 2)
    fake = C.c_void_p(0x10000)         # never dereferenced: every call below fails validation first
    bm, scans, rows, roff, nrows, scratch = fake, fake, fake, fake, fake, fake

    def call(bm=bm, scans=scans, ld=4, offs=offsets(0, 10, 30), batch=2, rows=rows, cap=100, roff=roff, nrows=nrows,
             scratch=scratch, nbytes=nbytes):
        return lib.sps_radius_batch(bm, scans, ld, offs, batch, rows, cap, roff, nrows, scratch, nbytes, None)

    assert call(bm=None) == BAD
    assert call(scans=None) == BAD
    assert call(rows=None) == BAD and call(roff=None) == BAD and call(nrows=None) == BAD and call(scratch=None) == BAD
    assert call(offs=None) == BAD
    assert call(ld=3) == BAD
    assert call(batch=0) == BAD and call(batch=256, offs=offsets(*range(257))) == BAD
    assert call(offs=offsets(1, 10, 30)) == BAD                    # must start at 0
    assert call(offs=offsets(0, 20, 10)) == BAD                    # must not decrease
    assert call(scratch=C.c_void_p(0x10010)) == BAD                # 256-byte alignment
    assert call(cap=-1) == BAD
    assert call(nbytes=nbytes - 1) == CAP
    # an empty batch needs no scan pointer; a bad one still fails on its other arguments
    assert call(scans=None, offs=offsets(0, 0, 0), nbytes=0) == CAP

    def fused(ctx=fake, net=fake, scores=fake, counts=fake, sums=fake, voxel=0.1, **kw):
        a = dict(bm=bm, scans=scans, ld=4, offs=offsets(0, 10, 30), batch=2, rows=rows, cap=100, roff=roff, nrows=nrows,
                 scratch=scratch, nbytes=nbytes)
        a.update(kw)
        return lib.sps_predict_radius_batch(ctx, net, a["bm"], a["scans"], a["ld"], a["offs"], a["batch"], a["rows"],
                                            a["cap"], a["roff"], a["nrows"], a["scratch"], a["nbytes"], voxel, 0.84,
                                            scores, counts, sums, None)

    assert fused(ctx=None) == BAD and fused(net=None) == BAD
    assert fused(scores=None) == BAD and fused(counts=None) == BAD and fused(sums=None) == BAD
    assert fused(voxel=0.0) == BAD
    assert fused(bm=None) == BAD and fused(ld=3) == BAD and fused(batch=0) == BAD
    assert fused(offs=offsets(0, 20, 10)) == BAD and fused(scratch=C.c_void_p(0x10010)) == BAD
    assert fused(nbytes=nbytes - 1) == CAP


def test_batch_parts_normalises_both_input_forms():
    from sps_b200.datasets import batch_parts
    a, b = torch.zeros(3, 4), torch.ones(5, 4)
    parts, offs, ld = batch_parts([a, torch.zeros(0, 4), b])
    assert offs == [0, 3, 3, 8] and ld == 4 and [s for _, s in parts] == [0, 3, 3]
    parts, offs, ld = batch_parts(torch.zeros(8, 6), [0, 3, 8])
    assert offs == [0, 3, 8] and ld == 6 and len(parts) == 1
    with pytest.raises(ValueError):
        batch_parts(torch.zeros(8, 4))                     # offsets missing
    with pytest.raises(ValueError):
        batch_parts(torch.zeros(8, 4), [0, 3, 7])          # do not cover the tensor
    with pytest.raises(ValueError):
        batch_parts(torch.zeros(8, 4), [0, 5, 3, 8])       # decreasing
    with pytest.raises(ValueError):
        batch_parts([a, torch.zeros(2, 6)])                # widths differ
    with pytest.raises(ValueError):
        batch_parts([torch.zeros(2, 3)])                   # no label column
    with pytest.raises(ValueError):
        batch_parts([a] * 256)                             # more scans than batch indices
