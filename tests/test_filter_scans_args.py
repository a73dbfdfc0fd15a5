"""CPU-side checks of the batched sensor-frame filter call (sps_filter_scans_batch, SPSModel.filter_scans_async): bad
arguments are rejected before any CUDA call."""
import ctypes as C

import numpy as np
import pytest
import torch


def offsets(*v):
    return (C.c_int64 * len(v))(*v)


def test_filter_scans_batch_argument_validation_without_gpu():
    from sps_b200 import _cabi
    lib = _cabi.load()
    BAD, CAP = _cabi.SPS_ERR_BAD_ARG, _cabi.SPS_ERR_CAPACITY
    assert lib.sps_filter_scans_batch_scratch_bytes(524288, 8) > lib.sps_filter_scans_batch_scratch_bytes(1000, 8)
    assert lib.sps_filter_scans_batch_scratch_bytes(0, 1) == lib.sps_filter_scans_batch_scratch_bytes(1, 1) > 0
    # the map-frame xyz, the prune carve and the filter's ranks come on top of sps_prune_batch's scratch
    prune = lib.sps_prune_batch_scratch_bytes(1000, 8)
    assert lib.sps_filter_scans_batch_scratch_bytes(1000, 8) >= prune + 1000 * (12 + 4)
    nbytes = lib.sps_filter_scans_batch_scratch_bytes(30, 2)
    fake = C.c_void_p(0x10000)         # never dereferenced: every call below fails validation first

    def call(ctx=fake, net=fake, m=fake, scans=fake, ld=4, offs=offsets(0, 10, 30), batch=2, poses=fake, eps=0.84,
             voxel=0.1, rows=fake, roff=fake, nrows=fake, counts=fake, scores=fake, mcounts=fake, msums=fake, kept=fake,
             koff=fake, scratch=fake, nbytes=nbytes):
        return lib.sps_filter_scans_batch(ctx, net, m, scans, ld, offs, batch, poses, eps, voxel, rows, roff, nrows,
                                          counts, scores, mcounts, msums, kept, koff, scratch, nbytes, None)

    # the arguments sps_infer_prune_batch checks
    assert call(ctx=None) == BAD and call(net=None) == BAD and call(m=None) == BAD and call(scans=None) == BAD
    assert call(rows=None) == BAD and call(roff=None) == BAD and call(nrows=None) == BAD and call(counts=None) == BAD
    assert call(scores=None) == BAD and call(scratch=None) == BAD and call(offs=None) == BAD
    assert call(voxel=0.0) == BAD and call(voxel=-0.1) == BAD and call(voxel=float("nan")) == BAD
    assert call(batch=0) == BAD and call(batch=256, offs=offsets(*range(257))) == BAD
    assert call(offs=offsets(1, 10, 30)) == BAD                    # must start at 0
    assert call(offs=offsets(0, 20, 10)) == BAD                    # must not decrease
    assert call(offs=offsets(0, 10, 0x40000000)) == BAD            # row indices are int32: 2 n_total must fit
    assert call(scratch=C.c_void_p(0x10010)) == BAD                # 256-byte alignment
    # the filter's own arguments
    assert call(ld=3) == BAD                                       # column 3 is the intensity / label
    assert call(poses=None) == BAD
    assert call(kept=None) == BAD and call(koff=None) == BAD
    assert call(mcounts=None) == BAD and call(msums=None) == BAD
    for misaligned in (0x10004, 0x10008, 0x1000c):                 # the published rows are written as float4
        assert call(kept=C.c_void_p(misaligned)) == BAD
    assert call(eps=float("nan")) == BAD
    # scratch: sps_prune_batch's size is not enough
    assert call(nbytes=nbytes - 1) == CAP
    assert call(nbytes=lib.sps_prune_batch_scratch_bytes(30, 2)) == CAP
    # an empty batch needs no scan pointer; a bad one still fails on its other arguments
    assert call(scans=None, offs=offsets(0, 0, 0), nbytes=0) == CAP
    assert call(scans=None, offs=offsets(0, 0, 0), poses=None) == BAD
    # (2 n_total above the context's max_points -> SPS_ERR_CAPACITY needs a real context: tests/test_gpu_filter_scans.py)


def test_filter_scans_async_checks_scans_and_poses_before_the_device():
    from sps_b200.models import FilteredScans, SPSModel
    model = SPSModel(0.1).eval()
    scans = [torch.zeros(5, 4), torch.zeros(0, 4), torch.zeros(3, 4)]
    eye = np.repeat(np.eye(4)[None], 3, axis=0)
    with pytest.raises(ValueError):
        model.filter_scans_async([s[:, :3] for s in scans], eye, None, 0.5)        # no intensity / label column
    with pytest.raises(ValueError):
        model.filter_scans_async(scans, eye[:2], None, 0.5)                       # one pose per scan
    with pytest.raises(ValueError):
        model.filter_scans_async(scans, eye.astype(np.float32), None, 0.5)        # float64, as util.to_tr_matrix builds it
    with pytest.raises(ValueError):
        model.filter_scans_async(scans, eye.reshape(3, 16), None, 0.5)
    with pytest.raises(ValueError):
        model.filter_scans_async([torch.zeros(1, 4)] * 256, np.repeat(np.eye(4)[None], 256, axis=0), None, 0.5)
    with pytest.raises(ValueError):
        model.filter_scans_async(torch.zeros(8, 4), eye, None, 0.5)               # one tensor needs its offsets
    # valid arguments get as far as the device check: there is no CPU path
    with pytest.raises(RuntimeError):
        model.filter_scans_async(scans, eye, None, 0.5)
    with pytest.raises(RuntimeError):
        model.filter_scans_async(torch.zeros(8, 4), torch.as_tensor(eye), None, 0.5, offsets=[0, 5, 5, 8])
    assert FilteredScans._fields == ("scan_scores", "kept", "kept_offsets", "counts", "metric_counts", "metric_sums")
