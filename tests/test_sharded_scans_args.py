"""CPU-side checks of the batch-sharded sequence calls (parallel.ShardPlan / ShardedScans) and of the segment
reassembly (sps_gather_segments): the batch -> rank assignment, the buffer sizes, and bad arguments rejected before any
CUDA call."""
import ctypes as C

import numpy as np
import pytest
import torch


def test_batch_to_rank_assignment_and_capacities():
    from sps_b200.parallel import ShardPlan
    sizes = [5, 0, 7, 3, 4, 9, 2]                       # S = 7, B = 2: batches (0,1) (2,3) (4,5) (6)
    p = ShardPlan(sizes, 2, 3)
    assert p.bounds == [(0, 2), (2, 4), (4, 6), (6, 7)]
    assert p.owner == [0, 1, 2, 0] and p.batches(0) == [0, 3] and p.batches(1) == [1] and p.batches(2) == [2]
    assert p.rows == [5, 10, 13, 2]
    # rank 0 holds batches 0 and 3 back to back: rows 0..4 and 5..6, scans 0..1 and 2
    assert p.row_start == [0, 0, 0, 5] and p.slot_start == [0, 0, 0, 2]
    assert p.cap == 13 and p.slots == 3                 # the largest rank block: rank 2's 13 rows, rank 0's 3 scans
    assert p.scan_index == [0, 1, 3, 4, 6, 7, 2]        # scan i -> rank * slots + slot
    # fewer batches than ranks: the others hold nothing
    p = ShardPlan([4, 4, 4], 8, 4)
    assert p.bounds == [(0, 3)] and p.owner == [0] and p.batches(1) == [] and p.cap == 12 and p.slots == 3
    # one rank: every batch in order, the plan of the single-process loop
    p = ShardPlan(sizes, 3, 1)
    assert p.owner == [0, 0, 0] and p.row_start == [0, 12, 28] and p.cap == 30 and p.scan_index == list(range(7))
    # every scan lands in exactly one slot, whatever the world size
    rng = np.random.default_rng(0)
    sizes = rng.integers(0, 50, 101).tolist()
    for world in range(1, 9):
        for B in (1, 4, 255):
            p = ShardPlan(sizes, B, world)
            assert sorted(p.scan_index) == sorted(set(p.scan_index)) and len(p.scan_index) == len(sizes)
            assert max(p.scan_index) < world * p.slots
            assert all(p.row_start[k] + p.rows[k] <= p.cap for k in range(len(p.bounds)))
            assert sum(p.rows) == sum(sizes)


def test_sharded_scans_python_argument_rules():
    from sps_b200.models import SPSModel
    from sps_b200.parallel import ShardedScans
    model = SPSModel(0.1).eval()
    for bad in (0, 256, -1):
        with pytest.raises(ValueError):
            ShardedScans(model, 0.5, bad)
    ShardedScans(model, 0.5, 1)
    ss = ShardedScans(model, 0.5, 255)
    scans = [torch.zeros(5, 4), torch.zeros(0, 4), torch.zeros(3, 4)]
    eye = np.repeat(np.eye(4)[None], 3, axis=0)
    with pytest.raises(ValueError):
        ss.replay(scans, eye[:2], None)                               # one pose per scan
    with pytest.raises(ValueError):
        ss.replay(scans[:2], eye, None)
    with pytest.raises(ValueError):
        ss.replay(scans, eye.astype(np.float32), None)                # float64, as util.to_tr_matrix builds it
    with pytest.raises(ValueError):
        ss.replay(scans, eye.reshape(3, 16), None)
    with pytest.raises(ValueError):
        ss.replay([s[:, :3] for s in scans], eye, None)               # no intensity / label column
    with pytest.raises(ValueError):
        ss.evaluate([s[:, :3] for s in scans], None)
    with pytest.raises(ValueError):
        ss.evaluate(torch.zeros(8, 4), None)                          # a list of scans, not one tensor
    with pytest.raises(ValueError):
        ss.evaluate([], None)
    # valid arguments get as far as the device check: there is no CPU path
    with pytest.raises(RuntimeError):
        ss.replay(scans, eye, None)
    with pytest.raises(RuntimeError):
        ss.evaluate(scans, None)


def test_gather_segments_wrapper_needs_cuda_tensors():
    from sps_b200.parallel import gather_segments
    src, out = torch.zeros((2, 9, 4)), torch.zeros((11, 4))
    lens, offs = torch.zeros(3, dtype=torch.int32), torch.zeros(4, dtype=torch.int32)
    with pytest.raises(ValueError):                                   # host tensors: there is no CPU path
        gather_segments(src, [1, 0, 0], [4, 0, 6], [3, 5, 3], lens, out, offs)
    with pytest.raises(ValueError):                                   # one entry per segment in each host list
        gather_segments(src, [1, 0, 0], [4, 0], [3, 5, 3], lens, out, offs)
    with pytest.raises(ValueError):                                   # out rows of the source rows' width
        gather_segments(src, [1, 0, 0], [4, 0, 6], [3, 5, 3], lens, torch.zeros((11, 2)), offs)


def arr(ctype, *v):
    return (ctype * max(len(v), 1))(*v)


def test_gather_segments_argument_validation_without_gpu():
    from sps_b200 import _cabi
    lib = _cabi.load()
    BAD, CAP = _cabi.SPS_ERR_BAD_ARG, _cabi.SPS_ERR_CAPACITY
    fake = C.c_void_p(0x10000)         # never dereferenced: every call below fails validation first

    def call(src=fake, world=2, cap=10, width=4, n_seg=3, rank=(0, 1, 0), start=(0, 0, 6), rows=(6, 10, 4), lens=fake,
             out=fake, out_cap=20, offs=fake):
        return lib.sps_gather_segments(src, world, cap, width, n_seg, arr(C.c_int32, *rank), arr(C.c_int64, *start),
                                       arr(C.c_int64, *rows), lens, out, out_cap, offs, None)

    assert call(world=0) == BAD and call(cap=-1) == BAD and call(width=0) == BAD and call(n_seg=-1) == BAD
    assert call(out_cap=-1) == BAD and call(offs=None) == BAD
    assert call(src=None) == BAD and call(out=None) == BAD and call(lens=None) == BAD
    assert lib.sps_gather_segments(fake, 2, 10, 4, 3, None, arr(C.c_int64, 0, 0, 6), arr(C.c_int64, 6, 10, 4), fake, fake,
                                   20, fake, None) == BAD
    assert lib.sps_gather_segments(fake, 2, 10, 4, 3, arr(C.c_int32, 0, 1, 0), None, arr(C.c_int64, 6, 10, 4), fake, fake,
                                   20, fake, None) == BAD
    assert lib.sps_gather_segments(fake, 2, 10, 4, 3, arr(C.c_int32, 0, 1, 0), arr(C.c_int64, 0, 0, 6), None, fake, fake,
                                   20, fake, None) == BAD
    assert call(rank=(0, 2, 0)) == BAD and call(rank=(0, -1, 0)) == BAD          # ranks 0 .. world - 1
    assert call(start=(0, -1, 6)) == BAD and call(rows=(6, -1, 4)) == BAD
    assert call(start=(0, 0, 7)) == BAD and call(rows=(6, 11, 4)) == BAD         # start + rows within the block
    assert call(start=(0, 0, 11), rows=(6, 10, 0)) == BAD                        # a start past the block
    for misaligned in ("src", "out", "lens", "offs"):                            # 4-byte elements
        assert call(**{misaligned: C.c_void_p(0x10002)}) == BAD
    assert call(cap=1 << 58) == BAD                                              # world * cap * width beyond 2^59
    assert call(world=1, cap=1 << 31, n_seg=2, rank=(0, 0), start=(0, 0), rows=(1 << 30, 1 << 30),
                out_cap=1 << 32) == BAD                                          # int32 offsets: sum of rows < 2^31
    assert call(out_cap=19) == CAP                                               # room for every segment full
    # segments that hold no rows need no source or output, but the offsets are always written
    assert call(src=None, out=None, rows=(0, 0, 0), out_cap=0, offs=None) == BAD
