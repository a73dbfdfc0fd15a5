"""Batched voxel-prune submaps + collation + forward in the library (MapHash.prune_batch, SPSModel.infer_scans_async)
against the per-scan path the ROS node runs (c_ws/src/sps_filter/scripts/sps_node.py:111-120: util.prune, then
util.infer), oracle.prune and oracle.infer."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sps_oracle as O

pytestmark = pytest.mark.gpu

DS = 0.1


@pytest.fixture(scope="module")
def world():
    from sps_b200 import synth
    w = synth.World(2)
    base = synth.base_map(w, "hdl-32", n_poses=6, seed=2, voxel=DS).astype(np.float32)
    return w, base


@pytest.fixture(scope="module")
def map_hash(world):
    from sps_b200.engine import MapHash
    return MapHash(torch.as_tensor(world[1]).cuda(), DS)


@pytest.fixture(scope="module")
def state_dict():
    return O.make_state_dict(seed=0, randomize_bn=True)


def hdl_scans(w, base, variant=0):
    """B = 6 scans: a full hdl-32 scan, a truncated one, an empty one, one 500 m away from the map (no submap), the
    points of one with x, y < 0 (trunc, not floor, and the x ds round trip at negative coordinates), and one whose
    points all fall into the voxel of a map point, duplicates included."""
    from sps_b200 import synth
    full = synth.scan(w, "hdl-32", pose=(1.0, -2.0, 0.3 + variant), seed=5 + variant)
    part = synth.scan(w, "hdl-32", pose=(-0.5, 0.5, 1.1 + variant), seed=6 + variant)[: 30000 - 1000 * variant]
    far = synth.scan(w, "hdl-32", pose=(0.0, 0.0, 0.0), seed=7)[:5000] + np.float32(500.0)
    neg = synth.scan(w, "hdl-32", pose=(-1.0, -1.5, 2.0 + variant), seed=8)
    neg = neg[(neg[:, 0] < 0) & (neg[:, 1] < 0)]
    p = base[1234 + 17 * variant]
    jitter = p + np.random.default_rng([9, variant]).uniform(-0.02, 0.02, (400, 3)).astype(np.float32)
    same = jitter[np.all(O.to_coords(jitter, DS) == O.to_coords(p[None], DS), axis=1)][:40]
    one = np.vstack([np.repeat(p[None], 25, axis=0), same, same[:10]]).astype(np.float32)
    assert len(one) > 30 and len(np.unique(O.to_coords(one, DS), axis=0)) == 1
    return [full.astype(np.float32), part.astype(np.float32), np.zeros((0, 3), np.float32), far.astype(np.float32),
            neg.astype(np.float32), one]


def per_scan_reference(mh, scans_dev):
    """The per-scan path: MapHash.crop_voxel, util.infer's rows (batch column b), stacked; crop_voxel's counts."""
    rows, counts, subs = [], [], []
    for b, s in enumerate(scans_dev):
        sub, nuniq = mh.crop_voxel(s)
        data = torch.vstack([torch.hstack([s[:, :3], torch.ones(len(s), 1, device="cuda")]),
                             torch.hstack([sub, torch.zeros(len(sub), 1, device="cuda")])])
        rows.append(torch.hstack([torch.full((len(data), 1), float(b), device="cuda"), data]))
        counts.append((len(sub), nuniq))
        subs.append(sub)
    return torch.vstack(rows), counts, subs


@pytest.fixture
def pattern_sort(request):
    """Engines made inside the test use shape-sort mode `request.param` (sps_ctx_set_pattern_sort)."""
    from sps_b200 import engine
    old = engine.DEFAULTS["pattern_sort"]
    engine.set_defaults(pattern_sort=request.param)
    yield request.param
    engine.set_defaults(pattern_sort=old)


def make_model(state_dict, backend=None, lanes=3):
    from sps_b200.models import SPSModel
    model = SPSModel(DS)
    model.MinkUNet.load_state_dict({k: torch.as_tensor(v) for k, v in state_dict.items()})
    model = model.cuda().eval()
    model.lanes = lanes
    if backend is not None:
        model.set_conv_backend(backend)
    return model


def test_rows_bit_identical_to_the_per_scan_path(world, map_hash):
    w, base = world
    scans = hdl_scans(w, base)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    rows, roff, counts = map_hash.prune_batch(dev)
    ref, ref_counts, subs = per_scan_reference(map_hash, dev)
    assert rows.shape == ref.shape and rows.shape[1] == 5
    assert torch.equal(rows, ref)
    sizes = [len(s) + len(sub) for s, sub in zip(scans, subs)]
    assert roff.cpu().tolist() == np.concatenate([[0], np.cumsum(sizes)]).tolist()
    assert counts.dtype == torch.int32 and counts.cpu().tolist() == [list(c) for c in ref_counts]
    assert ref_counts[2] == (0, 0) and ref_counts[3][0] == 0 and ref_counts[3][1] > 0   # empty scan; far scan
    assert ref_counts[5] == (1, 1)                                                       # one voxel, in the map
    # every submap is util.prune's, bit for bit (oracle.prune), in first-occurrence order
    for s, sub, (m, nuniq) in zip(scans, subs, ref_counts):
        ref_sub, ref_n = O.prune(base, s, DS)
        assert (m, nuniq) == (len(ref_sub), ref_n)
        got = sub.cpu().numpy()
        assert (O.canonical(got.view(np.int32)) == O.canonical(ref_sub.view(np.int32))).all()
    # the other input forms: one concatenated tensor + offsets, pinned host tensors, wider rows
    offs = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).tolist()
    cat = torch.as_tensor(np.vstack(scans)).cuda()
    for got in (map_hash.prune_batch(cat, offs), map_hash.prune_batch([torch.as_tensor(s).pin_memory() for s in scans]),
                map_hash.prune_batch([torch.hstack([d, torch.full((len(d), 2), 7.0, device="cuda")]) for d in dev])):
        assert torch.equal(got[0], ref) and torch.equal(got[1], roff) and torch.equal(got[2], counts)


_ORACLE = {}


def oracle_scores(scans, subs, state_dict):
    """oracle.infer per scan on its own submap (computed once per module: the fp32 numpy forward is slow)."""
    if not _ORACLE:
        for b, (s, sub) in enumerate(zip(scans, subs)):
            if len(s):
                _ORACLE[b] = O.infer(s, sub.cpu().numpy(), DS, state_dict)
    return _ORACLE


@pytest.mark.parametrize("pattern_sort", [0, 2], indirect=True)
@pytest.mark.parametrize("backend", [0, 1])
def test_scores_match_forward_on_the_rows_and_the_oracle(world, map_hash, state_dict, pattern_sort, backend):
    w, base = world
    scans = hdl_scans(w, base)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    model = make_model(state_dict, backend)
    scan_scores, counts = model.infer_scans_async(dev, map_hash).result()
    rows, roff, ref_counts = map_hash.prune_batch(dev)
    ref = model(rows)
    model.check()
    assert scan_scores.shape == (sum(len(s) for s in scans),) and scan_scores.is_cuda
    assert torch.equal(scan_scores, ref[rows[:, 4] == 1])
    assert torch.equal(counts, ref_counts)
    _, _, subs = per_scan_reference(map_hash, dev)
    want = oracle_scores(scans, subs, state_dict)
    tol = 2e-3 if backend == 0 else 2e-5
    offs = np.concatenate([[0], np.cumsum([len(s) for s in scans])])
    got = scan_scores.cpu().numpy()
    for b, r in want.items():
        assert np.abs(got[offs[b]:offs[b + 1]] - r).max() < tol, b


def test_coordinate_out_of_key_range_raises_at_result(world, map_hash, state_dict):
    from sps_b200._cabi import SPS_ERR_COORD_RANGE, SpsError
    w, base = world
    scans = [torch.as_tensor(s).cuda() for s in hdl_scans(w, base)[:2]]
    scans[1] = scans[1].clone()
    scans[1][7, 0] = 2.0e4                        # 200 000 voxels of 0.1 m: past the key's x range
    model = make_model(state_dict)
    h = model.infer_scans_async(scans, map_hash)
    with pytest.raises(SpsError) as e:
        h.result()
    assert e.value.code == SPS_ERR_COORD_RANGE
    # the point is left out of the crop, like sps_submap_crop_voxel does
    _, _, counts = map_hash.prune_batch(scans)
    sub, nuniq = map_hash.crop_voxel(scans[1])
    assert counts[1].tolist() == [len(sub), nuniq]
    model.infer_scans_async(scans[:1], map_hash).result()     # the status word was cleared: the next call is fine


@pytest.mark.parametrize("on_device", [False, True])
def test_pipelined_calls_match_synchronous_calls(world, map_hash, state_dict, on_device):
    w, base = world
    batches = []
    for k in range(5):
        scans = hdl_scans(w, base, variant=k % 3)[k % 2:]
        batches.append([torch.as_tensor(s).cuda() if on_device else torch.as_tensor(s).pin_memory() for s in scans])
    model = make_model(state_dict, lanes=3)
    sync = [tuple(t.clone() for t in model.infer_scans_async(b, map_hash).result()) for b in batches]
    pending, got = [], []
    for b in batches:
        pending.append(model.infer_scans_async(b, map_hash))
        if len(pending) >= model.lanes:
            got.append(tuple(t.clone() for t in pending.pop(0).result()))
    got += [tuple(t.clone() for t in p.result()) for p in pending]
    assert len(got) == len(sync)
    for (a0, a1), (b0, b1) in zip(sync, got):
        assert a0.is_cuda == on_device
        assert torch.equal(a0, b0) and torch.equal(a1, b1)
    scores, counts = model.infer_scans_async(batches[0], map_hash).result()     # host scans: pinned host results
    assert scores.is_cuda == counts.is_cuda == on_device and scores.is_pinned() == counts.is_pinned() == (not on_device)


def test_full_size_config3_shape(state_dict):
    """Eight config-3 scans against the 1 M-voxel base map (above 400 000 rows, default settings): rows and scores bit
    for bit."""
    from sps_b200 import synth
    from sps_b200.engine import MapHash
    w = synth.World(0)
    traj = synth.loop_trajectory(radius=35.0, n=400)
    base = synth.base_map(w, "hdl-32", n_poses=400, seed=0, voxel=DS, trajectory=traj, target_voxels=1_000_000)
    scans = [torch.as_tensor(synth.scan(w, "hdl-32", traj(7 * i), seed=i)).cuda() for i in range(8)]
    mh = MapHash(torch.as_tensor(base).cuda(), DS)
    rows, roff, counts = mh.prune_batch(scans)
    assert len(rows) > 400_000
    ref, ref_counts, _ = per_scan_reference(mh, scans)
    assert torch.equal(rows, ref)
    assert counts.cpu().tolist() == [list(c) for c in ref_counts]
    model = make_model(state_dict, lanes=1)
    scan_scores, got_counts = model.infer_scans_async(scans, mh).result()
    want = model(rows)
    model.check()
    assert torch.equal(scan_scores, want[rows[:, 4] == 1])
    assert torch.equal(got_counts, counts)


def test_batch_size_limits_and_context_capacity(world, map_hash, state_dict):
    from sps_b200 import _cabi
    from sps_b200.engine import Engine, Net, _ptr, _stream
    w, base = world
    rng = np.random.default_rng(4)
    tiny = [base[rng.integers(0, len(base), 3)] + np.float32(0.01) for _ in range(255)]
    dev = [torch.as_tensor(t).cuda() for t in tiny]
    rows, roff, counts = map_hash.prune_batch(dev)
    ref, ref_counts, _ = per_scan_reference(map_hash, dev)
    assert torch.equal(rows, ref) and counts.cpu().tolist() == [list(c) for c in ref_counts]
    model = make_model(state_dict)
    scan_scores, got_counts = model.infer_scans_async(dev, map_hash).result()
    assert torch.equal(scan_scores, model(rows)[rows[:, 4] == 1]) and torch.equal(got_counts, counts)
    with pytest.raises(ValueError):
        model.infer_scans_async(dev + dev[:1], map_hash)
    with pytest.raises(ValueError):
        map_hash.prune_batch(dev + dev[:1])
    # only empty scans: no rows, zero counts
    empty = [torch.zeros((0, 3), device="cuda")] * 3
    scan_scores, got_counts = model.infer_scans_async(empty, map_hash).result()
    assert scan_scores.shape == (0,) and torch.all(got_counts == 0) and got_counts.shape == (3, 2)
    rows, roff, counts = map_hash.prune_batch(empty)
    assert rows.shape == (0, 5) and torch.all(roff == 0) and torch.all(counts == 0)
    # the C ABI: 2 n_total above the context's max_points
    lib = _cabi.load()
    n = 3 * 255
    eng = Engine(2 * n - 1, "cuda")
    net = Net(model.MinkUNet.state_dict(), "cuda")
    cat = torch.cat(dev)
    h_off = (C.c_int64 * 256)(*np.concatenate([[0], np.cumsum([3] * 255)]).tolist())
    nbytes = lib.sps_prune_batch_scratch_bytes(n, 255)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.empty((2 * n, 5), device="cuda")
    roff = torch.empty(256, dtype=torch.int32, device="cuda")
    n_rows = torch.empty(1, dtype=torch.int32, device="cuda")
    cnt = torch.empty((255, 2), dtype=torch.int32, device="cuda")
    sc = torch.empty(n, device="cuda")
    args = (net.handle, map_hash.handle, _ptr(cat), 3, h_off, 255, _ptr(out), _ptr(roff), _ptr(n_rows), _ptr(cnt),
            _ptr(scratch), nbytes, DS, _ptr(sc), _stream())
    assert lib.sps_infer_prune_batch(eng.handle, *args) == _cabi.SPS_ERR_CAPACITY
    eng2 = Engine(2 * n, "cuda")
    assert lib.sps_infer_prune_batch(eng2.handle, *args) == _cabi.SPS_OK
    assert lib.sps_ctx_status(eng2.handle, _stream()) == _cabi.SPS_OK
