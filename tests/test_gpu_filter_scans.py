"""The ROS node's callback for a batch of sensor-frame scans in one library call (sps_filter_scans_batch,
SPSModel.filter_scans_async) against the per-scan composition the node runs (sps_node.py:88-176):
util.transform_point_cloud, MapHash.prune_batch / infer_scans_async, the metric partials of parallel.device_partials
and util.filter_scan / oracle.filter_scan."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sps_oracle as O

pytestmark = pytest.mark.gpu

DS = 0.1


def translate(T, t):
    T = T.copy()
    T[:3, 3] = t
    return T


def rotation(ax, ay, az):
    """Rotation about x, then y, then z (radians) as a 4x4 float64 matrix."""
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    T = np.eye(4)
    T[:3, :3] = Rz @ Ry @ Rx
    return T


def distinct_poses(variant=0):
    """One pose per scan of hdl_scans, all different: the identity, a yaw plus a translation, a rotation about all three
    axes plus a translation, a matrix whose homogeneous row is not (0, 0, 0, 1), and two more rigid motions."""
    v = 0.1 * variant
    homog = translate(rotation(0.05, -0.1, 0.4 + v), (0.5, -0.25, 0.1))
    homog[3] = (2e-4, -1e-4, 3e-4, 1.02)
    return np.stack([np.eye(4),
                     translate(rotation(0, 0, 0.7 + v), (3.0, -2.0, 0.5)),
                     translate(rotation(0.3, -0.2, 1.1 + v), (-1.5, 2.5, -0.3)),
                     homog,
                     translate(rotation(0, 0, -2.0 + v), (0.2, 0.1, -0.1)),
                     translate(rotation(-0.05, 0.04, -2.5 + v), (1.0, 1.0, 0.2))]).astype(np.float64)


def to_sensor(xyz, T):
    """The map-frame points of a scan moved into the sensor frame of pose T (float64 inverse, homogeneous divide)."""
    h = np.hstack([xyz.astype(np.float64), np.ones((len(xyz), 1))]) @ np.linalg.inv(T).T
    return (h[:, :3] / h[:, 3:]).astype(np.float32)


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


def hdl_scans(w, base, poses, variant=0):
    """The B = 6 map-frame cases of test_gpu_prune_batch (full, truncated, empty, 500 m from the map, x, y < 0, one voxel)
    moved into the sensor frames of `poses`, with an intensity / label column (0, 1 or in between)."""
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
    rng = np.random.default_rng([10, variant])
    out = []
    for xyz, T in zip([full, part, np.zeros((0, 3), np.float32), far, neg, one], poses):
        n = len(xyz)
        label = np.where(rng.random(n) < 0.5, rng.integers(0, 2, n), rng.random(n)).astype(np.float32)
        out.append(np.hstack([to_sensor(xyz[:, :3], T), label[:, None]]).astype(np.float32))
    return out


def map_frame(dev, poses):
    """util.transform_point_cloud per scan (sps_transform_points), as the node does it."""
    from sps_b200 import util
    return [util.transform_point_cloud(s, T) if len(s) else torch.zeros((0, 3), device="cuda")
            for s, T in zip(dev, poses)]


def filtered_reference(dev, scan_scores, eps):
    """util.filter_scan per scan, concatenated, and the per-scan offsets."""
    from sps_b200 import util
    kept, offs, start = [], [0], 0
    for s in dev:
        n = len(s)
        buf, count = util.filter_scan(s, scan_scores[start:start + n], eps)
        kept.append(buf[:int(count.item())])
        offs.append(offs[-1] + int(count.item()))
        start += n
    return torch.vstack(kept), offs


def partials_reference(dev, scan_scores, eps):
    """parallel.device_partials on per-scan (b, x, y, z, t = 1, label) rows."""
    from sps_b200 import parallel
    counts, sums, start = [], [], 0
    for b, s in enumerate(dev):
        n = len(s)
        if n == 0:
            counts.append(torch.zeros(4, dtype=torch.int64, device="cuda"))
            sums.append(torch.zeros(5, dtype=torch.float64, device="cuda"))
            continue
        rows = torch.hstack([torch.full((n, 1), float(b), device="cuda"), s[:, :3], torch.ones((n, 1), device="cuda"),
                             s[:, 3:4]]).contiguous()
        c, sm = parallel.device_partials(scan_scores[start:start + n].contiguous(), rows, eps)
        counts.append(c)
        sums.append(sm)
        start += n
    return torch.stack(counts), torch.stack(sums)


def confusion_counts(scores, labels, eps):
    """(TP, TN, FP, FN) with pred = score < eps -> 0, gt = label < eps -> 0 (k_confusion's classes), in numpy."""
    p, g = scores >= eps, labels >= eps
    return [int(np.sum(g & p)), int(np.sum(~g & ~p)), int(np.sum(~g & p)), int(np.sum(g & ~p))]


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


def abi_call(eng, net, mh, cat, offs, poses, eps):
    """sps_filter_scans_batch through the C ABI on one concatenated device tensor: (return code, outputs)."""
    from sps_b200 import _cabi
    from sps_b200.engine import _ptr, _stream
    lib = _cabi.load()
    n, batch = offs[-1], len(offs) - 1
    nbytes = lib.sps_filter_scans_batch_scratch_bytes(n, batch)
    out = dict(rows=torch.empty((max(2 * n, 1), 5), device="cuda"),
               row_offsets=torch.empty(batch + 1, dtype=torch.int32, device="cuda"),
               n_rows=torch.empty(1, dtype=torch.int32, device="cuda"),
               counts=torch.empty((batch, 2), dtype=torch.int32, device="cuda"),
               scan_scores=torch.empty(max(n, 1), device="cuda"),
               metric_counts=torch.empty((batch, 4), dtype=torch.int64, device="cuda"),
               metric_sums=torch.empty((batch, 5), dtype=torch.float64, device="cuda"),
               kept=torch.empty((max(n, 1), 4), device="cuda"),
               kept_offsets=torch.empty(batch + 1, dtype=torch.int32, device="cuda"))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    d_poses = torch.as_tensor(poses, dtype=torch.float64).cuda().contiguous()
    h_off = (C.c_int64 * (batch + 1))(*offs)
    o = out
    rc = lib.sps_filter_scans_batch(eng.handle, net.handle, mh.handle, _ptr(cat), cat.stride(0), h_off, batch,
                                    _ptr(d_poses), eps, DS, _ptr(o["rows"]), _ptr(o["row_offsets"]), _ptr(o["n_rows"]),
                                    _ptr(o["counts"]), _ptr(o["scan_scores"]), _ptr(o["metric_counts"]),
                                    _ptr(o["metric_sums"]), _ptr(o["kept"]), _ptr(o["kept_offsets"]), _ptr(scratch),
                                    nbytes, _stream())
    torch.cuda.synchronize()
    return rc, out


def offsets_of(scans):
    return np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.int64).tolist()


def test_rows_and_counts_bit_identical_to_the_per_scan_transform_and_prune(world, map_hash, state_dict):
    from sps_b200 import _cabi
    from sps_b200.engine import Engine, Net
    w, base = world
    poses = distinct_poses()
    scans = hdl_scans(w, base, poses)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    moved = map_frame(dev, poses)
    ref_rows, ref_roff, ref_counts = map_hash.prune_batch(moved)
    offs = offsets_of(scans)
    net = Net(make_model(state_dict).MinkUNet.state_dict(), "cuda")
    rc, out = abi_call(Engine(2 * offs[-1], "cuda"), net, map_hash, torch.cat(dev), offs, poses, 0.84)
    assert rc == _cabi.SPS_OK
    n_rows = int(out["n_rows"].item())
    assert n_rows == len(ref_rows)
    assert torch.equal(out["rows"][:n_rows], ref_rows)
    assert torch.equal(out["row_offsets"], ref_roff) and torch.equal(out["counts"], ref_counts)
    # the rows hold the map-frame points of each scan: bit for bit the single-scan transform, and every pose matters
    for b, (m, T) in enumerate(zip(moved, poses)):
        r0 = int(ref_roff[b])
        assert torch.equal(out["rows"][r0:r0 + len(m), 1:4], m)
        if len(m):
            other = map_frame([dev[b]], [poses[(b + 1) % len(poses)]])[0]
            assert not torch.equal(other, m)
    # the per-scan cases still are what they are after the round trip through the sensor frame
    counts = ref_counts.cpu().tolist()
    assert counts[2] == [0, 0] and counts[3][0] == 0 and counts[3][1] > 0 and counts[0][0] > 0


@pytest.mark.parametrize("pattern_sort", [0, 2], indirect=True)
@pytest.mark.parametrize("backend", [0, 1])
def test_scores_bit_identical_to_infer_scans_on_the_moved_scans(world, map_hash, state_dict, pattern_sort, backend):
    w, base = world
    poses = distinct_poses()
    scans = hdl_scans(w, base, poses)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    model = make_model(state_dict, backend)
    got = model.filter_scans_async(dev, poses, map_hash, 0.84).result()
    ref_scores, ref_counts = model.infer_scans_async(map_frame(dev, poses), map_hash).result()
    assert got.scan_scores.is_cuda and got.scan_scores.shape == (sum(len(s) for s in scans),)
    assert torch.equal(got.scan_scores, ref_scores)
    assert torch.equal(got.counts, ref_counts)


@pytest.mark.parametrize("eps", [0.84, 0.0, 1.0, "median"])
def test_published_clouds_and_metrics_match_the_per_scan_node(world, map_hash, state_dict, eps):
    """eps "median": the median score, so that about half the points of the batch are published."""
    w, base = world
    poses = distinct_poses()
    scans = hdl_scans(w, base, poses)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    model = make_model(state_dict)
    if eps == "median":
        eps = float(model.filter_scans_async(dev, poses, map_hash, 0.84).result().scan_scores.median())
    got = model.filter_scans_async(dev, poses, map_hash, eps).result()
    scores = got.scan_scores
    # published clouds: util.filter_scan scan by scan, laid end to end, and oracle.filter_scan
    ref_kept, ref_offs = filtered_reference(dev, scores, eps)
    assert got.kept_offsets.dtype == torch.int32 and got.kept_offsets.cpu().tolist() == ref_offs
    assert got.kept.shape == (ref_offs[-1], 4) and torch.equal(got.kept, ref_kept)
    host_scores = scores.cpu().numpy()
    offs = offsets_of(scans)
    for b, s in enumerate(scans):
        want = O.filter_scan(s, host_scores[offs[b]:offs[b + 1]], eps)
        part = got.kept[ref_offs[b]:ref_offs[b + 1]].cpu().numpy()
        assert part.shape == want.shape and (part.view(np.int32) == want.view(np.int32)).all()
    if eps == 0.0:
        assert ref_offs[-1] == 0
    elif eps == 1.0:
        assert ref_offs[-1] == offs[-1]
    elif eps != 0.84:
        assert 0 < ref_offs[-1] < offs[-1]
    # metrics: the counts exactly, the sums as parallel.device_partials on the scan's rows
    labels = np.concatenate([s[:, 3] for s in scans])
    for b in range(len(scans)):
        sl = slice(offs[b], offs[b + 1])
        assert got.metric_counts[b].cpu().tolist() == confusion_counts(host_scores[sl], labels[sl], np.float32(eps))
    ref_counts, ref_sums = partials_reference(dev, scores, eps)
    assert torch.equal(got.metric_counts, ref_counts)
    assert torch.allclose(got.metric_sums, ref_sums, rtol=1e-12, atol=0)
    assert torch.all(got.metric_counts[2] == 0) and torch.all(got.metric_sums[2] == 0)          # the empty scan
    assert int(got.metric_sums[0, 0]) == len(scans[0])


def test_coordinate_moved_out_of_key_range_raises_at_result(world, map_hash, state_dict):
    from sps_b200._cabi import SPS_ERR_COORD_RANGE, SpsError
    w, base = world
    poses = distinct_poses()[:2].copy()
    scans = [torch.as_tensor(s).cuda() for s in hdl_scans(w, base, poses)[:2]]
    model = make_model(state_dict)
    model.filter_scans_async(scans, poses, map_hash, 0.84).result()         # in range
    scans[1] = scans[1].clone()
    scans[1][7, :3] = torch.tensor([1.0e4, 0.0, 0.0])
    far = poses.copy()
    far[1] = translate(np.eye(4), (1.5e4, 0.0, 0.0))                        # 25 km: 250 000 voxels of 0.1 m, past x's range
    h = model.filter_scans_async(scans, far, map_hash, 0.84)
    with pytest.raises(SpsError) as e:
        h.result()
    assert e.value.code == SPS_ERR_COORD_RANGE
    got = model.filter_scans_async(scans[:1], poses[:1], map_hash, 0.84).result()   # the status word was cleared
    assert got.scan_scores.shape == (len(scans[0]),)


def assert_same(a, b):
    for x, y in zip(a, b):
        if x.dtype == torch.float64:
            assert torch.allclose(x.cpu(), y.cpu(), rtol=1e-12, atol=0)
        else:
            assert torch.equal(x.cpu(), y.cpu())


def test_host_inputs_give_the_device_results_in_pinned_memory(world, map_hash, state_dict):
    w, base = world
    poses = distinct_poses()
    scans = hdl_scans(w, base, poses)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    model = make_model(state_dict)
    want = tuple(t.clone() for t in model.filter_scans_async(dev, poses, map_hash, 0.84).result())
    for s_in, p_in in (([torch.as_tensor(s).pin_memory() for s in scans], poses),
                       ([torch.as_tensor(s).pin_memory() for s in scans], torch.as_tensor(poses).cuda()),
                       (dev, torch.as_tensor(poses)),
                       (torch.cat(dev), torch.as_tensor(poses).cuda())):
        kw = {"offsets": offsets_of(scans)} if isinstance(s_in, torch.Tensor) else {}
        got = model.filter_scans_async(s_in, p_in, map_hash, 0.84, **kw).result()
        on_device = isinstance(s_in, torch.Tensor) or s_in[0].is_cuda
        for t in got:
            assert t.is_cuda == on_device and (on_device or t.is_pinned())
        assert_same(got, want)


@pytest.mark.parametrize("on_device", [False, True])
def test_pipelined_calls_match_synchronous_calls(world, map_hash, state_dict, on_device):
    w, base = world
    batches = []
    for k in range(5):
        poses = distinct_poses(variant=k)
        scans = hdl_scans(w, base, poses, variant=k % 3)[k % 2:]
        batches.append(([torch.as_tensor(s).cuda() if on_device else torch.as_tensor(s).pin_memory() for s in scans],
                        poses[k % 2:]))
    model = make_model(state_dict, lanes=3)
    sync = [tuple(t.clone() for t in model.filter_scans_async(s, p, map_hash, 0.84).result()) for s, p in batches]
    pending, got = [], []
    for s, p in batches:
        pending.append(model.filter_scans_async(s, p, map_hash, 0.84))
        if len(pending) >= model.lanes:
            got.append(tuple(t.clone() for t in pending.pop(0).result()))
    got += [tuple(t.clone() for t in h.result()) for h in pending]
    assert len(got) == len(sync)
    for a, b in zip(sync, got):
        assert a[0].is_cuda == on_device
        assert_same(a, b)


def test_full_size_config3_shape(state_dict):
    """Eight config-3 scans in their sensor frames (above 400 000 rows, default settings): rows, scores and published
    rows bit for bit against the per-scan composition."""
    from sps_b200 import _cabi, synth
    from sps_b200.engine import Engine, MapHash, Net
    w = synth.World(0)
    traj = synth.loop_trajectory(radius=35.0, n=400)
    base = synth.base_map(w, "hdl-32", n_poses=400, seed=0, voxel=DS, trajectory=traj, target_voxels=1_000_000)
    mh = MapHash(torch.as_tensor(base).cuda(), DS)
    poses = np.stack([translate(rotation(0.0, 0.0, 0.3 * i), (35.0 * np.cos(i), 35.0 * np.sin(i), 0.1))
                      for i in range(8)])
    rng = np.random.default_rng(3)
    scans = []
    for i in range(8):
        xyz = synth.scan(w, "hdl-32", traj(7 * i), seed=i)[:, :3]
        scans.append(np.hstack([to_sensor(xyz, poses[i]), rng.random((len(xyz), 1))]).astype(np.float32))
    dev = [torch.as_tensor(s).cuda() for s in scans]
    moved = map_frame(dev, poses)
    rows, roff, counts = mh.prune_batch(moved)
    assert len(rows) > 400_000
    model = make_model(state_dict, lanes=1)
    want_scores = model(rows)[rows[:, 4] == 1]
    model.check()
    eps = float(want_scores.median())              # about half the points are published
    got = model.filter_scans_async(dev, poses, mh, eps).result()
    assert torch.equal(got.scan_scores, want_scores) and torch.equal(got.counts, counts)
    ref_kept, ref_offs = filtered_reference(dev, want_scores, eps)
    assert got.kept_offsets.cpu().tolist() == ref_offs and torch.equal(got.kept, ref_kept)
    assert 0 < ref_offs[-1] < len(want_scores)
    offs = offsets_of(scans)
    net = Net(model.MinkUNet.state_dict(), "cuda")
    rc, out = abi_call(Engine(2 * offs[-1], "cuda"), net, mh, torch.cat(dev), offs, poses, 0.84)
    assert rc == _cabi.SPS_OK and torch.equal(out["rows"][:len(rows)], rows) and torch.equal(out["row_offsets"], roff)


def test_batch_size_limits_empty_batches_and_context_capacity(world, map_hash, state_dict):
    from sps_b200 import _cabi
    from sps_b200.engine import Engine, Net, _stream
    w, base = world
    rng = np.random.default_rng(4)
    poses = np.stack([translate(rotation(0, 0, 0.01 * b), (0.1 * (b % 7), -0.05 * (b % 5), 0.0)) for b in range(255)])
    tiny = [np.hstack([to_sensor(base[rng.integers(0, len(base), 3)] + np.float32(0.01), T), rng.random((3, 1))])
            .astype(np.float32) for T in poses]
    dev = [torch.as_tensor(t).cuda() for t in tiny]
    model = make_model(state_dict)
    got = model.filter_scans_async(dev, poses, map_hash, 0.84).result()
    ref_scores, ref_counts = model.infer_scans_async(map_frame(dev, poses), map_hash).result()
    assert torch.equal(got.scan_scores, ref_scores) and torch.equal(got.counts, ref_counts)
    ref_kept, ref_offs = filtered_reference(dev, ref_scores, 0.84)
    assert got.kept_offsets.cpu().tolist() == ref_offs and torch.equal(got.kept, ref_kept)
    with pytest.raises(ValueError):
        model.filter_scans_async(dev + dev[:1], np.concatenate([poses, poses[:1]]), map_hash, 0.84)
    # only empty scans: zero counts, partials and offsets
    empty = [torch.zeros((0, 4), device="cuda")] * 3
    got = model.filter_scans_async(empty, poses[:3], map_hash, 0.84).result()
    assert got.scan_scores.shape == (0,) and got.kept.shape == (0, 4)
    assert torch.all(got.counts == 0) and torch.all(got.metric_counts == 0) and torch.all(got.metric_sums == 0)
    assert got.kept_offsets.cpu().tolist() == [0, 0, 0, 0]
    # the C ABI: 2 n_total above the context's max_points
    n = 3 * 255
    net = Net(model.MinkUNet.state_dict(), "cuda")
    offs = offsets_of(tiny)
    rc, _ = abi_call(Engine(2 * n - 1, "cuda"), net, map_hash, torch.cat(dev), offs, poses, 0.84)
    assert rc == _cabi.SPS_ERR_CAPACITY
    eng = Engine(2 * n, "cuda")
    rc, out = abi_call(eng, net, map_hash, torch.cat(dev), offs, poses, 0.84)
    assert rc == _cabi.SPS_OK and torch.equal(out["scan_scores"][:n], ref_scores)
    assert _cabi.load().sps_ctx_status(eng.handle, _stream()) == _cabi.SPS_OK
