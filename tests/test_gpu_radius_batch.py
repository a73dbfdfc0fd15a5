"""Batched radius submaps + collation + predict_step partials in the library (RadiusSubmap.make_batch,
SPSModel.predict_radius_async, SPSNet.predict_scans) against the per-scan path and scipy's query_ball_tree, the call
BLTDataset.select_closest_points makes (src/sps/datasets/blt_dataset.py:173-182,209-271, models.py:84-104)."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

R = 0.1
EPS = 0.5


@pytest.fixture(scope="module")
def world():
    from sps_b200 import synth
    w = synth.World(2)
    base = synth.base_map(w, "hdl-32", n_poses=6, seed=2, voxel=R).astype(np.float32)
    return w, base


def labelled(xyz, seed):
    lab = np.random.default_rng([seed, 5]).uniform(0, 1, (len(xyz), 1)).astype(np.float32)
    return np.hstack([xyz.astype(np.float32), lab])


def hdl_scans(w, variant=0):
    """B = 4 hdl-32 scans of different sizes: a full one, a part of one, an empty one, one far from the map."""
    from sps_b200 import synth
    a = synth.scan(w, "hdl-32", pose=(1.0, -2.0, 0.3 + variant), seed=5 + variant)
    b = synth.scan(w, "hdl-32", pose=(-0.5, 0.5, 1.1 + variant), seed=6 + variant)[: 30000 - 1000 * variant]
    far = synth.scan(w, "hdl-32", pose=(0.0, 0.0, 0.0), seed=7)[:5000] + np.float32(500.0)
    return [labelled(a, 1 + variant), labelled(b, 2 + variant), np.zeros((0, 4), np.float32), labelled(far, 3)]


def per_scan_rows(sub, scans_dev):
    """The per-scan path: make_item per scan, batch column in front, stacked (collate_fn)."""
    items = [sub.make_item(s) for s in scans_dev]
    return torch.vstack([torch.hstack([torch.full((len(it), 1), float(b), device="cuda"), it]) for b, it in enumerate(items)])


@pytest.fixture
def sort_always():
    """Shape-sort every forward (sps_ctx_set_pattern_sort 2): with the default mode the decision for the batched call
    follows the row capacity, for sps_forward the row count -- equal only on the same side of 400 000 rows."""
    from sps_b200 import engine
    old = engine.DEFAULTS["pattern_sort"]
    engine.set_defaults(pattern_sort=2)
    yield
    engine.set_defaults(pattern_sort=old)


def make_model(backend=None, lanes=3):
    from sps_b200.models import SPSModel
    from oracle import sps_oracle as O
    model = SPSModel(R)
    model.MinkUNet.load_state_dict({k: torch.as_tensor(v) for k, v in O.make_state_dict(seed=0, randomize_bn=True).items()})
    model = model.cuda().eval()
    model.lanes = lanes
    if backend is not None:
        model.set_conv_backend(backend)
    return model


def test_rows_bit_identical_to_the_per_scan_path(world):
    from sps_b200.datasets import RadiusSubmap
    w, base = world
    scans = hdl_scans(w)
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    rows, roff = sub.make_batch(dev, return_offsets=True)
    ref = per_scan_rows(sub, dev)
    assert rows.shape == ref.shape and rows.shape[1] == 6
    assert torch.equal(rows, ref)
    sizes = [len(s) + len(sub.select_closest_points(d)) for s, d in zip(scans, dev)]
    assert roff.cpu().tolist() == np.concatenate([[0], np.cumsum(sizes)]).tolist()
    assert sizes[2] == 0 and sizes[3] == len(scans[3])          # empty scan; far scan: its own rows, no submap
    # the other input forms: one concatenated tensor + offsets, host tensors
    cat = torch.as_tensor(np.vstack(scans)).cuda()
    offs = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).tolist()
    assert torch.equal(sub.make_batch(cat, offs), ref)
    assert torch.equal(sub.make_batch([torch.as_tensor(s) for s in scans]), ref)
    # wider scan rows (extra columns are ignored)
    wide = [torch.hstack([d, torch.full((len(d), 2), 7.0, device="cuda")]) for d in dev]
    assert torch.equal(sub.make_batch(wide), ref)


def test_submap_rows_are_the_reference_selection(world):
    """Per scan, the multiset of submap rows == map[np.concatenate(cKDTree(scan).query_ball_tree(cKDTree(map), r))]."""
    from scipy.spatial import cKDTree
    from sps_b200.datasets import RadiusSubmap
    w, base = world
    scans = hdl_scans(w)
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    rows, roff = sub.make_batch([torch.as_tensor(s).cuda() for s in scans], return_offsets=True)
    rows, roff = rows.cpu().numpy(), roff.cpu().numpy()
    tree = cKDTree(base)
    for b, s in enumerate(scans):
        mine = rows[roff[b]:roff[b + 1]]
        assert np.all(mine[:, 0] == b)
        assert np.array_equal(mine[: len(s), 1:4], s[:, :3]) and np.all(mine[: len(s), 4] == 1)
        assert np.array_equal(mine[: len(s), 5], s[:, 3])
        got = mine[len(s):]
        assert np.all(got[:, 4] == 0) and np.all(got[:, 5] == 1)
        lists = cKDTree(s[:, :3]).query_ball_tree(tree, R) if len(s) else []
        idx = np.concatenate([np.asarray(l, np.int64) for l in lists]) if len(lists) else np.zeros(0, np.int64)
        want = base[idx]
        assert len(got) == len(want)
        key = lambda a: a[np.lexsort(a.T[::-1])]
        assert np.array_equal(key(got[:, 1:4]), key(want))


def device_reference(model, rows, roff, eps):
    """SPSModel.forward on the rows, then parallel.device_partials scan by scan."""
    from sps_b200 import parallel
    scores = model(rows[:, :5])
    model.check()
    counts, sums = [], []
    for b in range(len(roff) - 1):
        if roff[b] == roff[b + 1]:       # a scan without points has no rows (and empty slices have no data pointer)
            counts.append(torch.zeros(4, dtype=torch.int64, device=rows.device))
            sums.append(torch.zeros(5, dtype=torch.float64, device=rows.device))
            continue
        c, s = parallel.device_partials(scores[roff[b]:roff[b + 1]], rows[roff[b]:roff[b + 1]], eps)
        counts.append(c)
        sums.append(s)
    return scores[rows[:, 4] == 1], torch.stack(counts), torch.stack(sums)


@pytest.mark.parametrize("backend", [0, 1])
def test_scores_and_partials_match_forward_on_the_rows(world, sort_always, backend):
    from sps_b200.datasets import RadiusSubmap
    w, base = world
    scans = [torch.as_tensor(s).cuda() for s in hdl_scans(w)]
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    model = make_model(backend)
    scan_scores, counts, sums = model.predict_radius_async(scans, sub, EPS).result()
    rows, roff = sub.make_batch(scans, return_offsets=True)
    ref_scores, ref_counts, ref_sums = device_reference(model, rows, roff.cpu().tolist(), EPS)
    assert scan_scores.shape == (sum(len(s) for s in scans),)
    assert torch.equal(scan_scores, ref_scores)
    assert torch.equal(counts, ref_counts)
    assert counts[2].sum() == 0 and torch.all(sums[2] == 0)                 # the empty scan
    assert torch.allclose(sums, ref_sums, rtol=1e-12, atol=0)


def test_predict_scans_summary_matches_predict_step_scan_by_scan(world):
    from sps_b200.datasets import RadiusSubmap
    from sps_b200.models import SPSNet
    w, base = world
    scans = [torch.as_tensor(s).cuda() for s in hdl_scans(w)]
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    ref_model = make_model(backend=1)
    hp = {"MODEL": {"VOXEL_SIZE": R}, "FILTER": {"THRESHOLD": EPS}}
    nets = []
    for _ in range(2):
        net = SPSNet(hp)
        net.model.MinkUNet.load_state_dict(ref_model.MinkUNet.state_dict())
        net.model = net.model.cuda()
        net.model.set_conv_backend(1)
        nets.append(net)
    batched, by_scan = nets
    scan_scores = batched.predict_scans(scans, sub)
    assert scan_scores.shape == (sum(len(s) for s in scans),)
    for s in scans:                      # predict.py with batch_size=1 (the empty scan has no item)
        if len(s):
            by_scan.predict_step(sub.make_batch([s]))
    a, b = batched.summary(), by_scan.summary()
    assert set(a) == set(b) == {"Loss", "R2", "dIoU", "Precision", "Recall", "F1"}
    assert len(batched.F1) == len(by_scan.F1) == 3
    for k in a:
        assert a[k] == pytest.approx(b[k], rel=1e-6, abs=1e-6), k


def test_capacity_overflow(world, sort_always):
    from sps_b200 import _cabi
    from sps_b200.datasets import RadiusSubmap, batch_parts
    from sps_b200.engine import Engine, Net, _ptr, _stream
    w, base = world
    scans = [torch.as_tensor(s).cuda() for s in hdl_scans(w)]
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    n_true = len(sub.make_batch(scans))
    model = make_model()
    # the C ABI: a capacity below the row count -> nothing scored, the true count, SPS_ERR_CAPACITY from the status word
    lib = _cabi.load()
    parts, offs, ld = batch_parts(scans)
    cat = torch.cat([t for t, _ in parts])
    eng = Engine(1 << 16, "cuda")
    net = Net(model.MinkUNet.state_dict(), "cuda")
    cap = 50000
    assert cap < n_true
    rows = torch.full((cap + 1, 6), -7.0, device="cuda")
    nbytes = lib.sps_radius_batch_scratch_bytes(offs[-1], 4)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    roff = torch.empty(5, dtype=torch.int32, device="cuda")
    n_rows = torch.zeros(1, dtype=torch.int32, device="cuda")
    scores = torch.zeros(offs[-1], device="cuda")
    counts = torch.full((4, 4), -1, dtype=torch.int64, device="cuda")
    sums = torch.full((4, 5), -1.0, dtype=torch.float64, device="cuda")
    h_off = (C.c_int64 * 5)(*offs)
    rc = lib.sps_predict_radius_batch(eng.handle, net.handle, sub.handle, _ptr(cat), ld, h_off, 4, _ptr(rows), cap, _ptr(roff),
                                      _ptr(n_rows), _ptr(scratch), nbytes, R, EPS, _ptr(scores), _ptr(counts), _ptr(sums),
                                      _stream())
    assert rc == _cabi.SPS_OK
    assert lib.sps_ctx_status(eng.handle, _stream()) == _cabi.SPS_ERR_CAPACITY
    assert int(n_rows.item()) == n_true
    assert torch.all(rows[cap] == -7.0)                                     # nothing past the capacity
    assert torch.isnan(scores).all() and torch.all(counts == 0) and torch.all(sums == 0)
    assert lib.sps_ctx_status(eng.handle, _stream()) == _cabi.SPS_OK        # the status word was cleared
    assert lib.sps_predict_radius_batch(eng.handle, net.handle, sub.handle, _ptr(cat), ld, h_off, 4, _ptr(rows), 1 << 17,
                                        _ptr(roff), _ptr(n_rows), _ptr(scratch), nbytes, R, EPS, _ptr(scores), _ptr(counts),
                                        _ptr(sums), _stream()) == _cabi.SPS_ERR_CAPACITY   # above the context's size
    # Python: lanes too small for the rows -> result() grows them and runs once more
    big = model.predict_radius_async(scans, sub, EPS).result()
    big = tuple(t.clone() for t in big)
    small = make_model()
    got = small._predict_radius(parts, offs, ld, sub, EPS, rows_guess=1024).result()
    assert small._pipe["engine"][0].max_points >= n_true
    assert torch.equal(got[0], big[0]) and torch.equal(got[1], big[1])
    assert torch.allclose(got[2], big[2], rtol=1e-12, atol=0)


def test_coordinate_out_of_key_range_raises_at_result(world):
    from sps_b200._cabi import SPS_ERR_COORD_RANGE, SpsError
    from sps_b200.datasets import RadiusSubmap
    w, base = world
    scans = [torch.as_tensor(s).cuda() for s in hdl_scans(w)[:2]]
    scans[1] = scans[1].clone()
    scans[1][7, 0] = 2.0e4                        # 200 000 voxels of 0.1 m: past the key's x range
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    model = make_model()
    h = model.predict_radius_async(scans, sub, EPS)
    with pytest.raises(SpsError) as e:
        h.result()
    assert e.value.code == SPS_ERR_COORD_RANGE
    model.predict_radius_async(scans[:1], sub, EPS).result()     # the status word was cleared: the next call is fine


@pytest.mark.parametrize("on_device", [False, True])
def test_pipelined_calls_match_synchronous_calls(world, on_device):
    from sps_b200.datasets import RadiusSubmap
    w, base = world
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    batches = []
    for k in range(5):
        scans = hdl_scans(w, variant=k % 3)[k % 2:]
        batches.append([torch.as_tensor(s).cuda() if on_device else torch.as_tensor(s).pin_memory() for s in scans])
    model = make_model(lanes=3)
    sync = [tuple(t.clone() for t in model.predict_radius_async(b, sub, EPS).result()) for b in batches]
    pending, got = [], []
    for b in batches:
        pending.append(model.predict_radius_async(b, sub, EPS))
        if len(pending) >= model.lanes:
            got.append(tuple(t.clone() for t in pending.pop(0).result()))
    got += [tuple(t.clone() for t in p.result()) for p in pending]
    for (a0, a1, a2), (b0, b1, b2) in zip(sync, got):
        assert a0.is_cuda == on_device
        assert torch.equal(a0, b0) and torch.equal(a1, b1)
        assert torch.allclose(a2, b2, rtol=1e-12, atol=0)


def test_full_size_config2_shape():
    """8 x 65 536 os1-64 scans against the benchmark's base map: rows and scores bit for bit (default settings)."""
    from sps_b200 import synth
    from sps_b200.datasets import RadiusSubmap
    w = synth.World(0)
    base = synth.base_map(w, "os1-64", n_poses=12, seed=0, voxel=R).astype(np.float32)
    rng = np.random.default_rng([1, 3])
    scans = []
    for b in range(8):
        pose = (rng.uniform(-1.5, 1.5), rng.uniform(-1.5, 1.5), rng.uniform(0, 2 * np.pi))
        scans.append(torch.as_tensor(labelled(synth.scan(w, "os1-64", pose, seed=1000 + b, dynamic=True), b)).cuda())
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), R)
    rows = sub.make_batch(scans)
    assert len(rows) > 2_000_000
    assert torch.equal(rows, per_scan_rows(sub, scans))
    model = make_model(lanes=1)
    scan_scores, counts, sums = model.predict_radius_async(scans, sub, EPS).result()
    ref = model(rows[:, :5])
    model.check()
    assert torch.equal(scan_scores, ref[rows[:, 4] == 1])
    assert int(counts.sum()) == 8 * 65536
