"""Batch-sharded sequence calls (parallel.ShardedScans) against the single-process loop over the batches, bit for bit
(the atomically accumulated float64 metric sums to rounding), at world size 1 and under NCCL at world size 2; the
segment reassembly kernel (sps_gather_segments) against numpy."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from test_gpu_filter_scans import DS, distinct_poses, hdl_scans as sensor_scans, make_model  # noqa: E402
from test_gpu_radius_batch import hdl_scans as map_scans  # noqa: E402

pytestmark = pytest.mark.gpu

EPS = 0.5


# ---------------------------------------------------------------------------------------------------------- kernel ---
def numpy_segments(src, ranks, starts, rows, lens):
    lens = np.clip(lens, 0, rows)
    parts = [src[r, s:s + l] for r, s, l in zip(ranks, starts, lens)]
    return np.concatenate(parts) if parts else src[0, :0], np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)


@pytest.mark.parametrize("width", [1, 4])
@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_gather_segments_matches_numpy(width, world):
    from sps_b200.parallel import gather_segments
    rng = np.random.default_rng([world, width])
    n_seg = 2500                                         # three launches of 1 024 segments
    ranks = rng.integers(0, world, n_seg)
    rows = rng.integers(0, 1200, n_seg) * (rng.random(n_seg) < 0.9)
    starts = np.zeros(n_seg, np.int64)
    used = np.zeros(world, np.int64)
    for s in range(n_seg):                               # each rank's segments back to back, as ShardPlan lays them out
        starts[s] = used[ranks[s]]
        used[ranks[s]] += rows[s]
    cap = int(used.max()) + 3
    assert rows.sum() > 1 << 20
    shape = (world, cap, width) if width > 1 else (world, cap)
    src = torch.randn(shape, device="cuda")
    # lengths that exist only on the device: some zero, some above the bound (clamped) and some negative (zero)
    g = torch.Generator(device="cuda").manual_seed(world)
    bound = torch.as_tensor(rows, device="cuda")
    lens = (torch.rand(n_seg, device="cuda", generator=g) * 1.2 * bound).to(torch.int32)
    lens[::7] = 0
    lens[::11] = -5
    out = torch.full((int(rows.sum()),) + shape[2:], float("nan"), device="cuda")
    offs = torch.empty(n_seg + 1, dtype=torch.int32, device="cuda")
    gather_segments(src, ranks.tolist(), starts.tolist(), rows.tolist(), lens, out, offs)
    want, want_off = numpy_segments(src.cpu().numpy(), ranks, starts, rows, lens.cpu().numpy())
    assert np.array_equal(offs.cpu().numpy(), want_off)
    got = out.cpu().numpy()
    assert np.array_equal(got[:len(want)].view(np.int32), want.view(np.int32))
    assert np.isnan(got[len(want):]).all()                # nothing past the written rows


def test_gather_segments_scalar_path_and_edge_cases():
    from sps_b200.parallel import gather_segments
    src = torch.arange(2 * 9 * 4, dtype=torch.float32, device="cuda").reshape(2, 9, 4)
    lens = torch.tensor([2, 0, 3], dtype=torch.int32, device="cuda")
    # an output that is not 16-byte aligned takes the scalar copies: same rows
    buf = torch.full((11 * 4 + 1,), -1.0, device="cuda")          # room for all three segments full: 3 + 5 + 3 rows
    out = buf[1:].view(11, 4)
    offs = torch.empty(4, dtype=torch.int32, device="cuda")
    gather_segments(src, [1, 0, 0], [4, 0, 6], [3, 5, 3], lens, out, offs)
    s = src.cpu()
    assert offs.cpu().tolist() == [0, 2, 2, 5]
    assert torch.equal(out[:5].cpu(), torch.cat([s[1, 4:6], s[0, 6:9]]))
    assert buf[0].item() == -1.0 and torch.all(out[5:] == -1.0)
    # no segments at all: the offsets are [0]
    offs = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    gather_segments(src, [], [], [], lens, out, offs)
    assert offs.cpu().tolist() == [0]


# ------------------------------------------------------------------------------------------------------ world 1 ---
@pytest.fixture(scope="module")
def world_map():
    from sps_b200 import synth
    w = synth.World(2)
    return w, synth.base_map(w, "hdl-32", n_poses=6, seed=2, voxel=DS).astype(np.float32)


@pytest.fixture
def sort_always():
    """Shape-sort every forward: with the default mode a radius call's decision follows its lane's row capacity, which
    depends on the calls the lanes served before."""
    from sps_b200 import engine
    old = engine.DEFAULTS["pattern_sort"]
    engine.set_defaults(pattern_sort=2)
    yield
    engine.set_defaults(pattern_sort=old)


def eval_sequence(w, n_rep=2):
    """Scans of test_gpu_radius_batch (full, part, empty, far) in several variants: S = 4 * n_rep - 1."""
    out = []
    for v in range(n_rep):
        out += map_scans(w, variant=v)
    return out[:-1]


def replay_sequence(w, base, n_rep=2):
    poses, scans = [], []
    for v in range(n_rep):
        p = distinct_poses(variant=v)
        poses.append(p)
        scans += sensor_scans(w, base, p, variant=v)
    return scans[:-1], np.concatenate(poses)[:-1]


def loop_evaluate(model, scans, submap, B):
    res = [tuple(t.clone() for t in model.predict_radius_async(scans[a:a + B], submap, EPS).result())
           for a in range(0, len(scans), B)]
    return [torch.cat([r[i].cuda() for r in res]) for i in range(3)]


def loop_replay(model, scans, poses, map_hash, eps, B):
    res = [tuple(t.clone() for t in model.filter_scans_async(scans[a:a + B], poses[a:a + B], map_hash, eps).result())
           for a in range(0, len(scans), B)]
    kept_offsets, base = [0], 0
    for r in res:
        kept_offsets += (r[2][1:].cpu() + base).tolist()
        base += len(r[1])
    out = [torch.cat([r[i].cuda() for r in res]) for i in range(6)]
    out[2] = torch.tensor(kept_offsets, dtype=torch.int32)
    return out


def assert_evaluate_equal(got, want):
    from sps_b200.parallel import metrics_from_partials
    scores, counts, sums = want
    assert torch.equal(got.scan_scores.cpu(), scores.cpu())
    assert torch.equal(got.metric_counts.cpu(), counts.cpu())
    assert_sums_close(got, sums, metrics_from_partials(counts.cpu(), sums.cpu()))
    assert got.kept is None and got.kept_offsets is None and got.counts is None


def assert_replay_equal(got, want):
    from sps_b200.parallel import metrics_from_partials
    scores, kept, kept_offsets, counts, mc, ms = want
    assert torch.equal(got.scan_scores.cpu(), scores.cpu())
    assert torch.equal(got.kept.cpu(), kept.cpu())
    assert got.kept_offsets.dtype == torch.int32 and torch.equal(got.kept_offsets.cpu(), kept_offsets)
    assert torch.equal(got.counts.cpu(), counts.cpu())
    assert torch.equal(got.metric_counts.cpu(), mc.cpu())
    assert_sums_close(got, ms, metrics_from_partials(mc.cpu(), ms.cpu()))


def assert_sums_close(got, sums, metrics):
    """The float64 sums are accumulated with atomics, so two runs of the same call agree to rounding only (as in
    test_gpu_filter_scans); the metrics computed from them likewise."""
    assert torch.allclose(got.metric_sums.cpu(), sums.cpu(), rtol=1e-12, atol=0)
    assert set(got.metrics) == set(metrics)
    for k in metrics:
        assert got.metrics[k] == pytest.approx(metrics[k], rel=1e-9, abs=1e-12, nan_ok=True), k


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("on_device", [True, False])
def test_evaluate_world1_equals_the_batch_loop(world_map, sort_always, B, on_device):
    from sps_b200.datasets import RadiusSubmap
    from sps_b200.parallel import ShardedScans
    w, base = world_map
    scans = [torch.as_tensor(s).cuda() if on_device else torch.as_tensor(s).pin_memory() for s in eval_sequence(w)]
    assert len(scans) % B or B == 1                                   # S = 7: not a multiple of 3
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), DS)
    sd = make_sd()
    got = ShardedScans(make_model(sd), EPS, B).evaluate(scans, sub)
    want = loop_evaluate(make_model(sd), scans, sub, B)
    assert_evaluate_equal(got, want)
    assert int(got.metric_counts[2].sum()) == 0                       # the empty scan


@pytest.mark.parametrize("B", [1, 4])
@pytest.mark.parametrize("on_device", [True, False])
def test_replay_world1_equals_the_batch_loop(world_map, B, on_device):
    from sps_b200.engine import MapHash
    from sps_b200.parallel import ShardedScans
    w, base = world_map
    mh = MapHash(torch.as_tensor(base).cuda(), DS)
    host, poses = replay_sequence(w, base)
    scans = [torch.as_tensor(s).cuda() if on_device else torch.as_tensor(s).pin_memory() for s in host]
    sd = make_sd()
    model = make_model(sd)
    eps = float(model.filter_scans_async(scans[:6], poses[:6], mh, 0.84).result().scan_scores.median())
    ss = ShardedScans(model, eps, B)
    got = ss.replay(scans, torch.as_tensor(poses).cuda() if on_device else poses, mh)
    want = loop_replay(make_model(sd), scans, poses, mh, eps, B)
    assert_replay_equal(got, want)
    assert 0 < len(got.kept) < len(got.scan_scores)                    # eps at the median: non-trivial clouds
    firsts = list(range(0, len(scans), B)) + [len(scans)]
    assert torch.equal(ss.batch_offsets.cpu(), got.kept_offsets[firsts].cpu())   # the kernel's offsets of the batches
    start, end = ss.gather_events
    assert start.elapsed_time(end) >= 0.0


def test_b255_and_empty_scans(world_map):
    from sps_b200.engine import MapHash
    from sps_b200.parallel import ShardedScans
    from test_gpu_filter_scans import rotation, to_sensor, translate
    w, base = world_map
    mh = MapHash(torch.as_tensor(base).cuda(), DS)
    rng = np.random.default_rng(4)
    S = 300                                                            # batches of 255 and 45 scans
    poses = np.stack([translate(rotation(0, 0, 0.01 * b), (0.1 * (b % 7), -0.05 * (b % 5), 0.0)) for b in range(S)])
    scans = [np.hstack([to_sensor(base[rng.integers(0, len(base), 3)] + np.float32(0.01), T), rng.random((3, 1))])
             .astype(np.float32) for T in poses]
    scans = [torch.as_tensor(s if b % 9 else s[:0]).cuda() for b, s in enumerate(scans)]
    sd = make_sd()
    got = ShardedScans(make_model(sd), 0.84, 255).replay(scans, poses, mh)
    assert_replay_equal(got, loop_replay(make_model(sd), scans, poses, mh, 0.84, 255))
    assert torch.all(got.metric_counts[::9] == 0)
    # all scans empty
    empty = [torch.zeros((0, 4), device="cuda")] * 5
    got = ShardedScans(make_model(sd), 0.84, 2).replay(empty, poses[:5], mh)
    assert got.scan_scores.shape == (0,) and got.kept.shape == (0, 4) and got.kept_offsets.tolist() == [0] * 6
    assert got.metrics == {}


def test_evaluate_b255_and_empty_scans(world_map, sort_always):
    from sps_b200.datasets import RadiusSubmap
    from sps_b200.parallel import ShardedScans
    w, base = world_map
    rng = np.random.default_rng(5)
    S = 300                                                            # batches of 255 and 45 scans
    scans = [np.hstack([base[rng.integers(0, len(base), 4)] + np.float32(0.01), rng.random((4, 1))]).astype(np.float32)
             for _ in range(S)]
    scans = [torch.as_tensor(s if b % 9 else s[:0]).cuda() for b, s in enumerate(scans)]
    sub = RadiusSubmap(torch.as_tensor(base).cuda(), DS)
    sd = make_sd()
    got = ShardedScans(make_model(sd), EPS, 255).evaluate(scans, sub)
    assert_evaluate_equal(got, loop_evaluate(make_model(sd), scans, sub, 255))
    assert torch.all(got.metric_counts[::9] == 0) and got.scan_scores.shape == (4 * (S - 34),)


def test_evaluate_batches_that_overflow_their_lane_run_again(sort_always):
    """A map so dense around the scans that every batch has ~31 rows per scan point: more than the 6 per point the lanes
    are sized for, so every call leaves its rows unscored and ShardedScans runs each batch again at the end, as the
    single call's result() does."""
    from sps_b200.datasets import RadiusSubmap
    from sps_b200.parallel import ShardedScans
    rng = np.random.default_rng(6)
    scans = [np.hstack([rng.uniform(-20, 20, (300, 3)), rng.random((300, 1))]).astype(np.float32) for _ in range(5)]
    pts = np.vstack([s[:, :3] for s in scans])
    dense = (np.repeat(pts, 30, axis=0) + rng.uniform(-0.02, 0.02, (30 * len(pts), 3))).astype(np.float32)
    sub = RadiusSubmap(torch.as_tensor(dense).cuda(), DS)
    dev = [torch.as_tensor(s).cuda() for s in scans]
    assert len(sub.make_batch(dev[:2])) > 12 * 600                     # above any lane sized for 6 rows per point
    sd = make_sd()
    model = make_model(sd)
    got = ShardedScans(model, EPS, 2).evaluate(dev, sub)
    assert_evaluate_equal(got, loop_evaluate(make_model(sd), dev, sub, 2))
    assert not torch.isnan(got.scan_scores).any() and int(got.metric_sums[:, 0].sum()) == 1500
    model.check()                                                      # no status word left behind


def test_coordinate_out_of_key_range_raises(world_map):
    from sps_b200._cabi import SPS_ERR_COORD_RANGE, SpsError
    from sps_b200.engine import MapHash
    from sps_b200.parallel import ShardedScans
    w, base = world_map
    mh = MapHash(torch.as_tensor(base).cuda(), DS)
    host, poses = replay_sequence(w, base)
    scans = [torch.as_tensor(s).cuda() for s in host[:4]]
    poses = poses[:4].copy()
    poses[3] = np.eye(4)
    poses[3, 0, 3] = 3.0e4                                             # 30 km: far past the key's 13.1 km x range
    model = make_model(make_sd())
    with pytest.raises(SpsError) as e:
        ShardedScans(model, 0.84, 2).replay(scans, poses, mh)
    assert e.value.code == SPS_ERR_COORD_RANGE
    got = ShardedScans(model, 0.84, 2).replay(scans[:3], poses[:3], mh)    # the status words were cleared
    assert got.scan_scores.shape == (sum(len(s) for s in scans[:3]),)


def test_gather_segments_wrapper_checks_its_tensors():
    from sps_b200.parallel import gather_segments
    src = torch.zeros((2, 9, 4), device="cuda")
    out = torch.zeros((11, 4), device="cuda")
    lens = torch.zeros(3, dtype=torch.int32, device="cuda")
    offs = torch.zeros(4, dtype=torch.int32, device="cuda")
    args = ([1, 0, 0], [4, 0, 6], [3, 5, 3])
    gather_segments(src, *args, lens, out, offs)
    for bad in (dict(lens=lens.long()), dict(lens=lens[:2]), dict(offs=offs.long()), dict(offs=offs[:3]),
                dict(src=src.double()), dict(src=torch.zeros((2, 4, 9), device="cuda").transpose(1, 2)),
                dict(out=out[:, :2]), dict(out=out.cpu()), dict(out=torch.zeros(44, device="cuda"))):
        a = {**dict(src=src, lens=lens, out=out, offs=offs), **bad}
        with pytest.raises(ValueError):
            gather_segments(a["src"], *args, a["lens"], a["out"], a["offs"])
    with pytest.raises(ValueError):
        gather_segments(src, [1, 0], [4, 0, 6], [3, 5, 3], lens, out, offs)


def make_sd():
    from oracle import sps_oracle as O
    return O.make_state_dict(seed=0, randomize_bn=True)


# ------------------------------------------------------------------------------------------------- NCCL world 2 ---
CASES = [("replay", 2, 4), ("replay", 5, 2), ("evaluate", 2, 4), ("evaluate", 5, 2)]   # (call, S, B): 1 and 3 batches


def _nccl_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from sps_b200 import engine, synth
    from sps_b200.datasets import RadiusSubmap
    from sps_b200.engine import MapHash
    from sps_b200.parallel import ShardedScans
    engine.set_defaults(pattern_sort=2)
    w = synth.World(2)
    base = synth.base_map(w, "hdl-32", n_poses=6, seed=2, voxel=DS).astype(np.float32)
    sd = make_sd()
    model = make_model(sd)
    mh, sub = MapHash(torch.as_tensor(base).cuda(), DS), RadiusSubmap(torch.as_tensor(base).cuda(), DS)
    for call, S, B in CASES:
        if call == "replay":
            host, poses = replay_sequence(w, base)
            scans = [torch.as_tensor(s).cuda() for s in host[:S]]
            eps = float(model.filter_scans_async(scans, poses[:S], mh, 0.84).result().scan_scores.median())
            got = ShardedScans(model, eps, B).replay(scans, poses[:S], mh)
        else:
            scans = [torch.as_tensor(s).cuda() for s in eval_sequence(w)[:S]]
            got = ShardedScans(model, EPS, B).evaluate(scans, sub)
        key = f"{call}{S}_{B}_rank{rank}"
        out[key] = {f: (t.cpu().numpy().copy() if isinstance(t, torch.Tensor) else t) for f, t in got._asdict().items()}
    # a coordinate out of range in batch 1 only, which rank 1 runs: both ranks raise, neither waits in a gather
    from sps_b200._cabi import SpsError
    host, poses = replay_sequence(w, base)
    poses = poses[:4].copy()
    poses[3] = np.eye(4)
    poses[3, 0, 3] = 3.0e4
    try:
        ShardedScans(model, 0.84, 2).replay([torch.as_tensor(s).cuda() for s in host[:4]], poses, mh)
        out[f"error_rank{rank}"] = 0
    except SpsError as e:
        out[f"error_rank{rank}"] = e.code
    dist.barrier()
    dist.destroy_process_group()


def test_world2_nccl_equals_the_single_process_loop(world_map, sort_always):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (NCCL: one rank per device)")
    from sps_b200.datasets import RadiusSubmap
    from sps_b200.engine import MapHash
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_nccl_worker, args=(2, port, out), nprocs=2, join=True)
    w, base = world_map
    sd = make_sd()
    mh, sub = MapHash(torch.as_tensor(base).cuda(), DS), RadiusSubmap(torch.as_tensor(base).cuda(), DS)
    from sps_b200._cabi import SPS_ERR_COORD_RANGE
    assert out["error_rank0"] == out["error_rank1"] == SPS_ERR_COORD_RANGE
    for call, S, B in CASES:
        r0, r1 = out[f"{call}{S}_{B}_rank0"], out[f"{call}{S}_{B}_rank1"]
        for f in ("scan_scores", "kept", "kept_offsets"):
            assert r1[f] is None                                       # rank 0 only
        np.testing.assert_equal(r0["metrics"], r1["metrics"])
        assert len(r0["metrics"]) == 6
        for f in ("metric_counts", "metric_sums", "counts"):
            assert (r0[f] is None and r1[f] is None) or np.array_equal(r0[f], r1[f])
        if call == "replay":
            host, poses = replay_sequence(w, base)
            scans = [torch.as_tensor(s).cuda() for s in host[:S]]
            model = make_model(sd)
            eps = float(model.filter_scans_async(scans, poses[:S], mh, 0.84).result().scan_scores.median())
            want = loop_replay(make_model(sd), scans, poses[:S], mh, eps, B)
            names = ("scan_scores", "kept", "kept_offsets", "counts", "metric_counts", "metric_sums")
            assert 0 < len(r0["kept"]) < len(r0["scan_scores"])
        else:
            scans = [torch.as_tensor(s).cuda() for s in eval_sequence(w)[:S]]
            want = loop_evaluate(make_model(sd), scans, sub, B)
            names = ("scan_scores", "metric_counts", "metric_sums")
        for f, t in zip(names, want):
            if f == "metric_sums":                                     # atomics: equal to rounding (assert_sums_close)
                assert np.allclose(r0[f], t.cpu().numpy(), rtol=1e-12, atol=0), (call, S, B, f)
            else:
                assert np.array_equal(r0[f], t.cpu().numpy()), (call, S, B, f)
