"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs.  Bar: voxel coordinates / inverse maps / kernel maps bit-exact (canonical sets), scores
within 2e-3 absolute (north star), thresholded labels >= 99.9 % equal."""
import numpy as np
import pytest
import torch

from conftest import make_case
from oracle import sps_oracle as O
from oracle import me_cpu

pytestmark = pytest.mark.gpu

SCORE_TOL = 2e-3   # BASELINE.json north_star: "per-point scores must match within 2e-3 absolute"
EPS = 0.84         # config/config.yaml:33


@pytest.fixture(scope="module")
def engine_mod():
    from sps_b200 import engine
    return engine


@pytest.fixture(autouse=True)
def conv_backend(request):
    """Exactness-oriented tests pin the fp32 CUDA-core kernels (backend 1); tests marked
    ``tensor_path`` run the default dispatch (tcgen05 TF32 where the layer shape allows)."""
    from sps_b200 import engine
    engine.set_defaults(conv_backend=0 if request.node.get_closest_marker("tensor_path") else 1)
    yield
    engine.set_defaults(conv_backend=0)


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).cuda()


def canon_kmap(nbr, coords_in, coords_out):
    return O.canonical_kernel_map(nbr, coords_in, coords_out)


def amplified(sd, gain=40.0):
    """Scale the head so that scores spread over (0,1) instead of hugging sigmoid(0)."""
    sd = dict(sd)
    sd["final.kernel"] = sd["final.kernel"] * np.float32(gain)
    return sd


@pytest.mark.parametrize("sensor,seed", [("tiny", 3), ("tiny", 11), ("hdl-32", 1)])
def test_voxelize_and_maps_bit_exact(engine_mod, sensor, seed):
    rows = make_case(sensor, seed=seed)
    pts = rows[:, :5]
    eng = engine_mod.Engine(len(pts))
    eng.voxelize(dev(pts), 0.1)
    eng.build_maps()
    eng.status()
    c0, inv = O.voxelize(pts, 0.1)
    lv = O.Levels(c0)
    # level 0: identical rows in identical (first-occurrence) order, identical inverse map
    got0 = eng.coords(0)
    assert got0.shape == c0.shape and (got0 == c0).all()
    assert (eng.inverse_map() == inv).all()
    for L in range(5):
        got = eng.coords(L)
        assert (got == lv.coords[L]).all(), f"level {L} coordinates differ"
        nbr = eng.kernel_map(L, "3")
        assert (canon_kmap(nbr, got, got) == canon_kmap(lv.nbr3[L], lv.coords[L], lv.coords[L])).all()
        assert (nbr == lv.nbr3[L]).all()
    assert (eng.kernel_map(0, "5") == lv.nbr5).all()
    for L in range(4):
        pk = eng.parent(L)
        assert (pk >> 3 == lv.parent[L]).all() and (pk & 7 == lv.koff[L]).all()
        child = eng.kernel_map(L + 1, "child")
        # child table is the stride-2 kernel map: child[k][c] = the fine voxel f with parent c, offset k
        exp = np.full_like(child, -1)
        exp[lv.koff[L], lv.parent[L]] = np.arange(len(lv.parent[L]))
        assert (child == exp).all()


def test_quantisation_quirks(engine_mod):
    """fp32 division then floor: -0.05/0.1 -> -1; x/0.1f differs from x*10 on some inputs."""
    rng = np.random.default_rng(0)
    xyz = rng.uniform(-100, 100, (200000, 3)).astype(np.float32)
    special = np.array([[-0.05, 0.05, -0.1], [0.3, -0.3, 0.7], [1e-7, -1e-7, 0.0], [-0.0, 0.1, 0.2]], np.float32)
    xyz = np.vstack([special, xyz])
    pts = np.hstack([np.zeros((len(xyz), 1), np.float32), xyz, np.ones((len(xyz), 1), np.float32)])
    eng = engine_mod.Engine(len(pts))
    eng.voxelize(dev(pts), 0.1)
    eng.status()
    c0, inv = O.voxelize(pts, 0.1)
    assert (eng.coords(0) == c0).all() and (eng.inverse_map() == inv).all()
    assert tuple(c0[inv[0]][1:4]) == (-1, 0, -1)


def test_edge_inputs(engine_mod, state_dict):
    net = engine_mod.Net(state_dict)
    eng = engine_mod.Engine(4096)
    # empty input
    out = eng.forward(net, torch.zeros((0, 5), device="cuda"), 0.1)
    eng.status()
    assert out.shape == (0,)
    # one point / all points in one voxel / duplicates
    for pts in (np.array([[0, 1.0, 2.0, 3.0, 1]], np.float32),
                np.tile(np.array([[0, 1.01, 2.02, 3.03, 1]], np.float32), (100, 1)),
                np.array([[0, 0, 0, 0, 1], [0, 0, 0, 0, 0], [1, 0, 0, 0, 1], [1, 0, 0, 0, 0]], np.float32)):
        got = eng.forward(net, dev(pts), 0.1).cpu().numpy()
        eng.status()
        ref = O.sps_forward(pts, 0.1, state_dict)
        assert np.abs(got - ref).max() < 1e-5


def test_coordinate_range_is_reported(engine_mod, state_dict):
    from sps_b200._cabi import SpsError, SPS_ERR_COORD_RANGE
    eng = engine_mod.Engine(1024)
    pts = np.array([[0, 0, 0, 0, 1], [0, 2.0e4, 0, 0, 1], [300, 0, 0, 0, 1], [0, float("nan"), 0, 0, 1]], np.float32)
    eng.voxelize(dev(pts), 0.1)
    with pytest.raises(SpsError) as e:
        eng.status()
    assert e.value.code == SPS_ERR_COORD_RANGE
    eng.status()  # sticky word was cleared


def spread_state_dict(sd, pts, gain=8.0, voxel=0.1):
    """A state_dict whose scores behave like a trained checkpoint's: the head is amplified so that the scores span
    (0.05, 1) and the bias is moved so that the decision threshold eps = 0.84 (config/config.yaml:33) cuts through the
    middle of the score distribution.  The random-init head alone squashes every score into [0.46, 0.84): a parity
    bound measured there says nothing about thresholded labels."""
    sd = amplified(sd, gain)
    ref, _, _ = me_cpu.forward(pts, voxel, me_cpu.pack_weights(sd))
    logit = np.log(ref.astype(np.float64) / (1.0 - ref.astype(np.float64) + 1e-12) + 1e-12)
    shift = np.log(EPS / (1.0 - EPS)) - np.median(logit)
    sd["final.bias"] = (sd["final.bias"] + np.float32(shift)).astype(np.float32)
    return sd


@pytest.mark.tensor_path
@pytest.mark.parametrize("sensor,seed,submap", [("tiny", 3, "voxel"), ("hdl-32", 2, "voxel"), ("os1-64", 0, "radius")])
def test_scores_match_oracle(engine_mod, state_dict, sensor, seed, submap):
    """Default arithmetic (tcgen05 on fp16 rows for every layer but conv0; the 8-output-channel layers fold the low parts
    of their weights into spare accumulator columns; the level-0 concat buffer is stored as fp16 hi|lo pairs) against
    the fp32 oracle at the north-star bar: 2e-3 on the scores, >= 99.9 % equal labels -- on the contract
    network AND on weights whose scores spread over (0,1) and straddle eps (1x tolerance for both)."""
    rows = make_case(sensor, seed=seed, submap=submap, n_map_poses=6)
    pts = rows[:, :5]
    for sd in (state_dict, spread_state_dict(state_dict, pts)):
        net = engine_mod.Net(sd)
        eng = engine_mod.Engine(len(pts))
        got = eng.forward(net, dev(pts), 0.1).cpu().numpy()
        eng.status()
        ref, _, _ = me_cpu.forward(pts, 0.1, me_cpu.pack_weights(sd))
        err = np.abs(got - ref)
        assert err.max() < SCORE_TOL, f"max |score diff| {err.max():.3e}"
        agree = np.mean(O.threshold_labels(got, EPS) == O.threshold_labels(ref, EPS))
        assert agree >= 0.999
        if sd is not state_dict:      # the labels are really decided by the scores: both classes populated, wide spread
            unstable = np.mean(ref >= EPS)
            assert 0.2 < unstable < 0.8, unstable
            assert sensor == "tiny" or (ref.min() < 0.3 and ref.max() > 0.95), (ref.min(), ref.max())
    if sensor == "tiny":
        ref64 = O.sps_forward(pts, 0.1, sd, dtype=np.float64)
        assert np.abs(got - ref64).max() < SCORE_TOL


@pytest.mark.parametrize("sensor,seed", [("tiny", 3), ("hdl-32", 2)])
def test_scores_fp32_path_is_tight(engine_mod, state_dict, sensor, seed):
    """The fp32 CUDA-core path reproduces the oracle to rounding (1e-5), also with a 40x head gain."""
    rows = make_case(sensor, seed=seed, n_map_poses=6)
    pts = rows[:, :5]
    for sd in (state_dict, amplified(state_dict)):
        net = engine_mod.Net(sd)
        eng = engine_mod.Engine(len(pts))
        got = eng.forward(net, dev(pts), 0.1).cpu().numpy()
        eng.status()
        ref, _, _ = me_cpu.forward(pts, 0.1, me_cpu.pack_weights(sd))
        assert np.abs(got - ref).max() < 2e-5


def test_batched_scans_are_independent(engine_mod, state_dict):
    """Batch index is a coordinate that receives no kernel offset (blt_dataset.py:173-182)."""
    rows = make_case("tiny", seed=5, batch=3)
    pts = rows[:, :5]
    net = engine_mod.Net(state_dict)
    eng = engine_mod.Engine(len(pts))
    got = eng.forward(net, dev(pts), 0.1).cpu().numpy()
    eng.status()
    for b in range(3):
        sel = pts[:, 0] == b
        one = pts[sel].copy()
        one[:, 0] = 0
        ref = O.sps_forward(one, 0.1, state_dict)
        assert np.abs(got[sel] - ref).max() < 1e-5


def test_host_entry_point_and_model_api(engine_mod, state_dict):
    """SPSModel / SPSNet keep the reference call shape (models.py:13-30, 56-60, 84-104)."""
    from sps_b200.models import SPSNet
    rows = make_case("tiny", seed=7, batch=2)
    cfg = {"MODEL": {"VOXEL_SIZE": 0.1}, "FILTER": {"THRESHOLD": EPS}, "DATA": {"SPLIT": {"TEST": ["synthetic"]}}}
    model = SPSNet(cfg)
    model.model.MinkUNet.load_state_dict({k: torch.as_tensor(v) for k, v in state_dict.items()})
    model = model.cuda()
    model.freeze()
    ref = O.sps_forward(rows[:, :5], 0.1, state_dict)
    batch = torch.as_tensor(rows)
    got_host = model(batch)                       # CPU tensor -> sps_forward_host
    assert not got_host.is_cuda and np.abs(got_host.numpy() - ref).max() < 1e-5
    got_dev = model(batch.cuda())                 # CUDA tensor -> sps_forward
    assert got_dev.is_cuda and np.abs(got_dev.cpu().numpy() - ref).max() < 1e-5
    h1 = model.model.forward_async(batch[:, :5].contiguous().pin_memory())     # pipelined host entry point
    h2 = model.model.forward_async(batch[:, :5].contiguous().pin_memory())
    assert np.abs(h1.result(check=True).numpy() - ref).max() < 1e-5 and np.abs(h2.result().numpy() - ref).max() < 1e-5
    model.predict_step(batch.cuda(), 0)
    m = O.predict_step_metrics(ref, rows[:, 5], rows[:, 4], EPS)
    s = model.summary()
    assert abs(s["Loss"] - m["loss"]) < 1e-5 and abs(s["dIoU"] - m["dIoU"]) < 1e-6
    assert abs(s["Precision"] - m["precision"]) < 1e-6 and abs(s["Recall"] - m["recall"]) < 1e-6
    assert abs(s["F1"] - m["f1"]) < 1e-6 and abs(s["R2"] - m["r2"]) < 1e-3


def test_prune_crop_and_streamed_infer(engine_mod, state_dict):
    """util.to_coords_features / prune / infer (util.py:67-114,163-184) incl. the trunc-vs-floor
    lattice mismatch and the x ds round trip at negative coordinates."""
    from sps_b200 import synth, util
    world = synth.World(2)
    map_xyz = synth.base_map(world, "tiny", n_poses=8, seed=2)
    scan = synth.scan(world, "hdl-32", pose=(1.0, -2.0, 0.3), seed=9)
    ref_sub, ref_n = O.prune(map_xyz, scan, 0.1)
    map_cf = util.to_coords_features(torch.as_tensor(map_xyz), "map", 0.1)
    scan_cf = util.to_coords_features(torch.as_tensor(scan), "scan", 0.1)
    assert (map_cf.cloud_coords.cpu().numpy() == O.to_coords(map_xyz, 0.1)).all()
    sub, n_scan_vox = util.prune(map_cf, scan_cf, 0.1)
    assert n_scan_vox == ref_n
    sub = sub.cpu().numpy()
    assert sub.shape == ref_sub.shape
    assert (O.canonical(sub.view(np.int32)) == O.canonical(ref_sub.view(np.int32))).all()   # bit-exact fp32
    # deterministic order: first occurrence among the scan points
    cs, _ = O.unique_first(O.to_coords(scan, 0.1))
    lo, rng = O._extent(cs, O.to_coords(map_xyz, 0.1))
    keep = np.isin(O._pack(cs, lo, rng), O._pack(O.to_coords(map_xyz, 0.1), lo, rng))
    assert (sub == cs[keep].astype(np.float32) * np.float32(0.1)).all()

    class M:  # util.infer only needs .forward
        def __init__(self):
            from sps_b200.models import SPSModel
            self.m = SPSModel(0.1)
            self.m.MinkUNet.load_state_dict({k: torch.as_tensor(v) for k, v in state_dict.items()})
            self.m = self.m.cuda().eval()
        def forward(self, t):
            return self.m(t)
    model = M()
    scores, _ = util.infer(torch.as_tensor(scan).cuda(), torch.as_tensor(sub).cuda(), model)
    ref = O.infer(scan, ref_sub[np.lexsort(ref_sub.T[::-1])], 0.1, state_dict)
    assert np.abs(scores.cpu().numpy() - ref).max() < 1e-5
    # fused streamed path: crop + assemble + forward without host sync
    mh = map_cf.map_hash
    eng = engine_mod.Engine(2 * len(scan))
    net = engine_mod.Net(state_dict)
    out, counts = mh.infer_scan(eng, net, torch.as_tensor(scan).cuda(), 0.1)
    eng.status()
    assert counts.cpu().tolist() == [len(ref_sub), ref_n]
    assert np.abs(out.cpu().numpy() - ref).max() < 1e-5
    # radius crop (mapmos_node.py:63-68)
    idx = mh.crop_radius((1.0, -2.0, 1.8), 30.0).cpu().numpy()
    assert (idx == O.radius_crop(map_xyz.astype(np.float64), np.array([1.0, -2.0, 1.8]), 30.0)).all()


def test_generic_unet_entry_matches_fused_forward(engine_mod, state_dict):
    """sps_unet_forward (explicit feature vector, 5x5x5x1 table materialised) against the fused
    sps_forward (conv0 computed straight off the block table)."""
    rows = make_case("hdl-32", seed=6, n_map_poses=5)
    pts = rows[:, :5]
    net = engine_mod.Net(state_dict)
    eng = engine_mod.Engine(len(pts))
    fused = eng.forward(net, dev(pts), 0.1).cpu().numpy()
    eng.status()
    eng.voxelize(dev(pts), 0.1)
    eng.build_maps()
    v0 = eng.count(0)
    logits = eng.unet_forward(net, torch.full((v0,), 0.5, device="cuda")).cpu().numpy()
    inv = eng.inverse_map()
    generic = 1.0 / (1.0 + np.exp(-logits[inv].astype(np.float64)))
    assert np.abs(generic - fused).max() < 1e-6
    # a non-constant feature vector goes through the generic path only: check it against the oracle
    rng = np.random.default_rng(0)
    f = rng.uniform(0, 1, v0).astype(np.float32)
    got = eng.unet_forward(net, dev(f)).cpu().numpy()
    c0, _ = O.voxelize(pts, 0.1)
    ref = O.unet_forward(O.Levels(c0), f[:, None], state_dict)[:, 0]
    assert np.abs(got - ref).max() < 5e-5


def test_level_views_after_sorted_and_unsorted_passes(engine_mod, state_dict):
    """What sps_ctx_level hands out at every level: the dense 3x3x3x3 table after an unsorted forward, only the
    shape-sorted processing order (perm, tile masks, tile slices) after a sorted fused forward on the default backend,
    the table again after sps_build_maps, and both after a sorted forward on the exact fp32 backend."""
    rows = make_case("tiny", seed=3)
    pts = dev(rows[:, :5])
    net = engine_mod.Net(state_dict)
    eng = engine_mod.Engine(len(pts))

    def views():
        eng.status()
        return [eng.level(L) for L in range(5)]

    eng.set_conv_backend(0)
    eng.set_pattern_sort(0)
    eng.forward(net, pts, 0.1)
    for L, v in enumerate(views()):
        assert v.nbr3 and not v.perm and not v.tile_mask and not v.tile_slices, L
    eng.set_pattern_sort(2)
    eng.forward(net, pts, 0.1)
    for L, v in enumerate(views()):
        assert not v.nbr3 and v.perm and v.tile_mask and v.tile_slices, L
    eng.build_maps()
    for L, v in enumerate(views()):
        assert v.nbr3 and v.perm and v.tile_mask and v.tile_slices, L
    eng.set_conv_backend(1)
    eng.forward(net, pts, 0.1)
    for L, v in enumerate(views()):
        assert v.nbr3 and v.perm and v.tile_mask and v.tile_slices, L


@pytest.mark.tensor_path
def test_scan_streamer_graph_replay_matches_eager_call(engine_mod, state_dict):
    """ScanStreamer: the per-scan loop of sps_node.py:111-120 (prune -> assemble -> forward) captured once as a CUDA graph.
    Replays must reproduce the eager `infer_scan` bit for bit, for full-size scans and for shorter (padded) ones."""
    from sps_b200 import synth, util
    world = synth.World(4)
    map_xyz = synth.base_map(world, "tiny", n_poses=8, seed=4)
    mh = engine_mod.MapHash(torch.as_tensor(np.ascontiguousarray(map_xyz, np.float32)).cuda(), 0.1)
    scans = [synth.scan(world, "tiny", pose=(0.3 * i, -0.2 * i, 0.1 * i), seed=20 + i).astype(np.float32) for i in range(4)]
    n_scan = len(scans[0])
    net = engine_mod.Net(state_dict)
    streamer = engine_mod.ScanStreamer(mh, engine_mod.Engine(2 * n_scan), net, n_scan, 0.1)
    eager_engine = engine_mod.Engine(2 * n_scan)
    for i, s in enumerate(scans):
        pts = s if i % 2 == 0 else s[: n_scan - 37 * i]            # every other scan is shorter than the captured size
        d = torch.as_tensor(np.ascontiguousarray(pts)).cuda()
        got = streamer.infer(d).clone()
        ref, _ = mh.infer_scan(eager_engine, net, d, 0.1)
        eager_engine.status()
        torch.cuda.synchronize()
        assert got.shape == ref.shape == (len(pts),)
        assert torch.equal(got, ref), (i, float((got - ref).abs().max()))


def test_forward_async_graph_replay_equals_eager(engine_mod, state_dict):
    """forward_async replays the whole forward as a CUDA graph from the third call with the same input buffer on a lane:
    bit-identical to the eager call, for device inputs and for pinned host inputs, also after the input CONTENT changed
    (device-side counts: the captured launches do not depend on the data)."""
    from sps_b200.models import SPSModel
    rows_a = make_case("tiny", seed=21, batch=2)[:, :5]
    rows_b = make_case("tiny", seed=22, batch=2)[:, :5]
    n = min(len(rows_a), len(rows_b))
    rows_a, rows_b = np.ascontiguousarray(rows_a[:n]), np.ascontiguousarray(rows_b[:n])
    model = SPSModel(0.1)
    model.MinkUNet.load_state_dict({k: torch.as_tensor(v) for k, v in state_dict.items()})
    model = model.cuda().eval()
    model.lanes = 1
    assert model.use_graphs
    eager = {}
    for name, rows in (("a", rows_a), ("b", rows_b)):
        eager[name] = model(torch.as_tensor(rows).cuda()).cpu().numpy()
        model.check()
    for make in (lambda r: torch.as_tensor(r).cuda(), lambda r: torch.as_tensor(r).pin_memory()):
        buf = make(rows_a)
        outs = [model.forward_async(buf).result().cpu().numpy().copy() for _ in range(4)]   # eager, capture + replay, replay, replay
        for o in outs:
            assert np.array_equal(o, eager["a"])
        buf.copy_(torch.as_tensor(rows_b))              # same buffer, new content: the graph is still the right one
        if buf.is_cuda:
            torch.cuda.synchronize()
        assert np.array_equal(model.forward_async(buf).result().cpu().numpy(), eager["b"])


def test_two_host_threads_two_contexts(engine_mod, state_dict):
    """The library keeps no process-wide mutable state (include/sps_b200.h): two host threads drive two contexts on two
    streams at once, in DIFFERENT arithmetic modes, and each gets exactly what it gets alone."""
    import threading
    rows = [make_case("tiny", seed=31, batch=2)[:, :5], make_case("hdl-32", seed=32)[:, :5]]
    backends = [1, 0]
    net = engine_mod.Net(state_dict)
    alone = []
    for r, b in zip(rows, backends):
        eng = engine_mod.Engine(len(r))
        eng.set_conv_backend(b)
        alone.append(eng.forward(net, dev(r), 0.1).cpu().numpy())
        eng.status()
    results, errors = [None, None], []

    def work(i):
        try:
            eng = engine_mod.Engine(len(rows[i]))
            eng.set_conv_backend(backends[i])
            eng.profile(i == 0)                               # per-context stage timers too
            stream = torch.cuda.Stream()
            d = dev(rows[i])
            torch.cuda.current_stream().synchronize()
            with torch.cuda.stream(stream):
                for _ in range(10):
                    out = eng.forward(net, d, 0.1)
                stream.synchronize()
            eng.status()
            results[i] = out.cpu().numpy()
        except Exception as e:   # noqa: BLE001
            errors.append(e)
    threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i in range(2):
        assert np.array_equal(results[i], alone[i])
