"""The level-0 paths of the fused forward against float64, read out through the network's own head with probe weights
(tests/probe_nets.py):

* probe A: the presence signature of conv0 -- ``k_conv0_const`` (``forward``) and ``k_conv0_blk`` (``forward_features``)
  must reproduce every voxel's 125-neighbour presence set exactly, on the fp32, TF32 and fp16 backends;
* probe A': conv0 with random weights on random per-voxel features against float64;
* probe B: conv1p1s2 -> identity block -> convtr7p2s2, i.e. the stride-2 map into level 1 and the transposed convolution
  back in child-class order (``k_up_order``'s ``perm_up`` / ``tmask_up`` on the TF32 and fp16 backends, ``k_conv_up`` on
  fp32), against float64 with the backend's storage roundings;

on inputs at the edges of the 4x4x4 blocks, the key lattice, the time planes and batches, the child-class tile
boundaries, on real data and on inputs large enough for the shape sort and for second turns of the grid-stride loops.
Also: points outside the key range score NaN, probe B does not depend on the shape sort, and the per-point-feature
path's voxel mean against float64."""
import numpy as np
import pytest
import torch

import probe_nets as P
from conftest import make_case
from oracle import sps_oracle as O

pytestmark = pytest.mark.gpu

BACKENDS = (1, 2, 0)            # exact fp32, TF32 operands on fp32 rows, fp16 rows (the default)
CASES = P.EDGE_CASES + ("hdl-32",) + P.LARGE_CASES
REPORT = {}                     # (probe, case, backend) -> largest error as a fraction of its bound


class Input:
    """Points on the device, their voxels in first-occurrence order, the sampled rows and their references' inputs."""

    def __init__(self, name):
        from sps_b200 import engine
        if name == "hdl-32":
            pts = make_case("hdl-32", seed=1)[:, :5].astype(np.float32)
            self.vs = 0.1
            self.c0, inv = O.voxelize(pts, self.vs)
        else:
            coords, bad = P.edge_input(name)
            pts = np.vstack([P.to_points(coords), P.to_points(bad)])
            self.vs = 1.0
            self.c0 = coords
            inv = np.concatenate([np.arange(len(coords)), np.full(len(bad), -1)])
        self.inv = np.asarray(inv, np.int64)
        V = len(self.c0)
        valid = np.flatnonzero(self.inv >= 0)
        self.bad = np.flatnonzero(self.inv < 0)
        self.first = np.full(V, -1, np.int64)
        self.first[self.inv[valid[::-1]]] = valid[::-1]
        assert np.bincount(self.inv[valid]).max() < 1 << (24 - P.FEAT_BITS)    # voxel means of equal features stay exact
        self.rows = P.sample_rows(V)
        self.lookup = P.Lookup(self.c0)
        self.nbr = P.nbr5_rows(self.lookup, self.c0, self.rows)
        self.vfeat = P.voxel_features(V, np.random.default_rng(5))
        pfeat = np.full(len(pts), 0.75)
        pfeat[valid] = self.vfeat[self.inv[valid]]
        self.pts = torch.from_numpy(pts).cuda()
        self.ones = torch.ones(len(pts), dtype=torch.float32, device="cuda")
        self.feat = torch.from_numpy(pfeat.astype(np.float32)).cuda()
        self.engine = engine.Engine(len(pts))

    def run(self, nets, feat=None, backend=None, sort=1):
        """Channel c of the probed tensor at the sampled voxels, [R, 8] (one forward per output column)."""
        eng = self.engine
        eng.set_conv_backend(backend)
        eng.set_pattern_sort(sort)
        cols = []
        for net in nets:
            if feat is None:
                cols.append(eng.forward(net, self.pts, self.vs))
            else:
                cols.append(eng.forward_features(net, self.pts, feat, self.vs))
        out = torch.stack(cols, 1).cpu().numpy()
        assert np.isnan(out[self.bad]).all(), "points outside the key range must score NaN"
        valid = self.inv >= 0
        vox = out[self.first]
        assert np.isfinite(vox).all()
        assert np.array_equal(out[valid], vox[self.inv[valid]])
        return vox[self.rows].astype(np.float64)


_inputs = {}


def get_input(name):
    if name not in _inputs:
        _inputs[name] = Input(name)
    return _inputs[name]


@pytest.fixture(scope="module")
def nets():
    from sps_b200 import engine
    mk = lambda sd: [engine.Net(sd, output_channel=c, apply_sigmoid=False) for c in range(8)]
    yield {"A0": mk(P.probe_a(0)), "A1": mk(P.probe_a(1)), "A'": mk(P.probe_a_numeric()), "B": mk(P.probe_b())}
    _inputs.clear()
    if REPORT:
        print("\nlargest error / bound (probe, case, backend):")
        for (probe, case, backend), r in sorted(REPORT.items()):
            print(f"  {probe:3s} {case:18s} backend {backend}: {r:.3e}")


def check_bound(probe, name, backend, got, ref, lim):
    err = np.abs(got - ref)
    ratio = float((err / lim).max(initial=0.0))
    REPORT[(probe, name, backend)] = ratio
    if ratio > 1:
        r, c = np.unravel_index(np.argmax(err / lim), err.shape)
        pytest.fail(f"probe {probe}, {name}, backend {backend}: row {r} channel {c}: got {got[r, c]!r}, "
                    f"want {ref[r, c]!r}, error {err[r, c]:.3e} > bound {lim[r, c]:.3e}")


@pytest.mark.parametrize("name", CASES)
def test_conv0_presence_signature(nets, name):
    """Probe A: both conv0 kernels find exactly the present neighbours of every voxel, in every storage format."""
    inp = get_input(name)
    present = inp.nbr >= 0
    for backend in BACKENDS:
        for feat, c, kernel in ((None, 0.5, "k_conv0_const"), (inp.ones, 1.0, "k_conv0_blk")):
            got = [inp.run(nets[f"A{p}"], feat, backend) for p in (0, 1)]
            for p in (0, 1):
                want = P.signature_values(present, c, p)
                bad = np.flatnonzero((got[p] != want).any(1))
                assert len(bad) == 0, (f"{kernel}, backend {backend}, pass {p}: {len(bad)} of {len(want)} rows differ, "
                                       f"first row {inp.rows[bad[0]]}: got {got[p][bad[0]]}, want {want[bad[0]]}")
            assert np.array_equal(P.decode_signature(got[0], got[1], c), present)
            REPORT[("A", name, backend)] = 0.0


@pytest.mark.parametrize("name", CASES)
def test_conv0_numerics(nets, name):
    """Probe A': k_conv0_blk with random weights and per-voxel features against float64, within 2^-22 S (fp32),
    2^-10 S (TF32 store) and 2^-19 S (hi|lo store), S = sum of |w x| and the shift."""
    inp = get_input(name)
    ref, S = P.conv0_rows(inp.nbr, inp.vfeat, P.probe_a_numeric())
    for backend in BACKENDS:
        got = inp.run(nets["A'"], inp.feat, backend)
        check_bound("A'", name, backend, got, ref, P.BOUND_A_NUMERIC[backend] * S)


@pytest.mark.parametrize("name", CASES)
def test_stride2_and_transposed_into_level0(nets, name):
    """Probe B: conv1p1s2 -> block1 -> block7's downsample -> convtr7p2s2 against float64 with the backend's storage
    roundings; the tensor-core backends give the same bits with the shape sort off and forced."""
    inp = get_input(name)
    sd = P.probe_b()
    for backend in BACKENDS:
        ref, S, flip = P.probe_b_rows(inp.lookup, inp.c0, inp.vfeat, sd, inp.rows, backend)
        got = inp.run(nets["B"], inp.feat, backend)
        check_bound("B", name, backend, got, ref, P.BOUND_B[backend] * S + flip)
        if backend != 1:
            for sort in (0, 2):
                assert np.array_equal(inp.run(nets["B"], inp.feat, backend, sort), got), f"backend {backend}, sort {sort}"


def test_voxel_mean_of_fractional_point_features():
    """forward_features averages the point features of a voxel: within n 2^-24 relative of the float64 mean for a
    voxel of n >= 2 points (n - 1 fp32 additions and a division), exact for one point; bit-identical from run to run
    for voxels of at most two points, whose sum does not depend on the order of the additions."""
    from sps_b200 import engine
    pts = make_case("hdl-32", seed=1)[:, :5].astype(np.float32)
    c0, inv = O.voxelize(pts, 0.1)
    n = np.bincount(inv)
    feats = np.random.default_rng(11).uniform(0.0, 1.0, len(pts)).astype(np.float32)
    mean = np.bincount(inv, weights=feats.astype(np.float64)) / n
    sd = P.zero_net("skip0")
    sd["conv0p1s1.kernel"][P.CENTRE, 0, 0] = 1.0         # channel 0 of skip0 = the voxel mean
    net = engine.Net(sd, output_channel=0, apply_sigmoid=False)
    eng = engine.Engine(len(pts))
    eng.set_conv_backend(1)
    p, f = torch.from_numpy(pts).cuda(), torch.from_numpy(feats).cuda()
    runs = [eng.forward_features(net, p, f, 0.1).cpu().numpy() for _ in range(2)]
    first = np.full(len(c0), -1, np.int64)
    first[inv[::-1]] = np.arange(len(pts))[::-1]
    got = runs[0][first].astype(np.float64)
    lim = np.where(n > 1, n * 2.0 ** -24 * mean, 0.0)
    assert (n >= 3).sum() > 100                       # the case has many voxels of three or more points
    bad = np.flatnonzero(np.abs(got - mean) > lim)
    assert len(bad) == 0, f"{len(bad)} voxels, first {bad[0]}: {got[bad[0]]!r} vs {mean[bad[0]]!r} ({n[bad[0]]} points)"
    small = n[inv] <= 2
    assert np.array_equal(runs[0][small], runs[1][small])
    print(f"\nvoxel mean: {(n >= 3).sum()} voxels of >= 3 points, {int((runs[0] != runs[1]).sum())} points differ "
          f"between two runs, largest error {float((np.abs(got - mean) / np.maximum(n * 2.0 ** -24 * mean, 1e-30)).max()):.3f}"
          " of the bound")
