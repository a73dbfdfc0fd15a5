"""Every layer of the fused forward beyond level 0 against float64, read out through the network's own head with probe
weights (tests/probe_nets.py, ``deep_probe``): the stride-2 convs into levels 2..4, both convs of every block (the
fused 1x1 downsample term with its BN shift, two-segment rows, hi|lo rows, folded low weight parts, the fused head),
and the transposed convs into levels 1..3, each on exact lifted inputs, against the float64 reference with the
backend's weight rounding (``PLAN``) within one storage ulp + 2^-20 S, on the fp32, TF32 and fp16 backends.  The
tensor-core backends run with the shape sort off and forced: 81-offset layers must meet the bound both ways, stride-2
and transposed layers must give the same bits.  The edge inputs also go through the generic ``sps_unet_forward``
(dense maps, physical-order tile masks) on the fp32 and TF32 backends."""
import numpy as np
import pytest
import torch

import probe_nets as P
from conftest import make_case
from oracle import sps_oracle as O

pytestmark = pytest.mark.gpu

BACKENDS = (1, 2, 0)
CASES = P.EDGE_CASES + P.DEEP_CASES + ("hdl-32",) + P.LARGE_CASES
LARGE_COLUMNS = (0, 7)          # the first and last channel of every group on the large inputs
REPORT = {}                     # (layer, backend) -> (largest error / bound, case)


class Input:
    """Points on the device, the levels of their voxels, the lifted tensors and the sampled rows."""

    def __init__(self, name):
        from sps_b200 import engine
        if name == "hdl-32":
            pts = make_case("hdl-32", seed=1)[:, :5].astype(np.float32)
            self.vs = 0.1
            c0, inv = O.voxelize(pts, self.vs)
            bad = np.zeros((0, 5), np.int64)
        else:
            c0, bad = P.edge_input(name)
            pts = np.vstack([P.to_points(c0), P.to_points(bad)])
            self.vs = 1.0
            inv = np.concatenate([np.arange(len(c0)), np.full(len(bad), -1)])
        self.inv = np.asarray(inv, np.int64)
        V = len(c0)
        valid = np.flatnonzero(self.inv >= 0)
        self.bad = np.flatnonzero(self.inv < 0)
        self.first = np.full(V, -1, np.int64)
        self.first[self.inv[valid[::-1]]] = valid[::-1]
        self.large = name in P.LARGE_CASES
        self.rows = P.sample_rows(V)
        vfeat = P.deep_features(V, np.random.default_rng(5))
        self.dl = P.DeepLevels(c0, vfeat)
        pfeat = np.full(len(pts), 0.75)
        pfeat[valid] = vfeat[self.inv[valid]]
        self.pts = torch.from_numpy(pts).cuda()
        self.feat = torch.from_numpy(pfeat.astype(np.float32)).cuda()
        self.engine = engine.Engine(len(pts))
        self.generic = None
        if name in P.EDGE_CASES:           # the generic entry: voxel features in the engine's level-0 row order
            self.generic = (torch.from_numpy(P.to_points(c0)).cuda(), torch.from_numpy(vfeat.astype(np.float32)).cuda())

    def run(self, nets, backend, sort=1):
        """[R, ncols] readout of the sampled level-0 voxels, one fused forward per column."""
        eng = self.engine
        eng.set_conv_backend(backend)
        eng.set_pattern_sort(sort)
        out = torch.stack([eng.forward_features(net, self.pts, self.feat, self.vs) for net in nets], 1).cpu().numpy()
        assert np.isnan(out[self.bad]).all(), "points outside the key range must score NaN"
        valid = self.inv >= 0
        vox = out[self.first]
        assert np.isfinite(vox).all()
        assert np.array_equal(out[valid], vox[self.inv[valid]])
        return vox[self.rows].astype(np.float64)

    def run_generic(self, nets, backend):
        pts, feat0 = self.generic
        eng = self.engine
        eng.set_conv_backend(backend)
        eng.set_pattern_sort(1)
        eng.voxelize(pts, 1.0)
        eng.build_maps()
        assert np.array_equal(eng.coords(0), self.dl.c[0])
        out = torch.stack([eng.unet_forward(net, feat0) for net in nets], 1).cpu().numpy()
        return out[self.rows].astype(np.float64)


_inputs = {}


def get_input(name):
    if name not in _inputs:
        _inputs.clear()                   # one input at a time: the large ones hold big engines
        _inputs[name] = Input(name)
    return _inputs[name]


@pytest.fixture(scope="module")
def nets():
    """layer -> [(column of the tensor under test, Net)], each Net built once."""
    from sps_b200 import engine
    cache = {}

    def get(layer):
        if layer not in cache:
            cols = []
            for g in range(P.deep_groups(layer)):
                sd = P.deep_probe(layer, g)
                cols += [(8 * g + c, engine.Net(sd, output_channel=c, apply_sigmoid=False)) for c in range(8)]
            cache[layer] = cols
        return cache[layer]
    yield get
    cache.clear()
    _inputs.clear()
    if REPORT:
        print("\nlargest error / bound per layer and backend (case):")
        for (layer, backend), (r, case) in sorted(REPORT.items()):
            print(f"  {layer:14s} backend {backend}: {r:.3e} ({case})")


def check(layer, name, backend, got, ref, lim, what=""):
    err = np.abs(got - ref)
    ratio = float((err / lim).max(initial=0.0))
    key = (layer, backend)
    if ratio >= REPORT.get(key, (-1.0, ""))[0]:
        REPORT[key] = (ratio, name + what)
    if ratio > 1:
        r, c = np.unravel_index(np.argmax(err / lim), err.shape)
        pytest.fail(f"{layer}, {name}{what}, backend {backend}: row {r} column {c}: got {got[r, c]!r}, want {ref[r, c]!r}, "
                    f"error {err[r, c]:.3e} > bound {lim[r, c]:.3e}")


def same_per_ancestor(inp, layer, got):
    """Every sampled level-0 descendant of a level-L voxel reads the same value."""
    L = P.probe_info(layer)[0]
    anc = inp.dl.ancestors(L, inp.rows)
    _, first = np.unique(anc, return_index=True)
    _, inv = np.unique(anc, return_inverse=True)
    assert np.array_equal(got, got[first][inv]), f"{layer}: descendants of one level-{L} voxel differ"


@pytest.mark.parametrize("layer", P.DEEP_LAYERS)
@pytest.mark.parametrize("name", CASES)
def test_deep_probe(nets, layer, name):
    inp = get_input(name)
    cols = nets(layer)
    if inp.large:
        cols = [(ch, net) for ch, net in cols if ch % 8 in LARGE_COLUMNS]
    ch = [c for c, _ in cols]
    sd = P.deep_probe(layer)
    logit = layer == "block8.conv2"
    for backend in BACKENDS:
        ref, lim, margin = (a[:, ch] for a in P.deep_reference(inp.dl, layer, sd, backend, inp.rows))
        if backend == 1 or logit:         # a lost product, weight half or shift cannot hide under the bound
            assert (margin > 0).all(), f"{layer}, {name}: bound not below the smallest product"
        nets_ = [net for _, net in cols]
        if backend == 1:
            got = inp.run(nets_, backend)
            same_per_ancestor(inp, layer, got)
            check(layer, name, backend, got, ref, lim)
            continue
        runs = [inp.run(nets_, backend, sort) for sort in (0, 2)]
        for sort, got in zip((0, 2), runs):
            same_per_ancestor(inp, layer, got)
            check(layer, name, backend, got, ref, lim, f" sort {sort}")
        if P.PLAN[layer][0] == 8:          # stride-2 and transposed layers: the tile order does not reach the bits
            assert np.array_equal(runs[0], runs[1]), f"{layer}, {name}, backend {backend}: sort 0 and 2 differ"


@pytest.mark.parametrize("layer", P.DEEP_LAYERS)
@pytest.mark.parametrize("name", P.EDGE_CASES)
def test_deep_probe_generic_entry(nets, layer, name):
    inp = get_input(name)
    cols = nets(layer)
    ch = [c for c, _ in cols]
    sd = P.deep_probe(layer)
    for backend in (1, 2):
        ref, lim, _ = (a[:, ch] for a in P.deep_reference(inp.dl, layer, sd, backend, inp.rows))
        got = inp.run_generic([net for _, net in cols], backend)
        check(layer, name, backend, got, ref, lim, " generic")
