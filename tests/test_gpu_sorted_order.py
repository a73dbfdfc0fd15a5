"""The shape-sorted processing order of the 3x3x3x3 convolutions, pinned bit for bit: perm, tile masks and tile slices of
all five levels against the numpy statement in tests/sorted_order_ref.py (integer equality), after a fused forward,
after sps_build_maps and after a forward on the exact fp32 backend; the layer-level convolution on those structures
against float64 numpy; and the sorted 4-D forward (three or more time planes) against the oracle."""
import contextlib
import functools

import numpy as np
import pytest
import torch

import sorted_order_ref as R
from conftest import make_case
from oracle import sps_oracle as O

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def default_pattern_sort(mode):
    from sps_b200 import engine
    old = engine.DEFAULTS["pattern_sort"]
    engine.set_defaults(pattern_sort=mode)
    try:
        yield
    finally:
        engine.set_defaults(pattern_sort=old)


@pytest.fixture
def sort_always():
    """Shape-sort every forward of the engines created in the test (sps_ctx_set_pattern_sort 2)."""
    with default_pattern_sort(2):
        yield


@pytest.fixture(scope="module")
def net():
    from sps_b200 import engine
    return engine.Net(O.make_state_dict(seed=0, randomize_bn=True))


# ---------------------------------------------------------------- inputs ----
def window(n_scans, seed=0):
    """A MOS4D sliding window: rows (b = 0, x, y, z, t = scan index 0..n_scans-1) of scans from a moving pose, plus a
    dense 6x6x6-voxel cube in three consecutive scans (the scans alone leave no tile with all 81 offsets)."""
    from sps_b200 import synth
    world = synth.World(seed)
    rows = []
    for i in range(n_scans):
        xyz = synth.scan(world, "tiny", pose=(0.4 * i, -0.2 * i, 0.05 * i), seed=seed + i).astype(np.float32)
        rows.append(np.hstack([np.zeros((len(xyz), 1), np.float32), xyz, np.full((len(xyz), 1), i, np.float32)]))
    g = np.arange(6)
    cube = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3) * 0.1 + np.array([100.05, 100.05, 0.05])
    for i in range(n_scans // 2 - 1, n_scans // 2 + 2):
        rows.append(np.hstack([np.zeros((len(cube), 1)), cube, np.full((len(cube), 1), i)]).astype(np.float32))
    return np.vstack(rows)


def compress_axis(v):
    """Shrink every gap of more than 64 between the distinct values of one axis by a multiple of 16.  Neighbourhoods
    (at most 16 apart at level 4), the stride-2^L cells and the row order are unchanged, so the oracle's maps of the
    shrunk coordinates are the maps of the originals -- whose extent over the whole key range the oracle cannot pack."""
    u = np.unique(v)
    gaps = np.diff(u)
    shift = np.concatenate([[0], np.cumsum(np.where(gaps > 64, (gaps - 64) // 16 * 16, 0))])
    return (u - shift)[np.searchsorted(u, v)]


def oracle_levels(c0):
    """Row counts and 3x3x3x3 kernel maps of the five levels (the oracle's Levels without the 5x5x5x1 map)."""
    c0 = np.array(c0, np.int64)
    for d in (1, 2, 3):
        c0[:, d] = compress_axis(c0[:, d])
    coords = [c0]
    for L in range(4):
        coords.append(O.stride_coords(coords[L], 2 ** (L + 1))[0])
    nbr3 = [O.kernel_map(coords[L], coords[L], O.kernel_offsets([3, 3, 3, 3], [2 ** L] * 3 + [1])) for L in range(5)]
    return [len(c) for c in coords], nbr3


def adversarial(delta):
    """Voxel size 1: an isolated voxel, a 6x6x6 cube present in three consecutive scans, voxels on the faces of the key
    range with a neighbour inside it along every axis, padded so that the keys of all levels number 2048 k + delta."""
    vox = [(0, 1000, 1000, 100, 7)]
    vox += [(0, 2000 + x, 2000 + y, 200 + z, t) for t in (4, 5, 6) for z in range(6) for y in range(6) for x in range(6)]
    for b in (0, 254):
        for x in (-131072, 131071):
            for y in (-131072, 131071):
                for z in (-32768, 32767):
                    for t in (0, 15):
                        inward = lambda c, lo: c + 1 if c == lo else c - 1
                        vox += [(b, x, y, z, t), (b, inward(x, -131072), y, z, t), (b, x, inward(y, -131072), z, t),
                                (b, x, y, inward(z, -32768), t), (b, x, y, z, inward(t, 0))]
    base = np.array(vox, np.int64)
    counts, _ = oracle_levels(base)
    total = sum(counts)
    k = total // R.SORT_TILE + 2                  # three sort tiles: look-back across two predecessors
    if R.SORT_TILE * k + delta - total < 20:
        k += 1
    pad = R.SORT_TILE * k + delta - total
    n_iso, n_pair = pad // 5, pad % 5
    # an isolated voxel adds one row to every level (its own stride-16 cell); a second voxel in the same stride-2 cell
    # as an isolated one adds one row at level 0 only
    iso = [(1, 5000 + 64 * i, 5000, 0, 3) for i in range(n_iso)]
    pair = [(1, 5000 + 64 * i + 1, 5000, 0, 3) for i in range(n_pair)]
    c = np.vstack([base, np.array(iso + pair, np.int64).reshape(-1, 5)])
    c = c[np.random.default_rng(7).permutation(len(c))]
    return c.astype(np.float32), R.SORT_TILE * k + delta


class Case:
    def __init__(self, name):
        self.name = name
        self.target = None
        if name == "tiny":
            self.pts, self.vs, self.mode = make_case("tiny", seed=3)[:, :5], 0.1, 2
        elif name == "hdl-32":
            self.pts, self.vs, self.mode = make_case("hdl-32", seed=1)[:, :5], 0.1, 2
        elif name == "os1-64-radius-b2":
            self.pts, self.vs, self.mode = make_case("os1-64", submap="radius", batch=2)[:, :5], 0.1, 1
        elif name.startswith("mos4d-"):
            self.pts, self.vs, self.mode = window(int(name.split("-")[1])), 0.1, 2
        elif name.startswith("edges"):
            delta = {"edges-1": -1, "edges+0": 0, "edges+1": 1}[name]
            (self.pts, self.target), self.vs, self.mode = adversarial(delta), 1.0, 2
        self.pts = np.ascontiguousarray(self.pts, np.float32)
        q = O.quantize(self.pts, self.vs).astype(np.int64)      # O.voxelize, with the spatial axes shrunk first
        for d in (1, 2, 3):
            q[:, d] = compress_axis(q[:, d])
        c0, _ = O.unique_first(q)
        self.counts, self.nbr3 = oracle_levels(c0)
        self.ref = [R.level_order(self.nbr3[L], L) for L in range(5)]

    def stats(self):
        """Largest number of present offsets of a tile per level, sort tiles, rows with both t-1 and t+1 neighbours."""
        both = sum(int(((r["presence"][:, 0] != 0) & (r["presence"][:, 2] != 0)).sum()) for r in self.ref)
        return [int(r["nact"].max()) if len(r["nact"]) else 0 for r in self.ref], R.sort_tiles(self.counts), both


@functools.lru_cache(maxsize=None)
def case(name):
    return Case(name)


CASES = ["tiny", "hdl-32", "os1-64-radius-b2", "mos4d-4", "mos4d-16", "edges-1", "edges+0", "edges+1"]


# ---------------------------------------------------------------- structures ----
def read_level(eng, L, V):
    v = eng.level(L)
    assert v.perm and v.tile_mask and v.tile_slices, L
    nt = R.n_tiles(V)
    return (eng._read(v.perm, V, np.int32), eng._read(v.tile_mask, 4 * nt, np.uint32).reshape(nt, 4),
            eng._read(v.tile_slices, nt * R.SLICE_ENTRIES * R.TILE, np.int32).reshape(nt, R.SLICE_ENTRIES, R.TILE))


def check_levels(eng, c, where):
    got = []
    for L in range(5):
        ref = c.ref[L]
        V = c.counts[L]
        assert eng.count(L) == V, (where, L)
        perm, masks, slices = read_level(eng, L, V)
        assert np.array_equal(perm, ref["perm"]), (where, L, int((perm != ref["perm"]).sum()), "rows of perm differ")
        bad = np.nonzero((masks != ref["tile_mask"]).any(axis=1))[0]
        assert len(bad) == 0, (where, L, "tile masks differ", bad[:8])
        d = R.defined_entries(ref["nact"])
        bad = np.nonzero((slices[d] != ref["tile_slices"][d]).any(axis=1))[0]
        assert len(bad) == 0, (where, L, len(bad), "slice entries differ")
        got.append((perm, masks, slices[d]))
    return got


@pytest.mark.parametrize("name", CASES)
def test_sorted_order_structures_match_reference(name, net):
    """perm, tile masks and the defined tile-slice entries of all five levels equal the numpy statement exactly: twice
    after a fused forward on the default backend (sparse tables), after sps_build_maps (dense tables, which also equal
    the oracle's kernel maps), after a forward on the exact fp32 backend."""
    from sps_b200 import engine
    c = case(name)
    nact, tiles, both = c.stats()
    if name.startswith(("mos4d", "edges")):
        assert max(nact) == 81 and both > 0, (nact, both)      # every slice entry is used; rows see t-1 and t+1
    if c.target is not None:
        assert sum(c.counts) == c.target, (c.counts, c.target)
    eng = engine.Engine(len(c.pts))
    eng.set_conv_backend(0)
    eng.set_pattern_sort(c.mode)
    d = torch.as_tensor(c.pts).cuda()
    runs = []
    for rep in range(2):
        eng.forward(net, d, c.vs)
        eng.status()
        runs.append(check_levels(eng, c, f"forward {rep}"))
        assert not any(eng.level(L).nbr3 for L in range(5))    # the sorted forward keeps only present entries
    for a, b in zip(*runs):
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    eng.set_pattern_sort(2)
    eng.build_maps()
    eng.status()
    check_levels(eng, c, "build_maps")
    for L in range(5):
        assert np.array_equal(eng.kernel_map(L, "3"), c.nbr3[L]), L
    eng.set_pattern_sort(c.mode)
    eng.set_conv_backend(1)
    eng.forward(net, d, c.vs)
    eng.status()
    check_levels(eng, c, "fp32 forward")


def test_default_mode_sorts_from_400000_rows(net):
    from sps_b200 import engine
    c = case("os1-64-radius-b2")
    assert len(c.pts) > 400_000
    eng = engine.Engine(len(c.pts))
    eng.set_pattern_sort(1)
    d = torch.as_tensor(c.pts).cuda()
    for n, sorted_ in ((399_999, False), (400_000, True), (len(c.pts), True)):
        eng.forward(net, d[:n], c.vs)
        eng.status()
        assert all(bool(eng.level(L).perm) == sorted_ for L in range(5)), n


# ---------------------------------------------------------------- layer-level convolution ----
def f16(x):
    return np.ascontiguousarray(x, np.float32).astype(np.float16).astype(np.float32)


def ref_conv(x, nbr, w, shift=None, x2=None, w2=None, res=None, relu=False, quant=None):
    q = quant or (lambda v: v)
    K, V = nbr.shape
    out = np.zeros((V, w.shape[-1]), np.float64)
    xq, wq = q(x).astype(np.float64), q(w).astype(np.float64)
    for k in range(K):
        o = np.nonzero(nbr[k] >= 0)[0]
        out[o] += xq[nbr[k, o]] @ wq[k]
    if x2 is not None:
        out += q(x2).astype(np.float64) @ q(w2).astype(np.float64)
    if shift is not None:
        out += shift
    if res is not None:
        out += res
    return np.maximum(out, 0) if relu else out


# the network's 3x3x3x3 layer shapes per level: (cin, cout, cin_split)
LAYERS = {0: [(8, 8, 0)], 1: [(16, 16, 0)], 2: [(32, 32, 0)], 3: [(64, 64, 0), (96, 64, 64)], 4: [(64, 64, 0)]}


@pytest.mark.parametrize("name", ["mos4d-16", "os1-64-radius-b2"])
def test_layer_convolution_on_the_sorted_order(name, net):
    """sps_conv_fwd with fp16 rows on every level's own perm / tile masks / tile slices of a sorted forward: equal to
    float64 numpy on the oracle's map at the fp16 bound, within one fp16 ulp plus fp32 reordering noise of the same call
    in physical order, and bit-equal to the call that gathers through perm from the dense map instead of the slices."""
    from sps_b200 import convops, engine, _cabi
    c = case(name)
    eng = engine.Engine(len(c.pts))
    eng.set_conv_backend(0)
    eng.set_pattern_sort(2)
    eng.forward(net, torch.as_tensor(c.pts).cuda(), c.vs)
    eng.status()
    rng = np.random.default_rng(11)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a)).cuda()
    calls = []
    for L, shapes in LAYERS.items():
        V = c.counts[L]
        n_out = torch.tensor([V], dtype=torch.int32, device="cuda")
        for cin, cout, cs in shapes:
            for kind in ("relu", "fused", "res"):
                x = rng.standard_normal((V, cin)).astype(np.float32)
                w = (rng.standard_normal((81, cin, cout)) / np.sqrt(cin * 8)).astype(np.float32)
                w2 = (rng.standard_normal((cin, cout)) / np.sqrt(cin)).astype(np.float32) if kind == "fused" else None
                shift = rng.standard_normal(cout).astype(np.float32)
                res = rng.standard_normal((V, cout)).astype(np.float32) if kind == "res" else None
                fold = cout == 8
                wt = convops.pack_kmajor_f16x(t(w), t(w2) if w2 is not None else None, cin_split=cs, fold_lo=fold)
                kw = dict(shift=t(shift), relu=kind != "res", in2=t(x).half() if w2 is not None else None,
                          weight2=t(w2) if w2 is not None else None, res=t(res).half() if res is not None else None,
                          weight_kmajor=wt, io_f16=True, backend=_cabi.SPS_BACKEND_F16, cin_split=cs,
                          flags=_cabi.SPS_CONV_FOLD_LO if fold else 0, n_out_max=V)
                calls.append(dict(L=L, shape=(cin, cout, cs, kind), x=x, w=w, w2=w2, shift=shift, res=res, fold=fold,
                                  xd=t(x).half(), wd=t(w), n_out=n_out, kw=kw))
    # (a) the forward's own views: sparse tables, so the slices are the only map
    for cl in calls:
        v = eng.level(cl["L"])
        assert not v.nbr3
        out = convops.conv_fwd(cl["xd"], cl["wd"], cl["n_out"], perm=v.perm, tile_mask=v.tile_mask,
                               tile_slices=v.tile_slices, **cl["kw"])
        cl["sorted"] = out[:c.counts[cl["L"]]].float().cpu().numpy()
    eng.build_maps()
    eng.status()
    for cl in calls:
        v = eng.level(cl["L"])
        V = c.counts[cl["L"]]
        # (b) physical order, tile masks of the dense map; (c) sorted order gathered through perm from the dense map
        phys = convops.conv_fwd(cl["xd"], cl["wd"], cl["n_out"], map=v.nbr3, map_ld=v.ld, **cl["kw"])
        via_perm = convops.conv_fwd(cl["xd"], cl["wd"], cl["n_out"], map=v.nbr3, map_ld=v.ld, perm=v.perm,
                                    tile_mask=v.tile_mask, **cl["kw"])
        phys = phys[:V].float().cpu().numpy()
        via_perm = via_perm[:V].float().cpu().numpy()
        got = cl["sorted"]
        nbr = c.nbr3[cl["L"]]
        # operands as the kernel sees them: fp16 rows; fp16 weights, or exact ones when the low parts are folded in
        xq = f16(cl["x"])
        wq, w2q = (cl["w"], cl["w2"]) if cl["fold"] else (f16(cl["w"]), None if cl["w2"] is None else f16(cl["w2"]))
        x2q = None if cl["w2"] is None else xq
        ref = ref_conv(xq, nbr, wq, shift=cl["shift"], x2=x2q, w2=w2q, res=None if cl["res"] is None else f16(cl["res"]),
                       relu=cl["kw"]["relu"])
        where = (cl["L"],) + cl["shape"]
        assert np.abs(got - ref).max() < 2e-3 * max(1.0, np.abs(ref).max()), (where, np.abs(got - ref).max())
        # The two orders sum the same products in the same offset order, but group them differently into tensor-core
        # instructions: one fp16 ulp of the output, plus fp32 reordering noise (2^-16 = 128 fp32 ulps) of the sum of the
        # products' magnitudes -- which decides where an output is small next to its products.  A dropped or doubled
        # product is far outside this bound.
        mag = ref_conv(np.abs(xq), nbr, np.abs(wq), x2=None if x2q is None else np.abs(x2q),
                       w2=None if w2q is None else np.abs(w2q))
        tol = 2.0 ** -10 * np.maximum(np.abs(got), np.abs(phys)) + 2.0 ** -24 + 2.0 ** -16 * mag
        err = np.abs(got - phys)
        i = np.unravel_index(np.argmax(err - tol), err.shape)
        assert (err <= tol).all(), (where, int((err > tol).sum()), got[i], phys[i], mag[i], ref[i])
        assert np.array_equal(got, via_perm), (where, np.abs(got - via_perm).max())


# ---------------------------------------------------------------- sorted 4-D forward ----
def state_dict3(seed=0):
    sd = O.make_state_dict(seed=seed, randomize_bn=True)
    rng = np.random.default_rng(seed + 77)
    sd["final.kernel"] = (rng.standard_normal((8, 3)) * np.sqrt(2.0 / 3)).astype(np.float32)
    sd["final.bias"] = rng.uniform(-0.3, 0.3, (1, 3)).astype(np.float32)
    return sd


@pytest.mark.parametrize("n_scans", [4, 16])
def test_sorted_4d_forward_matches_oracle(n_scans, sort_always):
    """MOS4DNet on windows of 4 and 16 scans in shape-sorted order: the bars of test_mos4dnet_matches_oracle, and the
    sorted and unsorted fp16 forwards agree to the same bar."""
    from sps_b200.models import MOS4DNet
    pts = window(n_scans)
    sd = state_dict3()
    ref = O.mos4d_forward(pts, 0.1, sd)
    scale = max(1.0, np.abs(ref).max())
    model = MOS4DNet(0.1)
    model.MinkUNet.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
    model = model.cuda().eval()
    d = torch.as_tensor(pts).cuda()
    out = {}
    for backend, tol in ((1, 2e-4), (0, 2e-2)):
        model.set_conv_backend(backend)
        got = model(d).cpu().numpy()
        model.check()
        assert all(model._engine.level(L).perm for L in range(5))
        assert np.abs(got - ref).max() < tol * scale, (backend, np.abs(got - ref).max(), scale)
        assert np.mean((got > 0) == (ref > 0)) >= 0.995
        out[backend] = got
    model._engine.set_pattern_sort(0)
    unsorted = model(d).cpu().numpy()
    model.check()
    assert not model._engine.level(0).perm
    assert np.abs(out[0] - unsorted).max() < 2e-2 * scale, np.abs(out[0] - unsorted).max()
    assert np.mean((out[0] > 0) == (unsorted > 0)) >= 0.995
