"""CPU checks of the probe networks in tests/probe_nets.py: the probe batch norm folds to the identity under the
product's fp32 arithmetic, each probe routes exactly the tensor under test to the network's output (through the
oracle's float64 forward), the references agree with the oracle, and the edge inputs are what they claim to be."""
import numpy as np
import pytest

import probe_nets as P
from oracle import sps_oracle as O

SMALL = tuple(n for n in P.EDGE_CASES)


def oracle_run(coords, sd, feat):
    c0, _ = O.voxelize(P.to_points(coords), 1.0)
    lv = O.Levels(c0)
    taps = {}
    final = O.unet_forward(lv, np.asarray(feat, np.float64)[:, None], P.for_oracle(sd), np.float64, taps)
    return lv, taps, final


@pytest.fixture(scope="module", params=SMALL)
def edge(request):
    coords, bad = P.edge_input(request.param)
    feat = P.voxel_features(len(coords), np.random.default_rng(1))
    return request.param, coords, bad, feat


def test_probe_bn_folds_to_scale_one_and_zero_shift():
    for sd in (P.probe_a(0), P.probe_a(1), P.probe_a_numeric(), P.probe_b()):
        for name, kind, shape in O.layer_shapes():
            if kind != "bn":
                continue
            scale, shift = P.bn_fold_f32(sd, name)
            assert np.all(scale == 1.0), name
            assert np.array_equal(shift, np.asarray(sd[name + ".bn.bias"], np.float64)), name
    scale, shift = P.bn_fold_f32(P.probe_b(), "bn1")
    assert np.all(shift > 0) and np.all(np.asarray(shift, np.float32) == shift)


def test_rounding_helpers():
    one = np.float32(1.0)
    ulp = 2.0 ** -10
    assert P.tf32_rna(one + np.float32(ulp / 2)) == 1 + ulp                 # tie: away from zero
    assert P.tf32_rne(one + np.float32(ulp / 2)) == 1.0                     # tie: to even
    assert P.tf32_rne(one + np.float32(1.5 * ulp)) == 1 + 2 * ulp
    assert P.tf32_rna(-(one + np.float32(ulp / 2))) == -(1 + ulp)
    x = np.float32(1 / 3)
    assert abs(P.f16_hilo(x) - float(x)) <= 2.0 ** -22 * float(x)
    assert P.ulp10(1.0) == 2.0 ** -10 and P.ulp10(0.75) == 2.0 ** -11 and P.ulp10(0.0) == 0.0
    assert P.ulp10(2.0 ** -20) == 2.0 ** -24


def test_edge_inputs_quantise_inside_the_key_range(edge):
    name, coords, bad, _ = edge
    assert len(coords) and P.in_range(coords).all()
    assert not P.in_range(bad).any()
    c0, inv = O.voxelize(P.to_points(coords), 1.0)
    assert np.array_equal(c0, coords) and np.array_equal(inv, np.arange(len(coords)))   # one point per voxel, row order
    if len(bad):
        q = O.quantize(P.to_points(bad), 1.0)
        assert np.array_equal(q, bad)
    if name in P.CLASS_CASES:
        assert tuple(np.bincount(P.child_class(coords), minlength=8)) == P.CLASS_CASES[name]


def test_class_cases_put_class_edges_where_they_claim():
    ends = np.cumsum(P.CLASS_CASES["cls-tile-edges"])
    assert {127, 256, 385} <= set(ends.tolist())
    counts = np.array(P.CLASS_CASES["cls-all-eight"])
    assert counts.min() >= 1 and counts.max() < 16 and counts.sum() <= 128


def test_signature_decoding_reproduces_nbr5(edge):
    """The oracle's own conv0 output under probe A decodes to the presence of the 125 neighbours, and the
    searchsorted lookup finds the same neighbours as the oracle's kernel map."""
    _, coords, _, _ = edge
    for feat in (0.5, 1.0):
        vals = []
        for p in (0, 1):
            lv, taps, final = oracle_run(coords, P.probe_a(p), np.full(len(coords), feat))
            assert np.array_equal(final, taps["out_p1"])                    # routing: bit for bit
            vals.append(taps["out_p1"])
        present = lv.nbr5.T >= 0
        assert np.array_equal(P.decode_signature(vals[0], vals[1], feat), present)
        for p in (0, 1):
            assert np.array_equal(P.signature_values(present, feat, p), vals[p])
    nb = P.nbr5_rows(P.Lookup(coords), coords, np.arange(len(coords)))
    assert np.array_equal(nb, lv.nbr5.T)


def test_probe_a_numeric_routes_and_matches_conv0_reference(edge):
    _, coords, _, feat = edge
    sd = P.probe_a_numeric()
    lv, taps, final = oracle_run(coords, sd, feat)
    assert np.array_equal(final, taps["out_p1"])
    out, S = P.conv0_rows(lv.nbr5.T, feat, sd)
    assert np.all(np.abs(out - taps["out_p1"]) <= 1e-13 * S)
    assert (out > 0).mean() > 0.3                                           # the probed values are not mostly clamped


def test_probe_b_routes_and_matches_stride_transpose_reference(edge):
    name, coords, _, feat = edge
    sd = P.probe_b()
    lv, taps, final = oracle_run(coords, sd, feat)
    assert np.all(np.abs(final - taps["convtr7p2s2"]) <= 1e-12 * np.maximum(np.abs(taps["convtr7p2s2"]), 1))
    # the chain by hand with the oracle's own layer functions
    x0 = np.maximum(np.asarray(feat, np.float64)[:, None] * np.asarray(sd["conv0p1s1.kernel"], np.float64)[P.CENTRE, 0], 0)
    e1 = np.maximum(O.conv_stride2(x0, lv.parent[0], lv.koff[0], sd["conv1p1s2.kernel"], len(lv.coords[1]), np.float64)
                    + P.bn_shift(sd, "bn1"), 0)
    b7 = np.hstack([e1, np.zeros_like(e1)])
    up = np.maximum(O.conv_transpose2(b7, lv.parent[0], lv.koff[0], sd["convtr7p2s2.kernel"], np.float64)
                    + P.bn_shift(sd, "bntr7"), 0)
    assert np.allclose(up, taps["convtr7p2s2"], rtol=1e-12, atol=1e-12)
    out, S, flip = P.probe_b_rows(P.Lookup(coords), coords, feat, sd, np.arange(len(coords)), 1)
    assert np.all(np.abs(out - up) <= 1e-12 * S) and not flip.any()
    if name not in ("pairs",):
        assert (out > 0).mean() > 0.2
    # the stored-format references differ from float64 by no more than their bounds allow
    for backend in (2, 0):
        o, S2, fl = P.probe_b_rows(P.Lookup(coords), coords, feat, sd, np.arange(len(coords)), backend)
        assert np.all(np.abs(o - up) <= 2.0 ** -9 * S2 + fl)


def test_large_inputs_have_the_claimed_sizes():
    coords, _ = P.edge_input("dense-430k")
    assert len(coords) >= 400_000
    coords, _ = P.edge_input("dense-1.3M")
    assert len(coords) > 148 * 32 * 256
    rows = P.sample_rows(len(coords))
    assert len(rows) == 20000 and np.array_equal(rows[-2000:], np.arange(len(coords) - 2000, len(coords)))
    # the sample lookup agrees with the oracle's kernel map on a window of the input
    sub = coords[:3000]
    lv = O.kernel_map(sub, sub, P.OFF5.astype(np.int32))
    assert np.array_equal(P.nbr5_rows(P.Lookup(sub), sub, np.arange(3000)), lv.T)


# ---------------------------------------------------------------- deep probes (levels 1..4) ----
DEEP_SMALL = P.EDGE_CASES + P.DEEP_CASES
ROUTE_CASES = ("cubes", "planes", "full81", "cls-l2", "lvl-129")


def deep_case(name):
    coords, _ = P.edge_input(name)
    feat = P.deep_features(len(coords), np.random.default_rng(5))
    return coords, feat, P.DeepLevels(coords, feat)


def tap_at_level0(lv, taps, tap, L):
    """The oracle's tap at level L, broadcast to the level-0 rows through the parent tables."""
    x = taps[tap]
    idx = np.arange(len(lv.coords[0]))
    for l in range(L):
        idx = lv.parent[l][idx]
    return x[idx]


@pytest.mark.parametrize("name", ROUTE_CASES)
def test_deep_probes_route_and_match_oracle(name):
    """Each probe routes the tensor under test to the head bit for bit through the oracle's float64 forward (per
    readout column, against the oracle's tap), and the float64 reference agrees with the oracle to 1e-12 S."""
    coords, feat, dl = deep_case(name)
    c0, _ = O.voxelize(P.to_points(coords), 1.0)
    lv = O.Levels(c0)
    rows = np.arange(len(coords))
    for layer in P.DEEP_LAYERS:
        L, _, tap, C = P.probe_info(layer)
        ref, _, _ = P.deep_reference(dl, layer, P.deep_probe(layer), None, rows)
        S = P.deep_reference(dl, layer, P.deep_probe(layer), 1, rows)[1] / P.BOUND_DEEP
        for g in range(P.deep_groups(layer)):
            taps = {}
            final = O.unet_forward(lv, feat[:, None], P.for_oracle(P.deep_probe(layer, g)), np.float64, taps)
            if layer == "block8.conv2":
                want = final
            else:
                want = tap_at_level0(lv, taps, tap, L)[:, 8 * g:8 * g + 8]
                assert np.array_equal(final, want), f"{layer} group {g}: the readout is not exact"
            r = ref[:, 8 * g:8 * g + 8]
            assert np.all(np.abs(r - want) <= 1e-12 * S[:, 8 * g:8 * g + 8]), f"{layer} group {g}"
        assert (ref > 0).mean() > 0.3 or layer == "block8.conv2", layer        # the outputs are not mostly clamped


@pytest.mark.parametrize("name", DEEP_SMALL)
def test_deep_lift_is_exact_and_distinct(name):
    """Every lifted value upstream of a layer under test is 0 or a multiple of 2^-8 below 8 (at most 11 significant
    bits: exact in fp16, TF32 and fp32) and at least 2^-14; both halves of every concat row are non-zero; no two
    channels of a lifted tensor are equal on every voxel; conv0's channels 0..3 carry low halves."""
    _, _, dl = deep_case(name)
    tensors = [("skip0[4:]", dl.skip[0][:, 4:])] + [(f"E{L}", dl.E[L]) for L in range(1, 5)] + \
        [(f"skip{L}", dl.skip[L]) for L in range(1, 5)] + [(f"B{l}", dl.B[l]) for l in dl.B] + \
        [(f"U{l}", dl.U[l]) for l in dl.U]
    for what, x in tensors:
        assert np.array_equal(x * 256, np.round(x * 256)) and x.max() < 8 and x.min() >= 0.25, what
        assert np.array_equal(np.asarray(x, np.float16).astype(np.float64), x), what
        assert np.array_equal(P.tf32_rna(x), x) and np.array_equal(P.tf32_rne(x), x), what
        if name in ("cubes", "planes", "mos4d-4scan"):     # sparse inputs lack whole child classes: constant channels
            same = [(i, j) for i in range(x.shape[1]) for j in range(i) if np.array_equal(x[:, i], x[:, j])]
            assert not same, (what, same)
    for l in range(4):
        cat = dl.cat(l, 1)
        up = DEC_UP = P.DEC[l][4]
        assert (cat[:, :up] != 0).all() and (cat[:, up:] != 0).all()
    hi = dl.skip[0][:, :4]
    assert np.array_equal(P.f16_hilo(hi), hi) and (P.f16_hilo(hi) != np.asarray(hi, np.float16)).mean() > 0.5


@pytest.mark.parametrize("name", DEEP_SMALL)
def test_deep_bound_is_below_the_smallest_product(name):
    """fp32 backend, and the fp32 logits of block8.conv2 + final on every backend: BOUND_DEEP * S is smaller than the
    smallest non-zero |w x| behind every output that survives the ReLU, so a dropped product, a lost weight half or a
    missing shift cannot hide under the bound; the stored-format references stay within their bounds of float64."""
    _, _, dl = deep_case(name)
    rows = P.sample_rows(len(dl.c[0]))
    for layer in P.DEEP_LAYERS:
        sd = P.deep_probe(layer)
        ref64, _, _ = P.deep_reference(dl, layer, sd, None, rows)
        for backend in (1, 2, 0):
            ref, lim, margin = P.deep_reference(dl, layer, sd, backend, rows)
            if backend == 1 or layer == "block8.conv2":
                assert (margin > 0).all(), (layer, backend)
            if backend == 1:
                assert np.all(np.abs(ref - ref64) <= lim), layer


# the precision plan as net.cu states it; a change to sps_net_finalize's plan must change this literal and PLAN
PLAN_LITERAL = {
    "conv1p1s2": "K8 8->8 fp16: FOLD_LO IN_SPLIT; tf32: simt",
    "block1.conv1": "K81 8->8 fp16: FOLD_LO; tf32: tc", "block1.conv2": "K81 8->8 fp16: FOLD_LO; tf32: tc",
    "conv2p2s2": "K8 8->8 fp16: FOLD_LO; tf32: simt",
    "block2.conv1": "K81 8->16 fp16: ; tf32: tc", "block2.conv2": "K81 16->16 +1x1 8 fp16: ; tf32: tc",
    "conv3p4s2": "K8 16->16 fp16: ; tf32: tc",
    "block3.conv1": "K81 16->32 fp16: ; tf32: tc", "block3.conv2": "K81 32->32 +1x1 16 fp16: ; tf32: tc",
    "conv4p8s2": "K8 32->32 fp16: ; tf32: tc",
    "block4.conv1": "K81 32->64 fp16: ; tf32: tc", "block4.conv2": "K81 64->64 +1x1 32 fp16: ; tf32: tc",
    "convtr4p16s2": "K8 64->64 fp16: ; tf32: tc",
    "block5.conv1": "K81 96->64 fp16:  split 64; tf32: tc", "block5.conv2": "K81 64->64 +1x1 96 fp16: ; tf32: tc",
    "convtr5p8s2": "K8 64->32 fp16: ; tf32: tc",
    "block6.conv1": "K81 48->32 fp16: ; tf32: tc", "block6.conv2": "K81 32->32 +1x1 48 fp16: ; tf32: tc",
    "convtr6p4s2": "K8 32->16 fp16: ; tf32: tc",
    "block7.conv1": "K81 24->16 fp16: ; tf32: tc", "block7.conv2": "K81 16->16 +1x1 24 fp16: ; tf32: tc",
    "convtr7p2s2": "K8 16->8 fp16: FOLD_LO OUT_SPLIT; tf32: tc",
    "block8.conv1": "K81 16->8 fp16: FOLD_LO IN_SPLIT; tf32: tc",
    "block8.conv2": "K81 8->8 +1x1 16 fp16: FOLD_LO IN2_SPLIT; tf32: tc",
}


def plan_from_rules():
    """sps_net_finalize's rules applied to the layer list: cout == 8 -> FOLD_LO; conv1p1s2 and block8.conv1 read the
    hi|lo level-0 rows, block8.conv2's 1x1 term does, convtr7p2s2 writes them; two K segments where a block reads more
    channels than it writes and writes 64; a K-major TF32 copy (tcgen05 on the TF32 backend) for K == 81 and for
    2x2x2 layers with cin >= 16."""
    out = {}
    enc = [("conv1p1s2", 8, 8), ("conv2p2s2", 8, 16), ("conv3p4s2", 16, 32), ("conv4p8s2", 32, 64)]
    dec = [("convtr4p16s2", 64, 64, 32), ("convtr5p8s2", 64, 32, 16), ("convtr6p4s2", 32, 16, 8), ("convtr7p2s2", 16, 8, 8)]

    def add(name, K, cin, cout, cin2=0, in_split=False, in2_split=False, out_split=False, seg=0):
        flags = " ".join(f for f, on in (("FOLD_LO", cout == 8), ("IN_SPLIT", in_split), ("IN2_SPLIT", in2_split),
                                         ("OUT_SPLIT", out_split)) if on)
        tc = K == 81 or (K == 8 and cin >= 16 and cin % 4 == 0)
        out[name] = (f"K{K} {cin}->{cout}" + (f" +1x1 {cin2}" if cin2 else "") + f" fp16: {flags}" +
                     (f" split {seg}" if seg else "") + f"; tf32: {'tc' if tc else 'simt'}")

    def block(b, cin, cout, tail=False):
        seg = cout if (not tail and cin > cout and cout == 64) else 0
        add(f"block{b}.conv1", 81, cin, cout, in_split=tail, seg=seg)
        add(f"block{b}.conv2", 81, cout, cout, cin if cin != cout else 0, in2_split=tail and cin != cout)

    for i, (name, cin, planes) in enumerate(enc):
        add(name, 8, cin, cin, in_split=i == 0)
        block(i + 1, cin, planes)
    for i, (name, cin, planes, skip) in enumerate(dec):
        add(name, 8, cin, planes, out_split=i == 3)
        block(5 + i, planes + skip, planes, tail=i == 3)
    return out


def test_precision_plan_is_pinned():
    """PLAN (what the references model) = the literal = sps_net_finalize's rules, and net.cu still states them."""
    assert plan_from_rules() == PLAN_LITERAL
    for layer, (K, cin, cout, cin2, flags, seg, tf32) in P.PLAN.items():
        s = f"K{K} {cin}->{cout}" + (f" +1x1 {cin2}" if cin2 else "") + f" fp16: {flags}" + \
            (f" split {seg}" if seg else "") + f"; tf32: {tf32}"
        assert PLAN_LITERAL[layer] == s, layer
    import os
    src = open(os.path.join(os.path.dirname(__file__), "..", "sps_b200", "csrc", "net.cu")).read()
    for line in ("cw.pack_flags = (cout == 8 ? SPS_PACK_FOLD_LO : 0) | (in_split ? SPS_PACK_IN_SPLIT : 0) | "
                 "(in2_split ? SPS_PACK_IN2_SPLIT : 0);",
                 "cw.conv_flags = (cout == 8 ? SPS_CONV_FOLD_LO : 0) | (out_split ? SPS_CONV_OUT_SPLIT : 0);",
                 "if (K == 81 || (K == 8 && cin >= 16 && cin % 4 == 0)) add_kmajor(p, w, K, cin, cout, nullptr, 0);",
                 "const int seg = (!tail && cin > cout && cout == 64) ? cout : 0;",
                 "plan(cw, cout, false, tail && cin != cout, false);",
                 "for (int c = 0; c < cout; ++c) sh[c] += sh2[c];",
                 "inpl, inpl, /*in_split=*/i == 0);",
                 "P[4 + i], false, /*out_split=*/i == 3);",
                 "P[4 + i] + skip[i], P[4 + i], /*tail=*/i == 3);"):
        assert line in src, line


@pytest.mark.parametrize("name", P.DEEP_CASES + ("lattice-x", "lattice-y", "lattice-z"))
def test_deep_edge_inputs_are_what_they_claim(name):
    coords, _ = P.edge_input(name)
    assert P.in_range(coords).all() and len(np.unique(coords, axis=0)) == len(coords)
    dl = P.DeepLevels(coords, np.ones(len(coords)))
    counts = [len(c) for c in dl.c]
    if name.startswith("lvl-"):
        assert counts[1:] == [int(name[4:])] * 4
    elif name == "full81":
        for L in (3, 4):
            nb = dl.nbr3(L, np.arange(counts[L]))
            assert (nb >= 0).all(1).sum() >= 1, L
        assert counts[3] == 648 and counts[4] == 81
    elif name.startswith("cls-l"):
        L = int(name[-1])
        assert tuple(np.bincount(dl.cls[L - 1] if False else P.child_class(dl.c[L] >> L), minlength=8)) == \
            P.CLASS_CASES["cls-tile-edges"]
        assert (dl.c[L][:, 1:4] < 0).any()
    elif name == "mos4d-4scan":
        assert set(np.unique(coords[:, 4]).tolist()) == {0, 1, 2, 3}
        for L in range(1, 5):
            nb = dl.nbr3(L, np.arange(counts[L]))
            t = np.array([o[3] for o in P.OFF3[L]])
            assert (nb[:, t == 1] >= 0).any() and (nb[:, t == -1] >= 0).any(), L
    else:                                       # the lattice cases reach the key-range ends at every level
        axis = {"x": 1, "y": 2, "z": 3}[name[-1]]
        lim = P.ZLIM if axis == 3 else P.XLIM
        for L in range(5):
            assert dl.c[L][:, axis].min() == -lim and dl.c[L][:, axis].max() == lim - 2 ** L, L
