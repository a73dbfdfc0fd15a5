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
