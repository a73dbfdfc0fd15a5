"""Probe networks for the level-0 paths of the fused forward, their float64 references and edge inputs (numpy only).

A probe state dict gives every layer zero kernels and a batch norm that folds to scale exactly 1 and shift 0, so every
layer outputs zeros except the path under test.  Block8's downsample reads one half of the level-0 concat buffer out
with the identity, ``final`` is the 8x8 identity, and the raw logit of column c (``engine.Net(sd, output_channel=c,
apply_sigmoid=False)``) is channel c of the probed tensor at the point's voxel:

* readout ``"skip0"`` (rows 8..15 of the concat buffer): conv0p1s1 + bn0 + ReLU, ``taps["out_p1"]`` of the oracle;
* readout ``"up"`` (rows 0..7): convtr7p2s2 + bntr7 + ReLU, ``taps["convtr7p2s2"]``.

Probe A (``probe_a``) puts ``2^(k - 8c - 64p)`` on the 8 offsets of channel c in pass p, so that the output is the
presence bit set of the 125 neighbours times the voxel feature, exact in every storage format.  Probe A'
(``probe_a_numeric``) uses random weights bounded away from zero.  Probe B (``probe_b``) runs conv1p1s2 -> block1
(identity) -> block7's downsample (identity onto channels 0..7) -> convtr7p2s2, so that the output at a level-0 voxel is
the transposed convolution of the stride-2 convolution of its parent's children.

The references look neighbours up in sorted 64-bit keys of the product's own packing, for any subset of rows, so that
they also serve inputs too large for the oracle's dense maps.
"""
from __future__ import annotations

import numpy as np

from oracle import sps_oracle as O

XLIM, ZLIM = 131072, 32768                  # key range: x, y in [-XLIM, XLIM), z in [-ZLIM, ZLIM), t < 16, b < 255
PROBE_VAR = np.float32(1 - 1e-5)            # running_var whose fp32 fold gives scale 1.0f
CENTRE = 62                                 # kernel offset (0, 0, 0) of the 5x5x5x1 conv0
OFF5 = O.kernel_offsets([5, 5, 5, 1], [1, 1, 1, 1]).astype(np.int64)
CHILD = np.array([[k & 1, (k >> 1) & 1, (k >> 2) & 1] for k in range(8)], np.int64)   # child class k -> (ox, oy, oz)
FEAT_BITS = 14                              # significant bits of the probe features (see voxel_features)


# ---------------------------------------------------------------- probe state dicts ----
def set_probe_bn(sd, prefix, C, shift=None):
    sd[prefix + ".bn.weight"] = np.ones(C, np.float32)
    sd[prefix + ".bn.bias"] = np.zeros(C, np.float32) if shift is None else np.asarray(shift, np.float32)
    sd[prefix + ".bn.running_mean"] = np.zeros(C, np.float32)
    sd[prefix + ".bn.running_var"] = np.full(C, PROBE_VAR, np.float32)


def bn_fold_f32(sd, prefix):
    """``bn_fold`` of net.cu: ``inv = 1.0f / sqrtf(var + 1e-5f)`` in fp32, then scale and shift in double."""
    g, b, m, v = (np.asarray(sd[prefix + ".bn." + s], np.float32) for s in ("weight", "bias", "running_mean", "running_var"))
    inv = np.float32(1) / np.sqrt(v + np.float32(1e-5))
    scale = g.astype(np.float64) * inv.astype(np.float64)
    return scale, b.astype(np.float64) - m.astype(np.float64) * scale


def zero_net(readout):
    """Every kernel zero, every BN the probe BN, ``final`` the 8x8 identity; block8's downsample reads the conv0 half
    (``"skip0"``) or the convtr7p2s2 half (``"up"``) of the level-0 concat buffer."""
    sd = {}
    for name, kind, shape in O.layer_shapes():
        if kind == "bn":
            set_probe_bn(sd, name, shape[0])
        elif kind == "bias":
            sd[name] = np.zeros((1, 8), np.float32)
        elif name == "final.kernel":
            sd[name] = np.eye(8, dtype=np.float32)
        else:
            sd[name] = np.zeros(shape, np.float32)
    r0 = {"up": 0, "skip0": 8}[readout]
    sd["block8.0.downsample.0.kernel"][r0:r0 + 8] = np.eye(8, dtype=np.float32)
    return sd


def for_oracle(sd):
    """The state dict as the float64 oracle should see it: the probe variance as the double 1 - 1e-5, for which the
    oracle's float64 batch norm is also exactly the identity (the float32 value is not, in float64)."""
    out = dict(sd)
    for k, v in sd.items():
        if k.endswith("running_var"):
            out[k] = np.where(np.asarray(v) == PROBE_VAR, 1 - 1e-5, np.asarray(v, np.float64))
    return out


def probe_a(p):
    """Pass p (0 or 1) of the presence signature: offset k = 64p + 8c + j -> weight 2^j on channel c."""
    sd = zero_net("skip0")
    w = sd["conv0p1s1.kernel"]
    for k in range(64 * p, min(125, 64 * p + 64)):
        w[k, 0, (k - 64 * p) // 8] = 2.0 ** ((k - 64 * p) % 8)
    return sd


def bounded(rng, shape):
    """Random weights with |w| in [0.5, 1.5] and random signs."""
    return (rng.uniform(0.5, 1.5, shape) * rng.choice([-1.0, 1.0], shape)).astype(np.float32)


def probe_a_numeric(seed=0):
    rng = np.random.default_rng(seed)
    sd = zero_net("skip0")
    sd["conv0p1s1.kernel"] = bounded(rng, (125, 1, 8))
    set_probe_bn(sd, "bn0", 8, rng.uniform(0.05, 0.5, 8))
    return sd


def probe_b(seed=0):
    """conv0: the centre offset only, 8-bit weights, so that skip0 = w * feature is exact in fp32; conv1p1s2 and
    convtr7p2s2 random and bounded away from zero; block7's downsample maps skip1 = E1 onto its channels 0..7."""
    rng = np.random.default_rng(seed)
    sd = zero_net("up")
    sd["conv0p1s1.kernel"][CENTRE, 0] = rng.integers(64, 193, 8) / 128.0
    sd["conv1p1s2.kernel"] = bounded(rng, (8, 8, 8))
    set_probe_bn(sd, "bn1", 8, rng.uniform(0.0, 0.25, 8))
    sd["block7.0.downsample.0.kernel"][16:24, 0:8] = np.eye(8, dtype=np.float32)
    sd["convtr7p2s2.kernel"] = bounded(rng, (8, 16, 8))
    set_probe_bn(sd, "bntr7", 8, rng.uniform(0.0, 0.25, 8))
    return sd


def bn_shift(sd, prefix):
    return np.asarray(sd[prefix + ".bn.bias"], np.float64)


# ---------------------------------------------------------------- storage roundings of the product ----
def tf32_rna(x):
    """``cvt.rna.tf32.f32`` (nearest, ties away from zero) of the fp32 value of x."""
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return (((u + 0x1000) & 0xFFFFE000).astype(np.uint32)).view(np.float32).astype(np.float64)


def tf32_rne(x):
    """The TF32 weight rounding of ``sps_conv_pack_kmajor`` (nearest even)."""
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0xFFF + ((u >> 13) & 1)) & 0xFFFFE000
    return u.astype(np.uint32).view(np.float32).astype(np.float64)


def f16_hilo(x):
    """``kStoreF16x2``: hi = fp16(v), lo = fp16(v - hi), read back as hi + lo."""
    v = np.asarray(x, np.float32)
    hi = v.astype(np.float16)
    lo = (v - hi.astype(np.float32)).astype(np.float16)
    return hi.astype(np.float64) + lo.astype(np.float64)


def ulp10(x):
    """Spacing of a 10-bit-mantissa format (fp16, TF32) at x; fp16 subnormals: 2^-24."""
    _, e = np.frexp(np.abs(np.asarray(x, np.float64)))
    return np.where(np.asarray(x) == 0, 0.0, np.ldexp(1.0, np.maximum(e - 11, -24)))


# ---------------------------------------------------------------- neighbour lookup ----
def in_range(c):
    c = np.asarray(c, np.int64)
    return ((c[:, 0] >= 0) & (c[:, 0] < 255) & (c[:, 1] >= -XLIM) & (c[:, 1] < XLIM) & (c[:, 2] >= -XLIM) &
            (c[:, 2] < XLIM) & (c[:, 3] >= -ZLIM) & (c[:, 3] < ZLIM) & (c[:, 4] >= 0) & (c[:, 4] < 16))


def pack(c):
    """The product's 64-bit key (b:8 | x:18 | y:18 | z:16 | t:4, biased) of in-range rows (b, x, y, z, t)."""
    c = np.asarray(c, np.int64)
    u = lambda a: a.astype(np.uint64)
    return ((u(c[:, 0]) << np.uint64(56)) | (u(c[:, 1] + XLIM) << np.uint64(38)) | (u(c[:, 2] + XLIM) << np.uint64(20)) |
            (u(c[:, 3] + ZLIM) << np.uint64(4)) | u(c[:, 4]))


class Lookup:
    """Row of a coordinate in ``coords`` (-1: absent or outside the key range) by binary search over sorted keys."""

    def __init__(self, coords):
        keys = pack(coords)
        self.order = np.argsort(keys, kind="stable")
        self.keys = keys[self.order]

    def __call__(self, q):
        q = np.asarray(q, np.int64)
        out = np.full(len(q), -1, np.int64)
        ok = np.flatnonzero(in_range(q))
        if len(ok) and len(self.keys):
            k = pack(q[ok])
            pos = np.minimum(np.searchsorted(self.keys, k), len(self.keys) - 1)
            hit = self.keys[pos] == k
            out[ok[hit]] = self.order[pos[hit]]
        return out


def nbr5_rows(lookup, c0, rows):
    """``nbr5[:, rows].T``: [len(rows), 125] rows of the 5x5x5x1 neighbours (-1 absent)."""
    c = np.asarray(c0, np.int64)[rows]
    out = np.empty((len(c), 125), np.int64)
    for k in range(125):
        q = c.copy()
        q[:, 1:5] += OFF5[k]
        out[:, k] = lookup(q)
    return out


# ---------------------------------------------------------------- references ----
def signature_values(present, feat, p):
    """Exact conv0 output of probe A pass p when every voxel carries the feature ``feat``: feat x sum of 2^j over the
    present offsets 64p + 8c + j."""
    code = np.zeros((len(present), 8), np.float64)
    for k in range(64 * p, min(125, 64 * p + 64)):
        code[:, (k - 64 * p) // 8] += present[:, k] * 2.0 ** ((k - 64 * p) % 8)
    return code * float(feat)


def decode_signature(vals0, vals1, feat):
    """Presence bits [R, 125] from the probe A outputs of both passes under the common feature ``feat`` (asserts that
    they are exact integer codes)."""
    bits = np.zeros((len(vals0), 125), bool)
    for p, vals in enumerate((vals0, vals1)):
        code = np.asarray(vals, np.float64) / float(feat)
        assert np.array_equal(code, np.round(code)) and code.min(initial=0) >= 0 and code.max(initial=0) <= 255
        code = code.astype(np.int64)
        for k in range(64 * p, min(125, 64 * p + 64)):
            bits[:, k] = (code[:, (k - 64 * p) // 8] >> ((k - 64 * p) % 8)) & 1
    return bits


def conv0_rows(nbr, feat, sd, chunk=4096):
    """conv0p1s1 + bn0 + ReLU at float64 on the rows of ``nbr`` ([R, 125]); returns (out, S) with S = sum of the
    magnitudes of the products and the BN shift, per output."""
    w = np.asarray(sd["conv0p1s1.kernel"], np.float64)[:, 0, :]
    shift = bn_shift(sd, "bn0")
    feat = np.asarray(feat, np.float64)
    out = np.empty((len(nbr), 8))
    S = np.empty((len(nbr), 8))
    for r in range(0, len(nbr), chunk):
        nb = nbr[r:r + chunk]
        x = np.where(nb >= 0, feat[np.maximum(nb, 0)], 0.0)
        out[r:r + chunk] = np.maximum(x @ w + shift, 0.0)
        S[r:r + chunk] = np.abs(x) @ np.abs(w) + np.abs(shift)
    return out, S


SKIP0_STORE = {1: lambda v: np.asarray(v, np.float64), 2: tf32_rna, 0: f16_hilo}


def probe_b_rows(lookup, c0, feat, sd, rows, backend):
    """Probe B at the level-0 rows ``rows``: (out, S, flip).  ``feat`` is the per-voxel feature.

    skip0 = relu(w_centre * feature) is exact in fp32 and is stored as the backend stores it (fp32, TF32, hi|lo).  E1 of
    the parent (conv1p1s2 over its children + bn1 + ReLU) is computed in float64 and rounded as the backend stores it
    (fp32; TF32; plain fp16 at level 1); the TF32 backend's transposed convolution uses TF32-rounded weights.  S sums the
    magnitudes of every product behind an output, E1's included; ``flip`` is one ulp of every stored E1 times |W_u|,
    what a last-bit fp32 difference can move an output by when it flips the rounding of E1."""
    c = np.asarray(c0, np.int64)[rows]
    feat = np.asarray(feat, np.float64)
    w0 = np.asarray(sd["conv0p1s1.kernel"], np.float64)[CENTRE, 0]
    w1 = np.asarray(sd["conv1p1s2.kernel"], np.float64)
    b1, bu = bn_shift(sd, "bn1"), bn_shift(sd, "bntr7")
    par = c.copy()
    par[:, 1:4] = np.floor_divide(c[:, 1:4], 2) * 2
    e1 = np.tile(b1, (len(c), 1))
    s1 = np.tile(np.abs(b1), (len(c), 1))
    for j in range(8):
        q = par.copy()
        q[:, 1:4] += CHILD[j]
        idx = lookup(q)
        x = np.where(idx[:, None] >= 0, np.maximum(np.outer(feat[np.maximum(idx, 0)], w0) + bn_shift(sd, "bn0"), 0.0), 0.0)
        x = SKIP0_STORE[backend](x)
        e1 += x @ w1[j]
        s1 += np.abs(x) @ np.abs(w1[j])
    e1 = np.maximum(e1, 0.0)
    if backend == 2:
        e1 = tf32_rna(e1)
    elif backend == 0:
        e1 = np.asarray(e1, np.float32).astype(np.float16).astype(np.float64)
    wu = np.asarray(sd["convtr7p2s2.kernel"], np.float64)[:, :8, :]          # rows 8..15 read block7's zero channels
    if backend == 2:
        wu = tf32_rne(wu)
    k = (c[:, 1] & 1) + 2 * (c[:, 2] & 1) + 4 * (c[:, 3] & 1)
    W = wu[k]                                                              # [R, 8 in, 8 out]
    out = np.maximum(np.einsum("ri,rio->ro", e1, W) + bu, 0.0)
    S = np.einsum("ri,rio->ro", s1, np.abs(W)) + np.abs(bu)
    flip = np.einsum("ri,rio->ro", ulp10(e1), np.abs(W)) if backend != 1 else np.zeros_like(out)
    return out, S, flip


BOUND_A_NUMERIC = {1: 2.0 ** -22, 2: 2.0 ** -10, 0: 2.0 ** -19}
BOUND_B = {1: 2.0 ** -21, 2: 2.0 ** -10, 0: 2.0 ** -19}


# ---------------------------------------------------------------- inputs ----
def to_points(coords):
    """Voxel size 1.0: the point at the centre of each voxel (exact in fp32 over the whole key range)."""
    p = np.asarray(coords, np.float64).astype(np.float32)
    p[:, 1:4] += np.float32(0.5)
    return p


def voxel_features(n, rng):
    """Per-voxel features in [0.5, 1) with FEAT_BITS significant bits: the mean of up to 2^(24 - FEAT_BITS) equal
    point features is exact in fp32 whatever the summation order, and w * feature is exact for 8-bit w."""
    return rng.integers(1 << (FEAT_BITS - 1), 1 << FEAT_BITS, n) / float(1 << FEAT_BITS)


def cube(lo, n, occupancy, rng, b=0, t=0):
    g = np.arange(n)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) + np.asarray(lo)
    if occupancy < 1:
        xyz = xyz[rng.random(len(xyz)) < occupancy]
    return np.hstack([np.full((len(xyz), 1), b), xyz, np.full((len(xyz), 1), t)]).astype(np.int64)


def pairs(origin=(0, 0, 0)):
    """Isolated voxels, and pairs at distance 2, 3 and 4 (inside and just outside the 5-window) along each axis and
    along face and body diagonals, 16 apart from each other."""
    dirs = [(1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, 1, 1), (1, -1, 0), (-1, 1, 1)]
    vox = [np.array([0, 0, 0]), np.array([16, 0, 0])]
    i = 2
    for d in dirs:
        for s in (2, 3, 4):
            a = np.array([16 * i, 0, 0])
            vox += [a, a + s * np.array(d)]
            i += 1
    xyz = np.array(vox, np.int64) + np.asarray(origin)
    return np.hstack([np.zeros((len(xyz), 1), np.int64), xyz, np.zeros((len(xyz), 1), np.int64)])


LATTICE_XY = (-131072, -131071, -131070, 131069, 131070, 131071)
LATTICE_Z = (-32768, -32767, -32766, 32765, 32766, 32767)


def lattice(axis, rng):
    """One axis at a time: at each value of the axis' end set a voxel with a 3x3x3 cube around it (clipped to the key
    range, 40 % occupied); the other axes stay small.  Returns (coords, out-of-range points)."""
    vals = LATTICE_Z if axis == 3 else LATTICE_XY
    lim = ZLIM if axis == 3 else XLIM
    rows = []
    other = [a for a in (1, 2, 3) if a != axis]
    for i, v in enumerate(vals):
        c = cube((0, 0, 0), 3, 0.4, rng)
        c[:, axis] += v - 1
        c[:, other[0]] += 12 * i
        c = c[(c[:, axis] >= -lim) & (c[:, axis] < lim)]
        centre = np.zeros(5, np.int64)
        centre[axis], centre[other[0]], centre[other[1]] = v, 12 * i + 1, 1
        rows += [c, centre[None]]
    coords = np.unique(np.vstack(rows), axis=0)
    bad = np.zeros((2, 5), np.int64)
    bad[0, axis] = lim                          # one past the top of the axis
    bad[1, axis] = -lim - 1                     # one below the bottom
    return coords, bad


def planes(rng):
    """The same xyz set (a sparse cube and the pairs) in time planes 0, 1, 7, 15 and batches 0, 1, 254, plus points
    in batch 255 and time plane 16 (outside the key range)."""
    xyz = np.vstack([cube((-6, -6, -6), 12, 0.35, rng), pairs((40, -8, 3))])[:, 1:4]
    rows = [np.hstack([np.full((len(xyz), 1), b), xyz, np.full((len(xyz), 1), t)])
            for b in (0, 1, 254) for t in (0, 1, 7, 15)]
    bad = np.array([[255, 0, 0, 0, 0], [0, 0, 0, 0, 16]], np.int64)
    return np.vstack(rows).astype(np.int64), bad


def classes(counts):
    """Level-0 voxels with counts[k] rows in child class k (ox + 2 oy + 4 oz); voxel i of every class lies in parent
    cell i, so parents gather children of several classes."""
    rows = []
    for k, n in enumerate(counts):
        i = np.arange(n)
        par = 2 * np.stack([i % 16, (i // 16) % 16, i // 256], -1)
        xyz = par + CHILD[k] - np.array([10, 10, 10])        # negative coordinates too
        rows.append(np.hstack([np.zeros((n, 1), np.int64), xyz, np.zeros((n, 1), np.int64)]))
    return np.vstack(rows)


def child_class(coords):
    c = np.asarray(coords, np.int64)
    return (c[:, 1] & 1) + 2 * (c[:, 2] & 1) + 4 * (c[:, 3] & 1)


CLASS_CASES = {
    "cls-even": (300, 0, 0, 0, 0, 0, 0, 0),          # every coordinate even: one class
    "cls-one-row": (150, 1, 60, 0, 33, 0, 0, 7),     # a class of exactly one row
    "cls-127-128-129": (127, 128, 129, 0, 40, 0, 0, 0),
    "cls-tile-edges": (127, 129, 129, 50, 0, 0, 0, 3),   # classes end 1 row before, at and 1 row after a 128-row tile edge
    "cls-all-eight": (3, 15, 1, 7, 9, 12, 5, 2),     # one tile meets all eight classes
}
EDGE_CASES = ("cubes", "pairs", "lattice-x", "lattice-y", "lattice-z", "planes") + tuple(CLASS_CASES)
LARGE_CASES = ("dense-430k", "dense-1.3M")


def random_box(lo, n, occupancy, rng):
    idx = np.flatnonzero(rng.random(n ** 3) < occupancy)
    xyz = np.stack([idx // (n * n), (idx // n) % n, idx % n], -1) + np.asarray(lo)
    return np.hstack([np.zeros((len(xyz), 1), np.int64), xyz, np.zeros((len(xyz), 1), np.int64)])


def edge_input(name, seed=0):
    """(voxel coords [V, 5] int64 in row order, out-of-range coords [M, 5]) of a named input; every voxel one point."""
    rng = np.random.default_rng(seed)
    bad = np.zeros((0, 5), np.int64)
    if name == "cubes":
        coords = np.vstack([cube((-6, -6, -6), 12, 0.35, rng), cube((-30, 11, -21), 9, 1.0, rng)])
    elif name == "pairs":
        coords = pairs((-100, 7, -3))
    elif name.startswith("lattice-"):
        coords, bad = lattice({"x": 1, "y": 2, "z": 3}[name[-1]], rng)
    elif name == "planes":
        coords, bad = planes(rng)
    elif name in CLASS_CASES:
        coords = classes(CLASS_CASES[name])
    elif name == "dense-430k":
        coords = random_box((-60, -60, -60), 112, 0.31, rng)
    elif name == "dense-1.3M":
        coords = random_box((-80, -80, -80), 160, 0.33, rng)
    else:
        raise KeyError(name)
    return coords[rng.permutation(len(coords))], bad


def sample_rows(V, n=20000, tail=2000, seed=0):
    """All rows of a small input; else n rows that include the last ``tail``."""
    if V <= n:
        return np.arange(V)
    head = np.random.default_rng(seed).choice(V - tail, n - tail, replace=False)
    return np.sort(np.concatenate([head, np.arange(V - tail, V)]))
