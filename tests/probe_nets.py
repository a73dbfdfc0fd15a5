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


LEVEL_COUNTS = (127, 128, 129, 255, 256, 257)
DEEP_CASES = tuple(f"lvl-{n}" for n in LEVEL_COUNTS) + ("full81", "cls-l1", "cls-l2", "cls-l3", "mos4d-4scan")


def deep_input(name, rng):
    """Edges at the coarse levels.  ``lvl-N``: N level-4 cells, each holding two level-0 voxels of one level-1 cell, so
    that every level 1..4 has exactly N voxels (tiles few, last tile 127/128/129 or 255/256/257 rows).  ``full81``: one
    level-0 voxel in each of 6x6x6 level-3 cells (3x3x3 level-4 cells) in time planes 0..2, so that level-3 voxels and
    the centre level-4 voxel meet all 81 offsets.  ``cls-lL``: the class counts of ``cls-tile-edges`` at level L (the
    level-0 coordinates of ``classes`` times 2^L).  ``mos4d-4scan``: four sparse scans in time planes 0..3."""
    if name.startswith("lvl-"):
        n = int(name[4:])
        i = np.arange(n)
        cell = 16 * np.stack([i % 8, (i // 8) % 8, i // 64], -1) - np.array([64, 48, 16])
        base = cell + 2 * rng.integers(0, 8, (n, 3))
        a = rng.integers(0, 8, n)
        b = (a + rng.integers(1, 8, n)) % 8
        xyz = np.vstack([base + CHILD[a], base + CHILD[b]])
        return np.hstack([np.zeros((2 * n, 1), np.int64), xyz, np.zeros((2 * n, 1), np.int64)])
    if name == "full81":
        g = np.arange(6)
        cells = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) * 8 + np.array([-16, -16, 32])
        rows = [np.hstack([np.zeros((216, 1), np.int64), cells + rng.integers(0, 8, (216, 3)), np.full((216, 1), t)])
                for t in range(3)]
        return np.vstack(rows).astype(np.int64)
    if name.startswith("cls-l"):
        c = classes(CLASS_CASES["cls-tile-edges"])
        c[:, 1:4] <<= int(name[-1])
        return c
    if name == "mos4d-4scan":
        rows = []
        for t in range(4):
            c = random_box((-20, -20, -20), 40, 0.05, rng)
            c[:, 4] = t
            rows.append(c)
        return np.vstack(rows)
    raise KeyError(name)


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
    elif name in DEEP_CASES:
        coords = deep_input(name, rng)
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


# ================================================================ levels 1-4: every other layer of the forward ====
# A deep probe tests one layer (``DEEP_LAYERS``) of the fused forward.  Three pieces make up its state dict:
#
# * lift (``LiftPlan``): exact inputs at the layer's level.  conv0 keeps the centre offset only; its channels 0..3 are
#   the voxel feature times an 11-bit weight (up to 19 significant bits: the
#   low halves of the hi|lo rows at level 0 are non-zero, read by block8 only); channels 4..7 are f, 2f, f + s, 2f + s'
#   (f the voxel feature, s, s' BN shifts).  Every stride-2 conv gives output
#   channel c one (child class, input channel) term of weight 1 plus a BN shift, every block on the way passes its input
#   on (block1: the identity residual; blocks 2-4: the downsample selects channel c % cin, plus a shift), and the
#   decoder-side inputs are built the same way: B_l = the skip part of the concat row through the downsample of the
#   decoder block at level l, U_l = B_(l+1) through the transposed conv into l, one input channel per (class, channel).
#   Features are multiples of 2^-8 in [0.5, 1) and shifts multiples of 2^-8 in [0.25, 0.5), so every lifted value but
#   conv0's channels 0..3 is a multiple of 2^-8 in [0.25, 8): at most 11 significant bits, exact in fp16, TF32 and fp32.
# * layer under test: random weights bounded away from zero and random BN; the other conv of its block is the
#   centre-offset identity (conv1 is read through conv2 = identity with the downsample zero, conv2 is fed H = its
#   block's input through conv1 = identity, with a random downsample).
# * readout: the value at level L, channel 8g + c reaches the logit of column c with weights 1.0 alone: the first
#   downsample or transposed conv after the layer selects channel group g, every transposed conv uses all eight child
#   classes, decoder blocks pass the "up" part of their concat row through the downsample, block8's downsample and
#   ``final`` are the identity.
OFF3 = [O.kernel_offsets([3, 3, 3, 3], [2 ** L] * 3 + [1]).astype(np.int64) for L in range(5)]
IDENTITY3 = 40                               # kernel offset (0, 0, 0, 0) of the 3x3x3x3 convs
DEEP_FEAT_BITS = 8
# level L -> (stride-2 conv into L, its BN, block at L, conv channels, block output channels)
ENC = {1: ("conv1p1s2", "bn1", "block1", 8, 8), 2: ("conv2p2s2", "bn2", "block2", 8, 16),
       3: ("conv3p4s2", "bn3", "block3", 16, 32), 4: ("conv4p8s2", "bn4", "block4", 32, 64)}
# level l -> (transposed conv into l, its BN, decoder block at l, its input channels, "up" channels, skip channels)
DEC = {3: ("convtr4p16s2", "bntr4", "block5", 64, 64, 32), 2: ("convtr5p8s2", "bntr5", "block6", 64, 32, 16),
       1: ("convtr6p4s2", "bntr6", "block7", 32, 16, 8), 0: ("convtr7p2s2", "bntr7", "block8", 16, 8, 8)}
DEEP_LAYERS = (("conv2p2s2", "conv3p4s2", "conv4p8s2") +
               tuple(f"block{b}.conv{i}" for b in (1, 2, 3, 4) for i in (1, 2)) +
               ("convtr4p16s2", "convtr5p8s2", "convtr6p4s2") +
               tuple(f"block{b}.conv{i}" for b in (5, 6, 7, 8) for i in (1, 2)))

# The arithmetic of every layer of the fused forward, restated from sps_net_finalize and conv_dispatch (net.cu, api.cu):
# layer -> (K, cin, cout, cin2 of the fused 1x1 term, fp16 forward's precision options, its cin_split, TF32 backend's
# kernel).  fp16 options: FOLD_LO = the low parts of the weights ride in accumulator columns 8..15 (weight hi + lo),
# IN_SPLIT / IN2_SPLIT = the input / the 1x1 term's input rows are hi|lo pairs, OUT_SPLIT = the output is.  TF32
# backend: "tc" = tcgen05 with TF32-rounded weights (every layer with a K-major TF32 copy), "simt" = fp32 CUDA cores.
PLAN = {
    "conv1p1s2": (8, 8, 8, 0, "FOLD_LO IN_SPLIT", 0, "simt"),
    "block1.conv1": (81, 8, 8, 0, "FOLD_LO", 0, "tc"),
    "block1.conv2": (81, 8, 8, 0, "FOLD_LO", 0, "tc"),
    "conv2p2s2": (8, 8, 8, 0, "FOLD_LO", 0, "simt"),
    "block2.conv1": (81, 8, 16, 0, "", 0, "tc"),
    "block2.conv2": (81, 16, 16, 8, "", 0, "tc"),
    "conv3p4s2": (8, 16, 16, 0, "", 0, "tc"),
    "block3.conv1": (81, 16, 32, 0, "", 0, "tc"),
    "block3.conv2": (81, 32, 32, 16, "", 0, "tc"),
    "conv4p8s2": (8, 32, 32, 0, "", 0, "tc"),
    "block4.conv1": (81, 32, 64, 0, "", 0, "tc"),
    "block4.conv2": (81, 64, 64, 32, "", 0, "tc"),
    "convtr4p16s2": (8, 64, 64, 0, "", 0, "tc"),
    "block5.conv1": (81, 96, 64, 0, "", 64, "tc"),
    "block5.conv2": (81, 64, 64, 96, "", 0, "tc"),
    "convtr5p8s2": (8, 64, 32, 0, "", 0, "tc"),
    "block6.conv1": (81, 48, 32, 0, "", 0, "tc"),
    "block6.conv2": (81, 32, 32, 48, "", 0, "tc"),
    "convtr6p4s2": (8, 32, 16, 0, "", 0, "tc"),
    "block7.conv1": (81, 24, 16, 0, "", 0, "tc"),
    "block7.conv2": (81, 16, 16, 24, "", 0, "tc"),
    "convtr7p2s2": (8, 16, 8, 0, "FOLD_LO OUT_SPLIT", 0, "tc"),
    "block8.conv1": (81, 16, 8, 0, "FOLD_LO IN_SPLIT", 0, "tc"),
    "block8.conv2": (81, 8, 8, 16, "FOLD_LO IN2_SPLIT", 0, "tc"),
}
# Bound of a deep probe: storage term + BOUND_DEEP * S.  Under every backend's model the products are exact (fp32 x
# fp32 is not, but the model's float64 product differs from fp32's by 2^-24 of it, inside S) and only the fp32
# accumulation rounds: at most 2^-24 of a partial sum per addition.  The partial sums of random-sign products stay
# far below S, their sum of absolute values; 2^-20 S allows sixteen additions that each round at the full S.
BOUND_DEEP = 2.0 ** -20


def deep_features(n, rng):
    return rng.integers(1 << (DEEP_FEAT_BITS - 1), 1 << DEEP_FEAT_BITS, n) / float(1 << DEEP_FEAT_BITS)


def grid_shift(rng, n):
    """n distinct multiples of 2^-8 in [0.25, 0.5)."""
    return (64 + rng.choice(64, n, replace=False)) / 256.0


class LiftPlan:
    """Weights of the lift, drawn once: the same lifted tensors serve every probe."""

    def __init__(self, seed=3):
        rng = np.random.default_rng(seed)
        self.w0 = np.concatenate([rng.integers(1024, 2048, 4) / 1024.0, [1.0, 2.0, 1.0, 2.0]])
        self.sh0 = np.concatenate([np.zeros(4), [0.0, 0.0], grid_shift(rng, 2)])
        self.down, self.blk, self.dec, self.up = {}, {}, {}, {}
        for L, (_, _, _, cin, cout) in ENC.items():
            cls = rng.permutation(8)[np.arange(cin) % 8]
            ch = 4 + rng.permutation(4)[np.arange(cin) % 4] if L == 1 else rng.permutation(cin)
            self.down[L] = (cls, ch, grid_shift(rng, cin))
            if L > 1:
                self.blk[L] = grid_shift(rng, cout)
        for l, (_, _, _, cin, up, skip) in DEC.items():
            self.up[l] = ((np.arange(up)[None, :] + 3 * np.arange(8)[:, None] + rng.integers(0, cin)) % cin,
                          grid_shift(rng, up))
            if l >= 1:
                self.dec[l] = grid_shift(rng, up)


LIFT = LiftPlan()


def install_encoder(sd, lp, upto, keep=()):
    """conv0 and the encoder's lift up to level ``upto``; layers named in ``keep`` are left alone."""
    sd["conv0p1s1.kernel"][CENTRE, 0] = lp.w0
    set_probe_bn(sd, "bn0", 8, lp.sh0)
    for L in range(1, upto + 1):
        conv, bn, blk, cin, cout = ENC[L]
        if conv not in keep:
            cls, ch, sh = lp.down[L]
            w = np.zeros((8, cin, cin), np.float32)
            w[cls, ch, np.arange(cin)] = 1.0
            sd[conv + ".kernel"] = w
            set_probe_bn(sd, bn, cin, sh)
        if L > 1 and blk not in keep:
            ds = np.zeros((cin, cout), np.float32)
            ds[np.arange(cout) % cin, np.arange(cout)] = 1.0
            sd[blk + ".0.downsample.0.kernel"] = ds
            set_probe_bn(sd, blk + ".0.downsample.1", cout, lp.blk[L])


def install_b(sd, lp, l):
    """B_l (l < 4): the skip part of the level-l concat row through its decoder block's downsample."""
    _, _, blk, _, up, skip = DEC[l]
    ds = np.zeros((up + skip, up), np.float32)
    ds[up + np.arange(up) % skip, np.arange(up)] = 1.0
    sd[blk + ".0.downsample.0.kernel"] = ds
    set_probe_bn(sd, blk + ".0.downsample.1", up, lp.dec[l])


def install_u(sd, lp, l):
    """U_l: B_(l+1) through the transposed conv into level l, input channel sel[k, d] for class k, channel d."""
    conv, bn, _, cin, up, _ = DEC[l]
    sel, sh = lp.up[l]
    w = np.zeros((8, cin, up), np.float32)
    w[np.arange(8)[:, None], sel, np.arange(up)[None, :]] = 1.0
    sd[conv + ".kernel"] = w
    set_probe_bn(sd, bn, up, sh)


def install_readout(sd, start, L, g):
    """Route channel group g of the tensor at level L to the head: ``start`` = "skip" / "up" (that part of the level-L
    concat row, read by the decoder block at L) or "B" (the decoder input at L: B4 or a decoder block's output)."""
    sel = 8 * g + np.arange(8)
    if start != "B":
        _, _, blk, _, up, skip = DEC[L]
        ds = np.zeros((up + skip, up), np.float32)
        ds[(up if start == "skip" else 0) + sel, np.arange(8)] = 1.0
        sd[blk + ".0.downsample.0.kernel"] = ds
        sel = np.arange(8)
    for l in range(L - 1, -1, -1):
        conv, _, blk, cin, up, skip = DEC[l]
        w = np.zeros((8, cin, up), np.float32)
        w[:, sel, np.arange(8)] = 1.0
        sd[conv + ".kernel"] = w
        sel = np.arange(8)
        if l >= 1:
            ds = np.zeros((up + skip, up), np.float32)
            ds[np.arange(8), np.arange(8)] = 1.0
            sd[blk + ".0.downsample.0.kernel"] = ds


def random_bn(sd, prefix, C, rng):
    """A random BN whose shift leans positive: the random-sign sums of a voxel with few neighbours are a few tenths,
    and a centred shift would let the ReLU clamp most of them."""
    sd[prefix + ".bn.weight"] = rng.uniform(0.5, 1.5, C).astype(np.float32)
    sd[prefix + ".bn.bias"] = rng.uniform(0.1, 0.4, C).astype(np.float32)
    sd[prefix + ".bn.running_mean"] = rng.uniform(-0.2, 0.2, C).astype(np.float32)
    sd[prefix + ".bn.running_var"] = rng.uniform(0.5, 1.5, C).astype(np.float32)


def random_kernel(rng, shape):
    """``bounded`` weights / sqrt(fan-in): random signs keep the partial sums of the products far below S (see
    BOUND_DEEP), and outputs stay far inside fp16's range."""
    fan = int(np.prod(shape[:-1]))
    return (bounded(rng, shape) / np.sqrt(fan)).astype(np.float32)


def identity3(cin, cout):
    w = np.zeros((81, cin, cout), np.float32)
    m = min(cin, cout)
    w[IDENTITY3, np.arange(m), np.arange(m)] = 1.0
    return w


def block_level(b):
    return b if b <= 4 else 8 - b


def probe_info(layer):
    """(level of the tensor under test, readout start, oracle tap, channels of the tensor under test)."""
    if layer in ("conv2p2s2", "conv3p4s2", "conv4p8s2"):
        L = int(layer[4])
        return L, "B" if L == 4 else "skip", layer, ENC[L][3]
    if layer.startswith("convtr"):
        l = {"convtr4p16s2": 3, "convtr5p8s2": 2, "convtr6p4s2": 1}[layer]
        return l, "up", layer, DEC[l][4]
    b = int(layer[5])
    L = block_level(b)
    if b <= 4:
        return L, "B" if L == 4 else "skip", f"block{b}", ENC[L][4]
    if b < 8:
        return L, "B", f"block{b}", DEC[L][4]
    return 0, None, "final" if layer.endswith("2") else "block8", 8


def deep_groups(layer):
    return 1 if layer == "block8.conv2" else probe_info(layer)[3] // 8


def deep_probe(layer, g=0, seed=0):
    """State dict of the probe of ``layer`` that reads channel group g; the random weights depend on the layer and
    ``seed`` only, not on g."""
    rng = np.random.default_rng([seed, DEEP_LAYERS.index(layer)])
    sd = zero_net("up")
    L, start, _, _ = probe_info(layer)
    if layer.startswith("conv") and not layer.startswith("convtr"):
        conv, bn, blk, cin, cout = ENC[L]
        install_encoder(sd, LIFT, L, keep=(conv, blk))
        sd[conv + ".kernel"] = random_kernel(rng, (8, cin, cin))
        random_bn(sd, bn, cin, rng)
        ds = np.zeros((cin, cout), np.float32)
        ds[np.arange(cin), np.arange(cin)] = 1.0
        sd[blk + ".0.downsample.0.kernel"] = ds
    elif layer.startswith("convtr"):
        conv, bn, _, cin, up, _ = DEC[L]
        install_encoder(sd, LIFT, 4)
        if L + 1 < 4:
            install_b(sd, LIFT, L + 1)
        sd[conv + ".kernel"] = random_kernel(rng, (8, cin, up))
        random_bn(sd, bn, up, rng)
    else:
        b, i = int(layer[5]), int(layer[-1])
        blk = f"block{b}"
        if b <= 4:
            install_encoder(sd, LIFT, L, keep=(blk,))
            cin, cout = ENC[L][3], ENC[L][4]
        else:
            install_encoder(sd, LIFT, 4)
            if L + 1 < 4:
                install_b(sd, LIFT, L + 1)
            install_u(sd, LIFT, L)
            cin, cout = DEC[L][4] + DEC[L][5], DEC[L][4]
        if i == 1:
            sd[blk + ".0.conv1.kernel"] = random_kernel(rng, (81, cin, cout))
            random_bn(sd, blk + ".0.norm1", cout, rng)
            sd[blk + ".0.conv2.kernel"] = identity3(cout, cout)
            if cin != cout:
                sd[blk + ".0.downsample.0.kernel"] = np.zeros((cin, cout), np.float32)
        else:
            sd[blk + ".0.conv1.kernel"] = identity3(cin, cout)
            sd[blk + ".0.conv2.kernel"] = random_kernel(rng, (81, cout, cout))
            random_bn(sd, blk + ".0.norm2", cout, rng)
            if cin != cout:
                sd[blk + ".0.downsample.0.kernel"] = random_kernel(rng, (cin, cout))
                random_bn(sd, blk + ".0.downsample.1", cout, rng)
        if b == 8 and i == 2:
            sd["final.kernel"] = bounded(rng, (8, 8))
            sd["final.bias"] = rng.uniform(-0.5, 0.5, (1, 8)).astype(np.float32)
    if start is not None:
        install_readout(sd, start, L, g)
    return sd


# ---------------------------------------------------------------- deep probes: arithmetic models ----
def fold(sd, kname, bn, backend):
    """Folded weights and shift of a layer as ``backend`` computes with them: None = float64 BN (the oracle's
    arithmetic), else sps_net_finalize's fp32 fold (``bn_fold_f32``, kernel x scale in double, rounded to fp32)."""
    k = np.asarray(sd[kname], np.float64)
    if backend is None:
        g, b, m, v = (np.asarray(sd[bn + ".bn." + s], np.float64) for s in ("weight", "bias", "running_mean", "running_var"))
        v = np.where(np.asarray(sd[bn + ".bn.running_var"]) == PROBE_VAR, 1 - 1e-5, v)
        scale = g / np.sqrt(v + 1e-5)
        return k * scale, b - m * scale
    scale, shift = bn_fold_f32(sd, bn)
    return np.asarray(k * scale, np.float32).astype(np.float64), shift


def model_weights(w, layer, backend):
    """The weights the backend multiplies with: fp32 (fp32 backend, CUDA-core layers of the TF32 backend), TF32
    nearest-even (tcgen05 layers of the TF32 backend), fp16 or fp16 hi + lo (FOLD_LO) on the fp16 backend."""
    if backend in (None, 1) or (backend == 2 and PLAN[layer][6] == "simt"):
        return w
    if backend == 2:
        return tf32_rne(w)
    return f16_hilo(w) if "FOLD_LO" in PLAN[layer][4] else np.asarray(w, np.float32).astype(np.float16).astype(np.float64)


def store_term(x, backend, logit=False):
    """One unit in the last place of the stored format at x: fp16 and TF32 rows; fp32 rows and logits are exact."""
    return np.zeros_like(x) if backend in (None, 1) or logit else ulp10(x)


def floor_to(c, s):
    c = np.array(c, np.int64)
    c[:, 1:4] = np.floor_divide(c[:, 1:4], s) * s
    return c


class DeepLevels:
    """Levels 0..4 of an input by floor-to-stride (row order of np.unique, not the product's), one ``Lookup`` per level,
    and the lifted tensors of every level under ``LIFT`` (float64, exact)."""

    def __init__(self, c0, feat, lp=LIFT):
        self.c = [np.asarray(c0, np.int64)]
        for L in range(1, 5):
            self.c.append(np.unique(floor_to(self.c[-1], 2 ** L), axis=0))
        self.lk = [Lookup(c) for c in self.c]
        self.par = [self.lk[L + 1](floor_to(self.c[L], 2 ** (L + 1))) for L in range(4)]
        self.cls = [child_class(self.c[L] >> L) for L in range(4)]        # child class inside the level-(L+1) parent
        self.skip = [np.asarray(feat, np.float64)[:, None] * lp.w0 + lp.sh0]
        self.E = [None]
        for L in range(1, 5):
            cls, ch, sh = lp.down[L]
            x = self.stride_in(L, self.skip[L - 1])
            self.E.append(x[np.arange(len(x))[:, None], cls[None, :], ch[None, :]] + sh)
            _, _, _, cin, cout = ENC[L]
            self.skip.append(self.E[L] if L == 1 else self.E[L][:, np.arange(cout) % cin] + lp.blk[L])
        self.B = {4: self.skip[4]}
        for l in (3, 2, 1):
            up, skip = DEC[l][4], DEC[l][5]
            self.B[l] = self.skip[l][:, np.arange(up) % skip] + lp.dec[l]
        self.U = {}
        for l in (3, 2, 1, 0):
            sel, sh = lp.up[l]
            self.U[l] = self.B[l + 1][self.par[l][:, None], sel[self.cls[l]]] + sh

    def children(self, L, rows=None):
        """[R, 8] rows of the level-(L-1) children of level-L voxels (-1 absent)."""
        c = self.c[L] if rows is None else self.c[L][rows]
        out = np.empty((len(c), 8), np.int64)
        for j in range(8):
            q = c.copy()
            q[:, 1:4] += CHILD[j] * 2 ** (L - 1)
            out[:, j] = self.lk[L - 1](q)
        return out

    def stride_in(self, L, x, rows=None):
        """[R, 8, C]: the children's rows of x (zero where absent)."""
        ch = self.children(L, rows)
        return np.where(ch[:, :, None] >= 0, x[np.maximum(ch, 0)], 0.0)

    def nbr3(self, L, rows):
        """[R, 81] rows of the 3x3x3x3 neighbours at level L (offsets x 2^L in x, y, z, +-1 in t)."""
        c = self.c[L][rows]
        out = np.empty((len(c), 81), np.int64)
        for k in range(81):
            q = c.copy()
            q[:, 1:5] += OFF3[L][k]
            out[:, k] = self.lk[L](q)
        return out

    def ancestors(self, L, rows0):
        return self.lk[L](floor_to(self.c[0][rows0], 2 ** L))

    def skip0(self, backend):
        """skip0 as the backend stores it (conv0's channels 0..3 carry up to 19 significant bits)."""
        return SKIP0_STORE[1 if backend is None else backend](self.skip[0])

    def cat(self, l, backend):
        return np.hstack([self.U[l], self.skip0(backend) if l == 0 else self.skip[l]])

    def layer_input(self, layer, backend):
        """(x, x2): the input rows of the layer under test and of its fused 1x1 term, at the layer's input level."""
        L, _, _, _ = probe_info(layer)
        if layer.startswith("conv") and not layer.startswith("convtr"):
            return self.skip[L - 1], None
        if layer.startswith("convtr"):
            return self.B[L + 1], None
        b, i = int(layer[5]), int(layer[-1])
        x = self.E[L] if b <= 4 else self.cat(L, backend)
        if i == 1:
            return x, None
        cout = ENC[L][4] if b <= 4 else DEC[L][4]
        h = np.zeros((len(x), cout))
        m = min(cout, x.shape[1])
        h[:, :m] = x[:, :m]
        return h, (x if b == 1 or x.shape[1] != cout else None)


def acc_rows(terms):
    """Sum of (x [R, n], w [R, n, C] or [n, C]) products -> (sum, S, smallest non-zero |x| over the terms)."""
    out = S = 0.0
    xmin = np.full(len(terms[0][0]), np.inf)
    for x, w in terms:
        if w.ndim == 2:
            out = out + x @ w
            S = S + np.abs(x) @ np.abs(w)
        else:
            out = out + np.einsum("rn,rnc->rc", x, w)
            S = S + np.einsum("rn,rnc->rc", np.abs(x), np.abs(w))
        ax = np.where(x != 0, np.abs(x), np.inf)
        xmin = np.minimum(xmin, ax.min(1, initial=np.inf))
    return out, S, xmin


def deep_reference(dl, layer, sd, backend, rows0):
    """The layer under test at the level-L ancestors of the level-0 rows ``rows0``, as read out through the head:
    (ref [R, C], bound [R, C], margin [R, C]).  ``backend`` None: float64 with the oracle's BN.  ``margin``: a lower
    bound of the smallest non-zero |w x| behind an output that survives the ReLU, minus BOUND_DEEP * S (inf for
    clamped outputs); where it is positive a lost product cannot hide under the accumulation term of the bound."""
    L, _, _, C = probe_info(layer)
    anc = dl.ancestors(L, rows0)
    assert (anc >= 0).all()
    u, inv = np.unique(anc, return_inverse=True)
    x, x2 = dl.layer_input(layer, backend)
    b = int(layer[5]) if layer.startswith("block") else 0
    res = None
    if layer.startswith("conv") and not layer.startswith("convtr"):
        conv, bn, _, cin, _ = ENC[L]
        w, sh = fold(sd, conv + ".kernel", bn, backend)
        w = model_weights(w, layer, backend)
        xs = dl.stride_in(L, x, u)
        out, S, xmin = acc_rows([(xs.reshape(len(u), -1), w.reshape(-1, cin))])
        wmin = np.abs(w).reshape(-1, cin).min(0)
    elif layer.startswith("convtr"):
        conv, bn = DEC[L][:2]
        w, sh = fold(sd, conv + ".kernel", bn, backend)
        w = model_weights(w, layer, backend)
        out, S, xmin = acc_rows([(x[dl.par[L][u]], w[dl.cls[L][u]])])
        wmin = np.abs(w).min((0, 1))
    else:
        i = int(layer[-1])
        blk = f"block{b}"
        pre = f"{blk}.0.conv{i}.kernel"
        w, sh = fold(sd, pre, f"{blk}.0.norm{i}", backend)
        w = model_weights(w, layer, backend)
        nb = dl.nbr3(L, u)
        xs = np.where(nb[:, :, None] >= 0, x[np.maximum(nb, 0)], 0.0)
        terms = [(xs.reshape(len(u), -1), w.reshape(-1, w.shape[-1]))]
        wmin = np.abs(w).reshape(-1, w.shape[-1]).min(0)
        if i == 2 and f"{blk}.0.downsample.0.kernel" in sd:
            w2, sh2 = fold(sd, f"{blk}.0.downsample.0.kernel", f"{blk}.0.downsample.1", backend)
            w2 = model_weights(w2, layer, backend)
            terms.append((x2[u], w2))
            sh = sh + sh2
            wmin = np.minimum(wmin, np.abs(w2).min(0))
        elif b == 1 and i == 2:
            res = dl.E[1][u]
        out, S, xmin = acc_rows(terms)
        if b == 1 and i == 1:
            res = dl.E[1][u]
    if backend is not None:
        sh = np.asarray(sh, np.float32).astype(np.float64)
    out = out + sh
    S = S + np.abs(sh)
    pmin = xmin[:, None] * wmin[None, :]            # lower bound of the smallest non-zero |w x| behind each output
    conv1_of_block1 = b == 1 and layer.endswith("1")
    if res is not None and not conv1_of_block1:     # block1.conv2: the identity residual, added before the ReLU
        out, S = out + res, S + res
    out = np.maximum(out, 0.0)
    alive = out > 0
    if conv1_of_block1:                             # read through conv2 = identity plus E1: one more stored sum
        h = out
        out = h + res
        bound = store_term(h, backend) + store_term(out, backend) + BOUND_DEEP * S
    elif layer == "block8.conv2":                   # the fp32 logit of the fused head: no storage rounding
        fk = np.asarray(sd["final.kernel"], np.float64)
        fb = np.asarray(sd["final.bias"], np.float64)[0]
        pmin = np.where(alive[:, :, None], pmin[:, :, None] * np.abs(fk)[None], np.inf).min(1)
        S = S @ np.abs(fk) + np.abs(out) @ np.abs(fk) + np.abs(fb)
        out = out @ fk + fb
        alive = np.isfinite(pmin)
        bound = BOUND_DEEP * S
    else:
        bound = store_term(out, backend) + BOUND_DEEP * S
    margin = np.where(alive, pmin - BOUND_DEEP * S, np.inf)
    return out[inv], bound[inv], margin[inv]
