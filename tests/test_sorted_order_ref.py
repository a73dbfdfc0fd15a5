"""CPU checks of the numpy statement of the shape-sorted processing order (tests/sorted_order_ref.py) on hand-built
kernel maps, so that the GPU comparison in test_gpu_sorted_order.py rests on a reference that is itself right."""
import numpy as np

import sorted_order_ref as R
from oracle import sps_oracle as O

OFFS3 = [O.kernel_offsets([3, 3, 3, 3], [2 ** L] * 3 + [1]) for L in range(5)]


def kmap(coords, level=0):
    c = np.asarray(coords, np.int32)
    return O.kernel_map(c, c, OFFS3[level])


def gray(r):
    return r ^ (r >> 1)


def raw_bits(key):
    """The shape bits a key ranks (inverse of the prefix XOR)."""
    return gray(int(key) & ((1 << 29) - 1))


def pres_of_raw(raw):
    """Presence words whose shape bits are `raw`: the spatial bits in plane 1, and one of them in plane 0 / 2 for
    has t-1 / has t+1 (the spatial bits are the OR over all three planes)."""
    spatial = 0
    for pos, k in enumerate(R.ORDER):
        if (raw >> pos) & 1:
            spatial |= 1 << k
    low = spatial & -spatial
    assert low or raw < (1 << 27)
    return np.array([[low if (raw >> 27) & 1 else 0, spatial, low if (raw >> 28) & 1 else 0]], np.uint32)


def test_order_table_is_a_permutation_by_distance():
    assert sorted(R.ORDER) == list(range(27))
    dist = [sum(abs(d) for d in ((k % 3) - 1, (k // 3) % 3 - 1, k // 9 - 1)) for k in R.ORDER]
    assert dist == sorted(dist) and dist[0] == 0 and dist.count(1) == 6 and dist.count(2) == 12 and dist.count(3) == 8


def test_isolated_voxel_has_the_centre_only():
    nbr = kmap([[0, 5, 5, 5, 1]])
    pres = R.presence(nbr)
    assert pres.tolist() == [[0, 1 << 13, 0]]
    for L in (0, 3, 4):
        key = R.shape_key(pres, L)
        assert key.tolist() == [1 | (L << 29)]
    o = R.level_order(nbr, 0)
    assert o["perm"].tolist() == [0]
    assert o["tile_mask"].tolist() == [[0, 1 << (40 - 32), 0, 0]]      # offset 40 = (dt 0, centre)
    assert o["nact"].tolist() == [1]
    s = o["tile_slices"]
    assert s[0, 0, 0] == 0 and (s[0, 0, 1:] == -1).all()               # the row is its own centre neighbour
    assert s[0, 1, 0] == 0 and (s[0, 1, 1:] == -1).all()               # entry nact = the tile's own rows
    assert (s[0, 2:] == -2).all()                                      # undefined entries are left alone


def test_full_plane_neighbourhood():
    cube = [[0, x, y, z, 3] for z in range(3) for y in range(3) for x in range(3)]
    nbr = kmap(cube)
    pres = R.presence(nbr)
    centre = 13
    assert pres[centre].tolist() == [0, (1 << 27) - 1, 0]
    key = R.shape_key(pres, 1)
    assert key[centre] >> 29 == 1 and raw_bits(key[centre]) == (1 << 27) - 1
    # corners have 8 neighbours (centre, 3 faces, 3 edges, 1 corner): 8 shape bits
    assert all(bin(raw_bits(k)).count("1") == 8 for k in key[[0, 2, 6, 8, 18, 20, 24, 26]])
    o = R.level_order(nbr, 1)
    assert o["nact"].tolist() == [27]
    assert R.mask_bits(o["tile_mask"])[0].nonzero()[0].tolist() == list(range(27, 54))
    assert sorted(o["perm"].tolist()) == list(range(27)) and (np.diff(key[o["perm"]].astype(np.int64)) >= 0).all()


def test_rows_with_only_earlier_or_only_later_neighbours():
    nbr = kmap([[0, 0, 0, 0, 4], [0, 0, 0, 0, 5], [0, 9, 9, 9, 7]])
    pres = R.presence(nbr)
    assert pres.tolist() == [[0, 1 << 13, 1 << 13], [1 << 13, 1 << 13, 0], [0, 1 << 13, 0]]
    key = R.shape_key(pres, 0)
    assert [raw_bits(k) for k in key] == [1 | (1 << 28), 1 | (1 << 27), 1]
    o = R.level_order(nbr, 0)
    assert o["perm"].tolist() == [2, 1, 0]            # ranks 1 < gray^-1(1 | 1 << 27) < gray^-1(1 | 1 << 28)
    assert o["nact"].tolist() == [3]                  # offsets 13 (t-1), 40 (centre), 67 (t+1)
    assert R.mask_bits(o["tile_mask"])[0].nonzero()[0].tolist() == [13, 40, 67]
    s = o["tile_slices"][0]
    assert s[0, :3].tolist() == [-1, 0, -1]           # offset 13 (dt = -1): only row 1 (t = 5) has it, and it is row 0
    assert s[1, :3].tolist() == [2, 1, 0]             # offset 40: every row is its own centre
    assert s[2, :3].tolist() == [-1, -1, 1]           # offset 67 (dt = +1): row 0 -> row 1
    assert s[3, :3].tolist() == [2, 1, 0]


def test_gray_rank_of_adjacent_shapes():
    # centre only -> rank 1; centre + the -x face (key bit 1) -> gray 3 = rank 2
    assert R.shape_key(pres_of_raw(0b1), 0)[0] == 1
    assert R.shape_key(pres_of_raw(0b11), 0)[0] == 2
    for r in (1, 2, 3, 100, 12345, (1 << 27) - 2, (1 << 27) - 1, (1 << 28) + 7, (1 << 29) - 3):
        k0 = R.shape_key(pres_of_raw(gray(r)), 2)[0]
        k1 = R.shape_key(pres_of_raw(gray(r + 1)), 2)[0]
        assert (k0, k1) == (r | (2 << 29), (r + 1) | (2 << 29)), r
        assert bin(gray(r) ^ gray(r + 1)).count("1") == 1


def naive_order(nbr3, level):
    """Row-by-row statement of the same structures (no vectorisation)."""
    V = nbr3.shape[1]
    keys = []
    for v in range(V):
        planes = [sum(1 << k3 for k3 in range(27) if nbr3[it * 27 + k3, v] >= 0) for it in range(3)]
        por = planes[0] | planes[1] | planes[2]
        g = sum(((por >> k) & 1) << pos for pos, k in enumerate(R.ORDER))
        g |= (planes[0] != 0) << 27 | (planes[2] != 0) << 28
        r = 0
        while g:
            r ^= g
            g >>= 1
        keys.append(r | level << 29)
    perm = sorted(range(V), key=lambda v: keys[v])
    masks, slices = [], []
    for t in range(R.n_tiles(V)):
        rows = perm[128 * t:128 * t + 128]
        ks = [k for k in range(81) if any(nbr3[k, v] >= 0 for v in rows)]
        masks.append(sum(1 << k for k in ks))
        rows = rows + [-1] * (128 - len(rows))
        slices.append([[nbr3[k, v] if v >= 0 else -1 for v in rows] for k in ks] + [rows])
    return keys, perm, masks, slices


def test_ragged_tiles_against_a_row_by_row_statement():
    rng = np.random.default_rng(4)
    # 300 voxels in three time planes of a small box: 3 tiles, the last one with 44 rows
    pts = np.unique(np.column_stack([np.zeros(900, np.int64), rng.integers(0, 12, (900, 3)), rng.integers(0, 3, 900)]),
                    axis=0)
    pts = pts[rng.permutation(len(pts))][:300].astype(np.int32)
    assert len(pts) == 300
    nbr = kmap(pts)
    o = R.level_order(nbr, 3)
    keys, perm, masks, slices = naive_order(nbr, 3)
    assert o["key"].tolist() == keys
    assert o["perm"].tolist() == perm
    assert len(o["tile_mask"]) == 3 and (o["tile_mask"][:, 3] == 0).all()
    got_masks = [int(a) | int(b) << 32 | int(c) << 64 for a, b, c, _ in o["tile_mask"]]
    assert got_masks == masks
    for t in range(3):
        n = o["nact"][t]
        assert n == len(slices[t]) - 1
        assert o["tile_slices"][t, :n + 1].tolist() == slices[t]
    assert (o["tile_slices"][2, :o["nact"][2] + 1, 44:] == -1).all()
    assert R.defined_entries(o["nact"]).sum() == int((o["nact"] + 1).sum())
