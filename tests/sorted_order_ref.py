"""numpy statement of the shape-sorted processing order of the 3x3x3x3 convolutions (csrc/maps.cu: k_kernel_map_blk3,
k_onesweep_pass, k_tile_masks_perm), computed from a dense kernel map nbr3[81, V] (-1 = absent, offset k = it * 27 + k3
with time plane it = dt + 1 and k3 = (dx+1) + 3 (dy+1) + 9 (dz+1)).

  presence    three 27-bit words per row, one per time plane
  shape_key   [level:3][Gray rank of: has t+1 | has t-1 | 27 spatial bits OR'd over the planes, in ORDER]
  perm        the rows in stable key order (the radix sort is stable and its input is 0..V-1)
  tile_masks  per 128-row tile in perm order: OR of the rows' 81-bit presence words, four uint32 words (the last one 0)
  tile_slices per tile [82][128]: entry e < popcount(mask) = input rows of the tile's e-th present offset (-1 where the
              row lacks it), entry popcount(mask) = the tile's own rows; rows past the level count are -1
"""
from __future__ import annotations

import numpy as np

TILE = 128            # rows of a convolution tile
SLICE_ENTRIES = 82    # SPS_TILE_SLICE_ENTRIES: 81 offsets + the tile's own rows
SORT_TILE = 2048      # keys of one onesweep tile (256 threads x 8 keys)

# shape_bits in csrc/maps.cu: key bit `pos` holds spatial offset ORDER[pos] -- centre, 6 faces, 12 edges, 8 corners
ORDER = (13,
         12, 14, 10, 16, 4, 22,
         9, 11, 15, 17, 3, 5, 21, 23, 1, 7, 19, 25,
         0, 2, 6, 8, 18, 20, 24, 26)


def presence(nbr3: np.ndarray) -> np.ndarray:
    """[81, V] kernel map -> uint32 [V, 3]: bit k3 of word it = offset it * 27 + k3 present."""
    nbr3 = np.asarray(nbr3)
    assert nbr3.shape[0] == 81
    bits = (nbr3 >= 0).reshape(3, 27, -1).astype(np.uint64)
    w = (np.uint64(1) << np.arange(27, dtype=np.uint64))[None, :, None]
    return (bits * w).sum(axis=1).T.astype(np.uint32)


def shape_key(pres: np.ndarray, level: int) -> np.ndarray:
    """uint32 [V] sort keys of one level's rows."""
    pres = np.asarray(pres, np.uint32)
    por = pres[:, 0] | pres[:, 1] | pres[:, 2]
    g = np.zeros(len(pres), np.uint32)
    for pos, k in enumerate(ORDER):
        g |= ((por >> np.uint32(k)) & np.uint32(1)) << np.uint32(pos)
    g |= (pres[:, 0] != 0).astype(np.uint32) << np.uint32(27)      # has t-1
    g |= (pres[:, 2] != 0).astype(np.uint32) << np.uint32(28)      # has t+1
    for s in (1, 2, 4, 8, 16):                                     # binary -> rank in Gray-code order
        g ^= g >> np.uint32(s)
    return g | (np.uint32(level) << np.uint32(29))


def sort_order(key: np.ndarray) -> np.ndarray:
    return np.argsort(key, kind="stable").astype(np.int32)


def mask_words(pres: np.ndarray) -> np.ndarray:
    """uint32 [V, 3]: the 81-bit presence word of every row (bit k = offset k)."""
    pres = np.asarray(pres, np.uint32)
    m0, m1, m2 = pres[:, 0], pres[:, 1], pres[:, 2]
    return np.stack([m0 | (m1 << np.uint32(27)), (m1 >> np.uint32(5)) | (m2 << np.uint32(22)), m2 >> np.uint32(10)],
                    axis=1)


def n_tiles(v: int) -> int:
    return (v + TILE - 1) // TILE


def tile_masks(pres: np.ndarray, perm: np.ndarray) -> np.ndarray:
    """uint32 [ntiles, 4]."""
    words = mask_words(pres)[perm]
    out = np.zeros((n_tiles(len(perm)), 4), np.uint32)
    if len(perm):
        out[:, :3] = np.bitwise_or.reduceat(words, np.arange(0, len(perm), TILE), axis=0)
    return out


def mask_bits(masks: np.ndarray) -> np.ndarray:
    """[ntiles, 4] uint32 -> bool [ntiles, 81]."""
    m = np.asarray(masks, np.uint32)
    k = np.arange(81)
    return ((m[:, k >> 5] >> (k & 31).astype(np.uint32)) & 1).astype(bool)


def tile_slices(nbr3: np.ndarray, pres: np.ndarray, perm: np.ndarray):
    """(slices int32 [ntiles, 82, 128], nact int [ntiles]).  Only entries 0..nact[t] of tile t are defined; the others
    hold -2."""
    nbr3 = np.asarray(nbr3)
    V = len(perm)
    nt = n_tiles(V)
    bits = mask_bits(tile_masks(pres, perm))
    nact = bits.sum(axis=1)
    klist = np.argsort(~bits, axis=1, kind="stable")       # present offsets first, in ascending order
    rows = np.full(nt * TILE, -1, np.int64)
    rows[:V] = perm
    rows = rows.reshape(nt, TILE)
    live = rows >= 0
    out = np.full((nt, SLICE_ENTRIES, TILE), -2, np.int32)
    for e in range(81):
        sel = np.nonzero(e < nact)[0]
        if len(sel) == 0:
            break
        r = rows[sel]
        vals = nbr3[klist[sel, e][:, None], np.where(live[sel], r, 0)]
        out[sel, e] = np.where(live[sel], vals, -1)
    out[np.arange(nt), nact] = rows
    return out, nact


def level_order(nbr3: np.ndarray, level: int) -> dict:
    """Everything the map pass builds for one level."""
    pres = presence(nbr3)
    key = shape_key(pres, level)
    perm = sort_order(key)
    slices, nact = tile_slices(nbr3, pres, perm)
    return {"presence": pres, "key": key, "perm": perm, "tile_mask": tile_masks(pres, perm), "tile_slices": slices,
            "nact": nact}


def defined_entries(nact: np.ndarray) -> np.ndarray:
    """bool [ntiles, 82]: the slice entries a tile defines (0..nact)."""
    return np.arange(SLICE_ENTRIES)[None, :] <= np.asarray(nact)[:, None]


def sort_tiles(counts) -> int:
    return (int(sum(counts)) + SORT_TILE - 1) // SORT_TILE
