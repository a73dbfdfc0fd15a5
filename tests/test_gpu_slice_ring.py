"""The tensor-core convolution stages each tile's kernel-map slice in a ring of 82 entries (nact + 1 per tile, up to
8 tiles in flight).  These layers give every CTA a sequence of tiles whose present-offset counts alternate between
small and all 81 (the ring wraps at a different entry on every pass), or stay small (8 tiles in flight, many wraps), and
check the output against the float64 numpy statement of test_gpu_conv.py -- in physical order from the dense map, and
in a permuted order from per-tile slices (the fused forward's path)."""
import numpy as np
import pytest
import torch

from test_gpu_conv import f16, ref_conv, tf32

pytestmark = pytest.mark.gpu

CTAS = 296        # persistent grid of the N <= 64 kernels: two CTAs on each of the B200's 148 SMs
PASSES = {81: 10, 8: 16}   # tiles per CTA: the ring wraps on nearly every CTA


def tile_offsets(rng, K, ntiles):
    """Present offsets of each tile in processing order.  CTA b takes tiles b, b + CTAS, ...: on two thirds of the CTAs
    the tiles alternate between 81 and 1-30 offsets (starting with either), on the rest they have 1-24."""
    sets = []
    for t in range(ntiles):
        b, it = t % CTAS, t // CTAS
        if K == 81 and b % 3 < 2 and (it + b) % 2 == 0:
            n = 81
        else:
            n = int(rng.integers(1, 31 if b % 3 < 2 else 25)) if K == 81 else int(rng.integers(1, K + 1))
        sets.append(np.sort(rng.choice(K, n, replace=False)))
    return sets


def sorted_map(rng, K, V, sets, density=0.5):
    """nbr[k][j] of the row processed at position j: a neighbour with probability `density` for the tile's present
    offsets (the tile's first row always has one), -1 for the others."""
    nbr = np.full((K, V), -1, np.int32)
    for t, ks in enumerate(sets):
        lo, hi = t * 128, min(V, (t + 1) * 128)
        hit = rng.random((len(ks), hi - lo)) < density
        hit[:, 0] = True
        nbr[ks, lo:hi] = np.where(hit, rng.integers(0, V, (len(ks), hi - lo)), -1)
    return nbr


def padded(nbr):
    """[K][ld] map with ld a multiple of 32: full tiles take the 16-byte copy path, the ragged last one the per-row path"""
    ld = (nbr.shape[1] + 31) // 32 * 32
    m = np.full((nbr.shape[0], ld), -1, np.int32)
    m[:, :nbr.shape[1]] = nbr
    return m, ld


def slices_and_masks(nbr_sorted, perm, sets):
    ntiles = len(sets)
    V = perm.shape[0]
    sl = np.full((ntiles, 82, 128), -1, np.int32)
    masks = np.zeros((ntiles, 4), np.uint32)
    for t, ks in enumerate(sets):
        lo, hi = t * 128, min(V, (t + 1) * 128)
        sl[t, :len(ks), :hi - lo] = nbr_sorted[ks, lo:hi]
        sl[t, len(ks), :hi - lo] = perm[lo:hi]
        for k in ks:
            masks[t, k >> 5] |= np.uint32(1 << (k & 31))
    return sl, masks.view(np.int32)


@pytest.mark.parametrize("K,cin,cout,cin_split,fused", [
    (81, 8, 16, 0, False),      # one 16-byte group per offset: 8 offsets per stage
    (81, 16, 32, 0, True),      # 4 offsets per stage, the 1x1 term in the slots after the last present offset
    (81, 32, 32, 0, False),
    (81, 64, 64, 0, True),      # weight slabs through TMA, the 1x1 term as a stage of its own
    (81, 96, 64, 64, False),    # two channel segments
    (8, 32, 32, 0, False),      # 2x2x2 kernel: 9 entries per tile, 8 tiles in flight
])
def test_mixed_slice_sizes_wrap_the_ring(K, cin, cout, cin_split, fused):
    from sps_b200 import convops, _cabi
    rng = np.random.default_rng(K * 1000 + cin * 10 + cout)
    V = CTAS * PASSES[K] * 128 - 50           # ragged last tile
    ntiles = (V + 127) // 128
    sets = tile_offsets(rng, K, ntiles)
    nbr_sorted = sorted_map(rng, K, V, sets)
    perm = rng.permutation(V).astype(np.int32)
    nbr_perm = np.empty_like(nbr_sorted)
    nbr_perm[:, perm] = nbr_sorted            # physical map of the permuted order: row perm[j] is processed at j
    x = rng.standard_normal((V, cin)).astype(np.float32)
    w = (rng.standard_normal((K, cin, cout)) / np.sqrt(cin * 8)).astype(np.float32)
    shift = rng.standard_normal(cout).astype(np.float32)
    cin2 = cin // 2 if fused else 0
    x2 = rng.standard_normal((V, cin2)).astype(np.float32) if fused else None
    w2 = (rng.standard_normal((cin2, cout)) / np.sqrt(cin2)).astype(np.float32) if fused else None
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a)).cuda()
    n_out = torch.tensor([V], dtype=torch.int32, device="cuda")
    wt = convops.pack_kmajor_f16x(t(w), t(w2) if fused else None, cin_split=cin_split)
    kw = dict(shift=t(shift), relu=True, in2=t(x2).half() if fused else None, weight2=t(w2) if fused else None,
              weight_kmajor=wt, io_f16=True, backend=_cabi.SPS_BACKEND_F16, cin_split=cin_split, n_out_max=V)
    # (a) physical order, dense map: the designed tile sequence as it is
    m, ld = padded(nbr_sorted)
    phys = convops.conv_fwd(t(x).half(), t(w), n_out, map=t(m), map_ld=ld, **kw)
    # (b) permuted order, per-tile slices and masks handed in
    sl, masks = slices_and_masks(nbr_sorted, perm, sets)
    perm_out = convops.conv_fwd(t(x).half(), t(w), n_out, perm=t(perm), tile_mask=t(masks), tile_slices=t(sl), **kw)
    torch.cuda.synchronize()
    x2q = f16(x2) if fused else None
    for got, nbr in ((phys, nbr_sorted), (perm_out, nbr_perm)):
        ref = ref_conv(f16(x), nbr, f16(w), shift=shift, x2=x2q, w2=f16(w2) if fused else None, relu=True)
        got = got[:V].float().cpu().numpy()
        assert np.abs(got - ref).max() < 2e-3 * max(1.0, np.abs(ref).max()), np.abs(got - ref).max()


def test_mixed_slice_sizes_tf32_rows():
    """The same ring on fp32 rows with TF32 operands (backend 2), physical order."""
    from sps_b200 import convops
    rng = np.random.default_rng(7)
    K, cin, cout = 81, 32, 64
    V = CTAS * PASSES[K] * 128 - 50
    sets = tile_offsets(rng, K, (V + 127) // 128)
    nbr = sorted_map(rng, K, V, sets)
    x = tf32(rng.standard_normal((V, cin)).astype(np.float32))
    w = (rng.standard_normal((K, cin, cout)) / np.sqrt(cin * 8)).astype(np.float32)
    shift = rng.standard_normal(cout).astype(np.float32)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a)).cuda()
    n_out = torch.tensor([V], dtype=torch.int32, device="cuda")
    m, ld = padded(nbr)
    out = convops.conv_fwd(t(x), t(w), n_out, map=t(m), map_ld=ld, shift=t(shift), relu=True,
                           weight_kmajor=convops.pack_kmajor(t(w)), backend=2)
    torch.cuda.synchronize()
    ref = ref_conv(x, nbr, w, shift=shift, relu=True, quant=tf32)
    assert np.abs(out[:V].cpu().numpy() - ref).max() < 2e-4 * max(1.0, np.abs(ref).max())
