"""The MinkowskiEngine-shaped layer API (sps_b200.minkowski): a MinkUNet14 built from shim layers
(graph restated here from minkunet.py:52-219) runs layer by layer and must agree with the fused
forward and the oracle; the reference's prune call sequence runs through the shim as written."""
import numpy as np
import pytest
import torch
import torch.nn as nn


class ShimUNet(nn.Module):
    """MinkUNet14 with PLANES (8,16,32,64,64,32,16,8), built from the shim's layers under the
    reference's attribute names (so a reference state_dict loads)."""

    def __init__(self, ME):
        super().__init__()
        P, D = (8, 16, 32, 64, 64, 32, 16, 8), 4
        self.inplanes = 8
        self.conv0p1s1 = ME.MinkowskiConvolution(1, 8, kernel_size=[5, 5, 5, 1], dimension=D)
        self.bn0 = ME.MinkowskiBatchNorm(8)

        def block(planes):
            ds = None
            if self.inplanes != planes:
                ds = nn.Sequential(ME.MinkowskiConvolution(self.inplanes, planes, kernel_size=1, dimension=D),
                                   ME.MinkowskiBatchNorm(planes))
            b = nn.Sequential(ME.BasicBlock(self.inplanes, planes, downsample=ds, dimension=D))
            self.inplanes = planes
            return b
        for i, name in enumerate(["conv1p1s2", "conv2p2s2", "conv3p4s2", "conv4p8s2"]):
            setattr(self, name, ME.MinkowskiConvolution(self.inplanes, self.inplanes, kernel_size=[2, 2, 2, 1],
                                                        stride=[2, 2, 2, 1], dimension=D))
            setattr(self, f"bn{i + 1}", ME.MinkowskiBatchNorm(self.inplanes))
            setattr(self, f"block{i + 1}", block(P[i]))
        skip = [32, 16, 8, 8]
        for i, name in enumerate(["convtr4p16s2", "convtr5p8s2", "convtr6p4s2", "convtr7p2s2"]):
            setattr(self, name, ME.MinkowskiConvolutionTranspose(self.inplanes, P[4 + i], kernel_size=[2, 2, 2, 1],
                                                                 stride=[2, 2, 2, 1], dimension=D))
            setattr(self, f"bntr{4 + i}", ME.MinkowskiBatchNorm(P[4 + i]))
            self.inplanes = P[4 + i] + skip[i]
            setattr(self, f"block{5 + i}", block(P[4 + i]))
        self.final = ME.MinkowskiConvolution(8, 1, kernel_size=1, bias=True, dimension=D)
        self.relu = ME.MinkowskiReLU(inplace=True)
        self.ME = ME

    def forward(self, x):
        ME = self.ME
        skips = [self.relu(self.bn0(self.conv0p1s1(x)))]
        out = skips[0]
        for i, name in enumerate(["conv1p1s2", "conv2p2s2", "conv3p4s2", "conv4p8s2"]):
            out = self.relu(getattr(self, f"bn{i + 1}")(getattr(self, name)(out)))
            out = getattr(self, f"block{i + 1}")(out)
            skips.append(out)
        for i, name in enumerate(["convtr4p16s2", "convtr5p8s2", "convtr6p4s2", "convtr7p2s2"]):
            out = self.relu(getattr(self, f"bntr{4 + i}")(getattr(self, name)(out)))
            out = ME.cat(out, skips[3 - i])
            out = getattr(self, f"block{5 + i}")(out)
        return self.final(out)


@pytest.mark.gpu
def test_layer_by_layer_shim_matches_fused_forward_and_oracle():
    from conftest import make_case
    from oracle import sps_oracle as O
    from sps_b200 import minkowski as ME, engine, _cabi
    rows = make_case("hdl-32", seed=8, n_map_poses=5)
    pts = rows[:, :5]
    sd = O.make_state_dict(seed=0, randomize_bn=True)
    net = ShimUNet(ME)
    net.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
    net = net.cuda().eval()
    coords = torch.as_tensor(pts).cuda() / torch.tensor([1.0, 0.1, 0.1, 0.1, 1.0], device="cuda")   # models.py:21
    feats = 0.5 * torch.ones(len(coords), 1, device="cuda")
    field = ME.TensorField(features=feats, coordinates=coords)
    sparse = field.sparse()
    with torch.no_grad():
        out = net(sparse).slice(field)
    scores = torch.sigmoid(out.features.reshape(-1)).cpu().numpy()
    ref = O.sps_forward(pts, 0.1, sd)
    assert np.abs(scores - ref).max() < 2e-5
    eng = engine.Engine(len(pts))
    eng.set_conv_backend(1)
    fused = eng.forward(engine.Net(sd), torch.as_tensor(pts).cuda(), 0.1).cpu().numpy()
    assert np.abs(scores - fused).max() < 2e-5
    # non-constant point features exercise the voxel mean
    f2 = torch.rand(len(coords), 1, device="cuda")
    st = ME.TensorField(features=f2, coordinates=coords).sparse()
    c0, inv = O.voxelize(pts, 0.1)
    mean = np.zeros(len(c0)); cnt = np.zeros(len(c0))
    np.add.at(mean, inv, f2.cpu().numpy()[:, 0]); np.add.at(cnt, inv, 1)
    assert np.abs(st.F.cpu().numpy()[:, 0] - mean / cnt).max() < 1e-5


@pytest.mark.gpu
def test_reference_prune_call_sequence_through_the_shim():
    """The body of the reference's util.prune (src/sps/datasets/util.py:85-114: SparseTensor x2 on one coordinate
    manager, MinkowskiUnion, mask on the one-hot feature product, MinkowskiPruning, coordinates * ds) runs against the
    shim as written, and agrees with the library's own prune (replicated map hash) and with the oracle."""
    import sps_b200.minkowski as ME
    from oracle import sps_oracle as O
    from sps_b200 import util, synth
    world = synth.World(2)
    base = synth.base_map(world, "tiny", n_poses=6, seed=2)
    scan = synth.scan(world, "tiny", (0.5, -1.0, 0.7), seed=9)
    scan[:50] *= -1.0                                          # negative coordinates: truncation, not floor (util.py:75)
    ds = 0.1
    map_cf = util.to_coords_features(torch.as_tensor(base).cuda(), "map", ds)
    scan_cf = util.to_coords_features(torch.as_tensor(scan).cuda(), "scan", ds)

    def reference_prune(map_coords_feat, scan_coords_feat, ds):
        map_sparse = ME.SparseTensor(features=map_coords_feat.features, coordinates=map_coords_feat.cloud_coords)
        scan_sparse = ME.SparseTensor(features=scan_coords_feat.features, coordinates=scan_coords_feat.cloud_coords,
                                      coordinate_manager=map_sparse.coordinate_manager)
        union = ME.MinkowskiUnion()
        output = union(scan_sparse, map_sparse)
        mask = (output.F[:, 0] * output.F[:, 1]) == 1
        pruning = ME.MinkowskiPruning()
        output = pruning(output, mask)
        submap_points = output.coordinates
        submap_points = submap_points * ds
        return submap_points, len(scan_sparse)

    got, n_scan = reference_prune(map_cf, scan_cf, ds)
    lib_pts, lib_n = util.prune(map_cf, scan_cf, ds)
    ora_pts, ora_n = O.prune(base, scan, ds)
    assert n_scan == lib_n == ora_n
    assert got.dtype == torch.float32
    assert np.array_equal(O.canonical(got.cpu().numpy()), O.canonical(ora_pts))
    assert np.array_equal(O.canonical(lib_pts.cpu().numpy()), O.canonical(ora_pts))
    # union semantics on their own: coincident coordinates add their features, rows in first-occurrence order
    a = ME.SparseTensor(features=torch.tensor([[1., 0.], [1., 0.], [1., 0.]]).cuda(), coordinates=torch.tensor([[1, 2, 3], [1, 2, 3], [4, 5, 6]]).int().cuda())
    b = ME.SparseTensor(features=torch.tensor([[0., 1.], [0., 1.]]).cuda(), coordinates=torch.tensor([[4, 5, 6], [7, 8, -9]]).int().cuda(),
                        coordinate_manager=a.coordinate_manager)
    assert len(a) == 2 and len(b) == 2
    u = ME.MinkowskiUnion()(a, b)
    assert u.C.cpu().tolist() == [[1, 2, 3], [4, 5, 6], [7, 8, -9]] and u.F.cpu().tolist() == [[1., 0.], [1., 1.], [0., 1.]]
