"""Host-side mirrors of the three thin model wrappers around the hot-path ops (SURVEY.md §8a):

    HardVoxelizer        paddle3d/models/voxelizers/voxelize.py:26-82
    VoxelMean            paddle3d/models/voxel_encoders/voxel_encoder.py:42-57
    PillarFeatureNet     paddle3d/models/voxel_encoders/pillar_encoder.py:115-210
    PointPillarsScatter  paddle3d/models/middle_encoders/pillar_scatter.py:27-105
    SparseResNet3D       paddle3d/models/middle_encoders/sparse_resnet.py:114-206
    SparseNet3D          paddle3d/models/middle_encoders/sparsenet.py:67-182 (PV-RCNN / Voxel-RCNN family)

Same constructor arguments (the YAML keys stay valid) and the same forward signatures; tensors are
torch CUDA tensors.  Data-dependent row counts stay on the device: the reference slices by a GPU
scalar (a D2H sync per sample, voxelize.py:43-45), here `num_voxels` travels with the tensors and
callers that need exact shapes call `.trim()`.
"""
import os

import numpy as np
import torch

from .ops import pillar_scatter as _ps
from .ops import sparse_nn as sp
from .ops import voxelize as _vox


def _grid(point_cloud_range, voxel_size):
    pcr = np.asarray(point_cloud_range, np.float32)
    vs = np.asarray(voxel_size, np.float32)
    return np.round((pcr[3:] - pcr[:3]) / vs).astype(np.int64)  # x, y, z


class VoxelBatch:
    """(voxels, coors, num_points) of HardVoxelizer.forward plus the device row count."""

    def __init__(self, voxels, coors, num_points, num_voxels):
        self.voxels, self.coors, self.num_points, self.num_voxels = voxels, coors, num_points, num_voxels

    def trim(self):
        """Exact-shape tensors as the reference returns them (costs the one D2H read the reference pays)."""
        n = int(self.num_voxels.sum().item())
        return self.voxels[:n], self.coors[:n], self.num_points[:n]


class HardVoxelizer:
    def __init__(self, voxel_size, point_cloud_range, max_num_points_in_voxel, max_num_voxels):
        self.voxel_size = list(map(float, voxel_size))
        self.point_cloud_range = list(map(float, point_cloud_range))
        self.max_num_points_in_voxel = int(max_num_points_in_voxel)
        self.max_num_voxels = list(max_num_voxels) if isinstance(max_num_voxels, (tuple, list)) else [max_num_voxels] * 2
        self.training = False

    def single_forward(self, point, max_num_voxels, bs_idx):
        voxels, coords, npv, nv = _vox.hard_voxelize(point, self.voxel_size, self.point_cloud_range,
                                                     self.max_num_points_in_voxel, max_num_voxels)
        coors = torch.nn.functional.pad(coords, (1, 0), value=int(bs_idx))  # (b, z, y, x), voxelize.py:51-57
        return voxels, coors, npv, nv

    def forward(self, points):
        """points: list of [N_i, F] tensors (one per sample) or one tensor (export mode, voxelize.py:79-82)."""
        cap = self.max_num_voxels[0] if self.training else self.max_num_voxels[1]
        if isinstance(points, torch.Tensor):
            points = [points]
        if len(points) == 1:
            v, c, n, nv = self.single_forward(points[0], cap, 0)
            return VoxelBatch(v, c, n, nv)
        # batch > 1: like the reference (voxelize.py:68-77) each sample is sliced by its own voxel count — one
        # D2H read per sample — and the pieces are concatenated; the row count of the result is exact.
        vs, cs, ns = [], [], []
        for b, p in enumerate(points):
            v, c, n, nv = self.single_forward(p, cap, b)
            k = int(nv.item())
            vs.append(v[:k])
            cs.append(c[:k])
            ns.append(n[:k])
        v, c, n = torch.cat(vs, 0), torch.cat(cs, 0), torch.cat(ns, 0)
        return VoxelBatch(v, c, n, torch.tensor([v.shape[0]], dtype=torch.int32, device=v.device))

    __call__ = forward


class VoxelMean:
    def __init__(self, in_channels=4):
        self.in_channels = in_channels

    def forward(self, features, num_voxels, coors=None, num=None):
        assert self.in_channels == features.shape[-1]
        return _vox.voxel_mean(features, num_voxels, num)

    __call__ = forward


class PointPillarsScatter:
    def __init__(self, in_channels, voxel_size, point_cloud_range):
        self.in_channels = in_channels
        g = _grid(point_cloud_range, voxel_size)
        self.nx, self.ny = int(g[0]), int(g[1])

    def forward(self, voxel_features, coords, batch_size, num=None):
        """[n, C] + [n, 4] (b, z, y, x) -> [batch, C, ny, nx]."""
        return _ps.pillar_scatter(voxel_features, coords, batch_size, self.ny, self.nx, num)

    __call__ = forward


class PillarFeatureNet:
    """PillarFeatureNet (voxel_encoders/pillar_encoder.py:115-210) with its one PFNLayer (Linear without bias,
    BatchNorm1D eps 1e-3, ReLU, max over the points of a pillar) as one launch.  Decoration: the point features, xyz minus
    the pillar's mean and xy minus the pillar's centre (F + 5 inputs).  `legacy` only changes the reference's training-time
    layer layout, not this inference arithmetic; several PFN layers and `with_distance` are not implemented."""

    def __init__(self, in_channels=4, feat_channels=(64,), with_distance=False, max_num_points_in_voxel=100,
                 voxel_size=(0.2, 0.2, 4), point_cloud_range=(0, -40, -3, 70.4, 40, 1), legacy=True):
        feat_channels = list(feat_channels)
        if len(feat_channels) != 1:
            raise ValueError("PillarFeatureNet: exactly one PFN layer is supported, got feat_channels=%s" % feat_channels)
        if with_distance:
            raise ValueError("PillarFeatureNet: with_distance=True is not supported")
        self.in_channels, self.out_channels = int(in_channels), int(feat_channels[0])
        self.max_num_points_in_voxel, self.legacy = int(max_num_points_in_voxel), legacy
        self.voxel_size = list(map(float, voxel_size))
        self.point_cloud_range = list(map(float, point_cloud_range))
        self.np = None
        self.weight = self.folded = None

    def init_weight(self, seed=0, device="cuda", bn_gain=1.0):
        """Seeded Linear weight [F + 5, C] (kaiming-uniform bound, as synth.kaiming_uniform) and BatchNorm1D with
        gamma = bn_gain, beta 0, mean 0, var 1; folded into (scale, shift) once.  device=None: numpy parameters only."""
        rng = np.random.default_rng(seed)
        d, c = self.in_channels + 5, self.out_channels
        from .synth import kaiming_uniform
        self.np = dict(weight=kaiming_uniform(rng, (d, c), d), gamma=np.full(c, bn_gain, np.float32),
                       beta=np.zeros(c, np.float32), mean=np.zeros(c, np.float32), var=np.ones(c, np.float32), eps=1e-3)
        if device is not None:
            from .ops.pillar_encoder import fold_bn
            p = self.np
            self.weight = torch.from_numpy(p["weight"]).to(device)
            self.folded = fold_bn(p["gamma"], p["beta"], p["mean"], p["var"], p["eps"], device)
        return self

    def forward(self, features, num_points_per_voxel, coors, num=None):
        """features [n, M, F], counts [n], coors [n, 4] (b, z, y, x) -> pillar features [n, C]."""
        from .ops.pillar_encoder import pillar_feature_net
        return pillar_feature_net(features, num_points_per_voxel, coors, self.weight, None, None, None, None, None,
                                  self.voxel_size, self.point_cloud_range, num_voxels=num, folded=self.folded)

    def forward_pixel_h16(self, features, num_points_per_voxel, coors, batch, ny, nx, num=None):
        """Same features, scattered straight into the pixel fp16-pair image: (rows [batch * ny * nx, 2 * C] float16,
        (batch, ny, nx, C)), the input of DenseRPNHead.forward_h16."""
        from .ops.pillar_encoder import pillar_feature_net_pixel_h16
        return pillar_feature_net_pixel_h16(features, num_points_per_voxel, coors, self.weight, None, None, None, None, None,
                                            self.voxel_size, self.point_cloud_range, batch, ny, nx, num_voxels=num,
                                            folded=self.folded)

    __call__ = forward


class _BasicBlock:
    """conv-bn-relu-conv-bn + identity -> relu over one shared rulebook (sparse_resnet.py:65-111)."""

    def __init__(self, channels, key):
        self.conv1 = sp.SubmConv3D(channels, channels, 3, padding=1, bias_attr=True, key=key)
        self.bn1 = sp.BatchNorm(channels, epsilon=1e-3, momentum=0.01)
        self.conv2 = sp.SubmConv3D(channels, channels, 3, padding=1, bias_attr=True, key=key)
        self.bn2 = sp.BatchNorm(channels, epsilon=1e-3, momentum=0.01)
        self.relu = sp.ReLU()

    def layers(self):
        return [self.conv1, self.bn1, self.conv2, self.bn2]

    def __call__(self, x):
        out = self.relu(self.bn1(self.conv1(x)))
        out = self.bn2(self.conv2(out))
        return self.relu(sp.add(out, x))


class SparseResNet3D:
    """21 sparse convs: 5 -> 16 (x5 SubM) -> 32 -> 64 -> 128 over 41x1440x1440 -> 2x180x180, then the dense
    [N, 128*2, 180, 180] BEV tensor (sparse_resnet.py:125-166, 185-206)."""

    STAGES = [  # (Conv3D out channels, kernel, stride, padding, rulebook key of the stage's blocks)
        (32, 3, 2, 1, "res1"),
        (64, 3, 2, 1, "res2"),
        (128, 3, 2, [0, 1, 1], "res3"),
    ]

    def __init__(self, in_channels=128, voxel_size=(0.2, 0.2, 4), point_cloud_range=(0, -40, -3, 70.4, 40, 1)):
        self.in_channels = in_channels
        g = _grid(point_cloud_range, voxel_size)
        self.sparse_shape = [int(g[2]) + 1, int(g[1]), int(g[0])]  # grid[::-1] + [1, 0, 0]
        self.conv_input = [sp.SubmConv3D(in_channels, 16, 3, bias_attr=False, key="res0"),
                           sp.BatchNorm(16, epsilon=1e-3, momentum=0.01), sp.ReLU()]
        self.blocks0 = [_BasicBlock(16, "res0"), _BasicBlock(16, "res0")]
        self.stages = []
        cin = 16
        for cout, k, s, p, key in self.STAGES:
            down = [sp.Conv3D(cin, cout, k, s, padding=p, bias_attr=False), sp.BatchNorm(cout, epsilon=1e-3, momentum=0.01),
                    sp.ReLU()]
            down[0].fuse_subm = ((3, 3, 3), key)  # the level's SubM map comes out of the strided conv's rulebook launch
            self.stages.append((down, [_BasicBlock(cout, key), _BasicBlock(cout, key)]))
            cin = cout
        self.extra_conv = [sp.Conv3D(128, 128, (3, 1, 1), (2, 1, 1), bias_attr=False),
                           sp.BatchNorm(128, epsilon=1e-3, momentum=0.01), sp.ReLU()]
        self.level_caps = None  # optional capacities of the 4 strided index sets
        self.side_stream_rulebooks = os.environ.get("P3D_SIDE_STREAM", "0") != "0"  # measured: no gain (1.214 vs 1.189 ms), off by default
        self._side = {}

    def all_layers(self):
        out = list(self.conv_input[:2])
        for b in self.blocks0:
            out += b.layers()
        for down, blocks in self.stages:
            out += down[:2]
            for b in blocks:
                out += b.layers()
        out += self.extra_conv[:2]
        return out

    def init_weight(self, seed=0, device="cuda", randomize_bn=False, bn_gain=1.0):
        """Seeded stand-in for SparseResNet3D.init_weight (sparse_resnet.py:177-183); no checkpoints exist offline.
        bn_gain: see BatchNorm.init_parameters (sqrt(6) keeps activations O(1) through the 21 layers)."""
        rng = np.random.default_rng(seed)
        for l in self.all_layers():
            if isinstance(l, sp.BatchNorm):
                l.init_parameters(rng, device, randomize=randomize_bn, gain=bn_gain)
            else:
                l.init_parameters(rng, device)
        return self

    def set_precision(self, precision):
        for l in self.all_layers():
            if not isinstance(l, sp.BatchNorm):
                l.precision = precision
        return self

    def set_level_caps(self, caps):
        """Capacities (rows) of the index sets created by the 4 strided convs."""
        convs = [d[0] for d, _ in self.stages] + [self.extra_conv[0]]
        for c, cap in zip(convs, caps):
            c.out_cap = int(cap)
        return self

    def forward_sparse(self, voxel_features, coors, batch_size, num=None):
        shape = [batch_size] + self.sparse_shape + [self.in_channels]
        x = sp.sparse_coo_tensor(coors, voxel_features, shape, num=num)
        if self.side_stream_rulebooks:
            # index sets and neighbour maps of all levels depend on the voxel coordinates only: build them on a side
            # stream while the level-0 feature layers run (every consuming launch waits for its rulebook's event)
            dev = x.index.coords.device
            side = self._side.get(dev)
            if side is None:
                side = self._side[dev] = torch.cuda.Stream(device=dev)
            sp.prepare_rulebooks(x.index, [l for l in self.all_layers() if not isinstance(l, sp.BatchNorm)], side)
        for l in self.conv_input:
            x = l(x)
        for b in self.blocks0:
            x = b(x)
        feats = [x]
        for down, blocks in self.stages:
            for l in down:
                x = l(x)
            for b in blocks:
                x = b(x)
            feats.append(x)
        for l in self.extra_conv:
            x = l(x)
        return x, feats

    def join(self):
        """Join the rulebook side stream into the current stream. Every conv launch already waits for the rulebook it
        uses; this explicit join (after the lazily launched convs have been issued) is what stream capture needs."""
        for dev, side in self._side.items():
            torch.cuda.current_stream(dev).wait_stream(side)

    def forward(self, voxel_features, coors, batch_size, num=None, pixel_h16=False):
        """pixel_h16=False: the reference's dense BEV tensor [N, C*D, H, W] fp32.  True: the same tensor as pixel
        fp16-pair rows (rows, (N, H, W, C*D)) for DenseRPNHead.forward_h16 - no fp32 NCHW pass in between."""
        out, feats = self.forward_sparse(voxel_features, coors, batch_size, num)
        # device counters [n_out, overflow, ...] of the 4 strided index sets: overflow != 0 means output sites were
        # dropped (capacity from set_level_caps too small) and the BEV tensor is incomplete; callers surface it
        self.level_counters = [t.index.counters for t in feats[1:]] + [out.index.counters]
        dense = out.to_pixel_h16() if pixel_h16 else out.to_dense_bev()  # to_dense + transpose(0,4,1,2,3) + reshape
        self.join()
        return dense

    __call__ = forward


class SparseNet3D:
    """12 sparse convs 16/32/64/64 -> 128 (sparsenet.py:75-111); returns the dense BEV tensor and the four multi-scale
    sparse tensors that PV-RCNN / Voxel-RCNN consume (sparsenet.py:160-181)."""

    def __init__(self, in_channels=128, voxel_size=(0.2, 0.2, 4), point_cloud_range=(0, -40, -3, 70.4, 40, 1)):
        self.in_channels = in_channels
        g = _grid(point_cloud_range, voxel_size)
        self.sparse_shape = [int(g[2]) + 1, int(g[1]), int(g[0])]

        def cbr(cin, cout, k, stride=1, padding=0, subm=True):
            conv = (sp.SubmConv3D(cin, cout, k, bias_attr=False) if subm else
                    sp.Conv3D(cin, cout, k, stride, padding=padding, bias_attr=False))
            return [conv, sp.BatchNorm(cout, epsilon=1e-3, momentum=1 - 0.01), sp.ReLU()]

        self.conv_input = cbr(in_channels, 16, 3)
        self.conv1 = [cbr(16, 16, 3)]
        self.conv2 = [cbr(16, 32, 3, 2, 1, subm=False), cbr(32, 32, 3), cbr(32, 32, 3)]
        self.conv3 = [cbr(32, 64, 3, 2, 1, subm=False), cbr(64, 64, 3), cbr(64, 64, 3)]
        self.conv4 = [cbr(64, 64, 3, 2, [0, 1, 1], subm=False), cbr(64, 64, 3), cbr(64, 64, 3)]
        self.extra_conv = cbr(64, 128, (3, 1, 1), (2, 1, 1), 0, subm=False)
        self.num_point_features = 128
        self.backbone_channels = {"x_conv1": 16, "x_conv2": 32, "x_conv3": 64, "x_conv4": 64}

    def sequences(self):
        return [self.conv_input] + self.conv1 + self.conv2 + self.conv3 + self.conv4 + [self.extra_conv]

    def all_layers(self):
        return [l for seq in self.sequences() for l in seq[:2]]

    def init_weight(self, seed=0, device="cuda", randomize_bn=False):
        rng = np.random.default_rng(seed)
        for l in self.all_layers():
            if isinstance(l, sp.BatchNorm):
                l.init_parameters(rng, device, randomize=randomize_bn)
            else:
                l.init_parameters(rng, device)
        return self

    def set_precision(self, precision):
        for l in self.all_layers():
            if not isinstance(l, sp.BatchNorm):
                l.precision = precision
        return self

    def forward(self, voxel_features, coors, batch_size, num=None):
        x = sp.sparse_coo_tensor(coors, voxel_features, [batch_size] + self.sparse_shape + [self.in_channels], num=num)

        def run(seqs, t):
            for seq in seqs:
                for l in seq:
                    t = l(t)
            return t

        x = run([self.conv_input], x)
        x1 = run(self.conv1, x)
        x2 = run(self.conv2, x1)
        x3 = run(self.conv3, x2)
        x4 = run(self.conv4, x3)
        out = run([self.extra_conv], x4).to_dense_bev()
        return {"spatial_features": out, "spatial_features_stride": 8,
                "multi_scale_3d_features": {"x_conv1": x1, "x_conv2": x2, "x_conv3": x3, "x_conv4": x4},
                "multi_scale_3d_strides": {"x_conv1": 1, "x_conv2": 2, "x_conv3": 4, "x_conv4": 8}}

    __call__ = forward
