"""CenterPoint-pillars without a GPU: the geometry of the pillar dense head (down-sampling SecondFPN deblock), the CPU
frame at a tiny size, the configurations PillarFeatureNet refuses, and the host-side validation of the fused pillar
encoder entry point (every call below is rejected before any CUDA call)."""
import ctypes as C

import numpy as np
import pytest

from paddle3d_b200 import synth


def _pillar_head():
    from paddle3d_b200.dense_head import DenseRPNHead
    return DenseRPNHead(**synth.CP_PILLARS["backbone"]).init_weight(seed=1, device=None)


def _sizes(head, H, W):
    """Output size of every backbone block and of every deblock for an H x W input."""
    blocks, h, w = [], H, W
    for blk in head.blocks:
        for c in blk:
            h, w = (h + 2 * c.padding - c.k) // c.stride + 1, (w + 2 * c.padding - c.k) // c.stride + 1
        blocks.append((h, w))
    return blocks, [head.deblock_out_hw(de, h, w) for (h, w), de in zip(blocks, head.deblocks)]


def test_pillar_head_geometry():
    head = _pillar_head()
    d0, d1, d2 = head.deblocks
    assert (d0.k, d0.stride, d0.up, d0.cin, d0.cout) == (2, 2, 1, 64, 128)   # upsample_strides 0.5: Conv2D k = s = 2
    assert (d1.k, d1.stride, d1.up, d1.cin, d1.cout) == (1, 1, 1, 128, 128)
    assert (d2.k, d2.stride, d2.up, d2.cin, d2.cout) == (2, 2, 2, 256, 128)  # Conv2DTranspose k = s = 2
    blocks, de = _sizes(head, 512, 512)
    assert blocks == [(256, 256), (128, 128), (64, 64)]
    assert de == [(128, 128)] * 3
    assert head.fpn_channels == 384 and head.shared.cin == 384
    assert [len(b) for b in head.blocks] == [4, 6, 6]
    w = head.export_numpy()["deblocks"][0]
    assert w["weight"].shape == (128, 64, 2, 2) and (w["stride"], w["padding"], w["up"]) == (2, 0, 1)


def test_voxel_head_geometry_unchanged():
    from paddle3d_b200.dense_head import DenseRPNHead
    head = DenseRPNHead(in_channels=256).init_weight(seed=1, device=None)
    d0, d1 = head.deblocks
    assert (d0.k, d0.stride, d0.up) == (1, 1, 1) and (d1.k, d1.stride, d1.up) == (2, 2, 2)
    assert _sizes(head, 180, 180)[1] == [(180, 180)] * 2


def test_mismatched_deblock_sizes_raise():
    """upsample_strides that do not bring every level to one size cannot be concatenated."""
    from paddle3d_b200.dense_head import DenseRPNHead
    shapes = [(1, 32, 32, 64), (1, 16, 16, 128), (1, 8, 8, 256)]
    assert _pillar_head().fpn_out_hw(shapes) == (16, 16)
    head = DenseRPNHead(**dict(synth.CP_PILLARS["backbone"], upsample_strides=(1, 1, 2))).init_weight(seed=1, device=None)
    with pytest.raises(ValueError, match="different sizes"):
        head.fpn_out_hw(shapes)


def test_cpu_head_shapes_at_small_size(oracle_mod):
    from oracle.cpu_reference import CpuDenseHead
    head = _pillar_head()
    x = np.random.default_rng(0).normal(size=(1, 64, 32, 32)).astype(np.float32)
    out = CpuDenseHead(head.export_numpy()).run(x)
    assert sorted(out) == ["dim", "height", "hm", "reg", "rot", "vel"]
    assert [o.shape for o in out["hm"]] == [(1, c, 8, 8) for c in synth.CENTERPOINT_TASKS]
    for name, c in (("reg", 2), ("height", 1), ("dim", 3), ("rot", 2), ("vel", 2)):
        assert all(o.shape == (1, c, 8, 8) for o in out[name]), name


def test_pillar_feature_net_rejects_unsupported_configs():
    from paddle3d_b200.layers import PillarFeatureNet
    with pytest.raises(ValueError):
        PillarFeatureNet(5, (64, 64))
    with pytest.raises(ValueError):
        PillarFeatureNet(5, (64,), with_distance=True)
    net = PillarFeatureNet(5, [64], False, 20, [0.2, 0.2, 8], [-51.2, -51.2, -5, 51.2, 51.2, 3], legacy=False)
    net.init_weight(seed=0, device=None, bn_gain=2.0)
    assert net.np["weight"].shape == (10, 64) and float(net.np["gamma"][0]) == 2.0 and net.weight is None


def test_fused_pillar_encoder_argument_checks():
    from paddle3d_b200 import _lib
    L = _lib.lib()
    f = L.p3d_pillar_feature_net_pixel_h16
    p = C.c_void_p(256)    # non-null, 16-byte aligned dummy address: the checks below fail before it is touched
    odd = C.c_void_p(260)  # misaligned for the 16-byte checks
    vs, pcr = _lib.host_floats([0.2, 0.2, 8]), _lib.host_floats([-51.2, -51.2, -5, 51.2, 51.2, 3])

    def call(voxels=p, coors=p, n=10, M=20, F=5, Cc=64, weight=p, batch=1, ny=8, nx=8, out=p):
        return f(voxels, p, coors, None, n, M, F, Cc, weight, p, p, vs, pcr, batch, ny, nx, out, None, None)

    assert call(out=None) == -1
    assert call(weight=None) == -1
    assert call(voxels=None) == -1
    assert call(coors=odd) == -1
    assert call(out=odd) == -1
    assert call(batch=0) == -1
    assert call(Cc=0) == -1
    assert call(M=65) == -4
    assert call(F=9) == -4
    assert call(Cc=48) == -4
    assert f(p, p, p, None, 10, 20, 5, 64, p, p, p, None, pcr, 1, 8, 8, p, None, None) == -1  # voxel size


def test_cpu_pillar_frame_tiny(oracle_mod):
    """The CPU pillar frame runs end to end at a 32 x 32 grid: voxelizer, PFN, scatter, dense head, postprocess."""
    from cpu_pillar_frame import CpuPillarFrame
    from paddle3d_b200.layers import PillarFeatureNet
    cfg = dict(synth.CP_PILLARS, point_cloud_range=[-3.2, -3.2, -5.0, 3.2, 3.2, 3.0], num_points=2000, max_voxels=1024)
    net = PillarFeatureNet(5, (64,), False, cfg["max_points"], cfg["voxel_size"], cfg["point_cloud_range"])
    net.init_weight(seed=0, device=None, bn_gain=6.0 ** 0.5)
    weights = dict(pfn=net.np, dense=_pillar_head().export_numpy())
    pts = synth.lidar_cloud(dict(cfg, point_cloud_range=[-8, -8, -5, 8, 8, 3]), 3, num_points=cfg["num_points"])
    r = CpuPillarFrame(cfg, weights, synth.CP_PILLARS_TEST_CFG, synth.label_offsets(), use_ref_voxelizer=False).run(pts)
    assert 0 < r["num_voxels"] <= 1024
    assert r["bev"].shape == (1, 64, 32, 32)
    assert (r["bev"].reshape(64, -1).any(0)).sum() == r["num_voxels"]  # one occupied cell per pillar (ReLU(BN) > 0 here)
    assert r["head"]["hm"][0].shape == (1, 1, 8, 8)
    assert r["boxes"].shape[1] == 9 and len(r["boxes"]) == len(r["scores"]) == len(r["labels"]) >= len(synth.CENTERPOINT_TASKS)
