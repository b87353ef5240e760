"""GPU tests of CenterPoint-pillars: the fused pillar encoder (p3d_pillar_feature_net_pixel_h16) against the three-launch
chain it replaces and against the oracle, the pillar dense head (down-sampling SecondFPN deblock) against the CPU head,
and the whole CenterPointPillarsHotPath frame against the CPU pillar frame, in its eager, graph, sweep and deploy forms."""
import numpy as np
import pytest

from paddle3d_b200 import synth
from parity import rel_check

pytestmark = pytest.mark.gpu

GAIN = 6.0 ** 0.5
SMALL = dict(synth.CP_PILLARS, point_cloud_range=[-12.8, -12.8, -5.0, 12.8, 12.8, 3.0], num_points=20000)  # 128 x 128


def _voxelize(cuda, cfg, pts, P, V):
    import torch
    from paddle3d_b200.ops import voxelize as vox
    voxels, coords, npv, nv = vox.hard_voxelize(torch.from_numpy(pts).to(cuda), cfg["voxel_size"], cfg["point_cloud_range"],
                                                P, V)
    coors = torch.nn.functional.pad(coords, (1, 0), value=0)
    return voxels, npv, coors, nv


def _pfn(cuda, cfg, F, P, seed=0, gain=GAIN):
    from paddle3d_b200.layers import PillarFeatureNet
    return PillarFeatureNet(F, (64,), False, P, cfg["voxel_size"], cfg["point_cloud_range"]).init_weight(seed, cuda, gain)


def _grid(cfg):
    from paddle3d_b200.layers import _grid
    g = _grid(cfg["point_cloud_range"], cfg["voxel_size"])
    return int(g[1]), int(g[0])  # ny, nx


def _chain(net, voxels, npv, coors, nv, batch, ny, nx):
    """The three launches the fused kernel replaces: rows, fp32 NCHW canvas, pixel fp16-pair image."""
    from paddle3d_b200.ops import dense_conv as dc
    from paddle3d_b200.ops import pillar_scatter as ps
    return dc.nchw_to_pixel_h16(ps.pillar_scatter(net(voxels, npv, coors, num=nv), coors, batch, ny, nx, num=nv))


def _compare(cuda, oracle_mod, cfg, pts, P, V, batch=1, split=False):
    import torch
    from paddle3d_b200.ops import dense_conv as dc
    F = pts.shape[1]
    voxels, npv, coors, nv = _voxelize(cuda, cfg, pts, P, V)
    k = int(nv.item())
    if split:
        coors[k // 2:k, 0] = 1
    net = _pfn(cuda, cfg, F, P)
    ny, nx = _grid(cfg)
    img, shape = net.forward_pixel_h16(voxels, npv, coors, batch, ny, nx, num=nv)
    want = _chain(net, voxels, npv, coors, nv, batch, ny, nx)
    assert shape == (batch, ny, nx, 64) and img.shape == want.shape
    assert torch.equal(img, want)
    c = coors.cpu().numpy()[:k]
    p = net.np
    feats = oracle_mod.pillar_feature_net(voxels.cpu().numpy()[:k], npv.cpu().numpy()[:k], c, p["weight"], p["gamma"], p["beta"],
                                          p["mean"], p["var"], p["eps"], cfg["voxel_size"], cfg["point_cloud_range"])
    rel_check("pillar image %s b%d" % (cfg["name"], batch), dc.pixel_h16_to_nchw(img, shape).cpu().numpy(),
              oracle_mod.pillar_scatter(feats, c, batch, ny, nx))
    return k


def test_fused_encoder_full_size_frame(cuda, oracle_mod):
    cfg = synth.CP_PILLARS
    k = _compare(cuda, oracle_mod, cfg, synth.lidar_cloud(cfg, 1), cfg["max_points"], cfg["max_voxels"])
    assert k > 1000


def test_fused_encoder_c2_geometry_and_batch_of_two(cuda, oracle_mod):
    cfg = synth.C2  # F = 4, P = 32, 496 x 432
    pts = synth.lidar_cloud(cfg, 2)
    assert _grid(cfg) == (496, 432)
    _compare(cuda, oracle_mod, cfg, pts, 32, 12000)
    _compare(cuda, oracle_mod, cfg, pts, 32, 12000, batch=2, split=True)


def test_fused_encoder_edge_cases(cuda):
    import torch
    from paddle3d_b200.ops import sparse_nn as sp
    cfg = synth.C2
    P, V = 32, 3000
    voxels, npv, coors, nv = _voxelize(cuda, cfg, synth.lidar_cloud(cfg, 5, num_points=6000), P, V)
    net = _pfn(cuda, cfg, 4, P)
    ny, nx = _grid(cfg)
    # no pillars: an all-zero image
    zero = torch.zeros_like(nv)
    img, _ = net.forward_pixel_h16(voxels, npv, coors, 1, ny, nx, num=zero)
    assert not img.any()
    # rows outside the grid and rows of a batch index >= batch are skipped, like the scatter skips them
    k = int(nv.item())
    bad = coors.clone()
    bad[0, 3], bad[1, 2], bad[2, 3], bad[3, 0], bad[4, 0] = nx, ny, -1, 1, -1
    img, _ = net.forward_pixel_h16(voxels, npv, bad, 1, ny, nx, num=nv)
    assert torch.equal(img, _chain(net, voxels, npv, bad, nv, 1, ny, nx))
    good, _ = net.forward_pixel_h16(voxels[5:], npv[5:], coors[5:].contiguous(), 1, ny, nx, num=nv - 5)
    assert torch.equal(img, good)
    occupied = img.view(ny * nx, -1).any(1).sum().item()
    assert 0 < occupied <= k - 5
    # values above fp16's range: saturated to 65504 and bit 0 of the status word set
    st = sp.status_tensor(cuda)
    st.zero_()
    img, _ = net.forward_pixel_h16(voxels, npv, coors, 1, ny, nx, num=nv)
    torch.cuda.synchronize()
    assert int(st.item()) == 0
    big = _pfn(cuda, cfg, 4, P, gain=GAIN * 1e6)
    img, _ = big.forward_pixel_h16(voxels, npv, coors, 1, ny, nx, num=nv)
    torch.cuda.synchronize()
    assert int(st.item()) & 1
    hi = img.view(ny * nx, 2, 2, 32)[:, :, 0].float()  # [pixel][group][hi 32]
    assert float(hi.max()) == 65504.0
    st.zero_()


def test_pillar_dense_head_matches_cpu_head(cuda, oracle_mod):
    """The pillar head (k2 s2 down-sampling deblock, 1x1 and transposed deblocks, 384-channel concat) on a 64 x 64 x 64
    input against the CPU head, the bar of test_frame_with_dense_head; forward_h16 on the pixel image equals forward."""
    import torch
    from oracle.cpu_reference import CpuDenseHead
    from paddle3d_b200.dense_head import DenseRPNHead
    from paddle3d_b200.ops import dense_conv as dc
    head = DenseRPNHead(**synth.CP_PILLARS["backbone"]).init_weight(seed=2, device=cuda, bn_gain=GAIN)
    x = np.maximum(np.random.default_rng(0).normal(size=(1, 64, 64, 64)), 0).astype(np.float32)
    xt = torch.from_numpy(x).to(cuda)
    got = head(xt)
    h16 = head.forward_h16(dc.nchw_to_pixel_h16(xt), (1, 64, 64, 64))
    torch.cuda.synchronize()
    want = CpuDenseHead(head.export_numpy()).run(x)
    for name in want:
        for g, g16, w in zip(got[name], h16[name], want[name]):
            assert g.shape == (1, w.shape[1], 16, 16)
            assert np.abs(g.cpu().numpy() - w).max() <= 1e-4 * max(1.0, np.abs(w).max()), name
            assert torch.equal(g, g16), name


def _pipe(cuda, cfg=SMALL, **kw):
    from paddle3d_b200.ops import sparse_nn as sp
    from paddle3d_b200.pipeline import CenterPointPillarsHotPath
    sp.status_tensor(cuda).zero_()  # the device's status word is sticky: start these frames from a clean one
    return CenterPointPillarsHotPath(cfg, cuda, seed=3, **kw)


def test_frame_matches_cpu_pillar_frame(cuda, oracle_mod):
    import torch
    from cpu_pillar_frame import CpuPillarFrame
    from oracle.cpu_reference import CpuDenseHead
    pipe = _pipe(cuda)
    pts = synth.lidar_cloud(SMALL, 11)
    pipe.points.copy_(torch.from_numpy(pts).to(cuda))
    with torch.cuda.stream(pipe.stream):
        out = pipe.forward_device()
    pipe.stream.synchronize()
    pipe.out = out
    w = pipe.export_weights_numpy()
    ref = CpuPillarFrame(SMALL, w, pipe.test_cfg, pipe.label_off).run(pts)
    assert int(out["num_voxels"][0].item()) == ref["num_voxels"]
    bev = pipe.bev_nchw().cpu().numpy()
    assert bev.shape == ref["bev"].shape == (1, 64, 128, 128)
    rel_check("pillar frame canvas", bev, ref["bev"])
    # head tensors: the CPU head on the GPU's own canvas (the canvas itself is checked just above)
    head = {k: [t.cpu().numpy() for t in v] for k, v in out["head"].items()}
    want = CpuDenseHead(w["dense"]).run(bev)
    for name in want:
        for g, wv in zip(head[name], want[name]):
            assert g.shape == wv.shape == (1, wv.shape[1], 32, 32)
            assert np.abs(g - wv).max() <= 1e-4 * max(1.0, np.abs(wv).max()), name
    # postprocess of the GPU's own head tensors against the oracle's on the same tensors
    tc, cfg = pipe.test_cfg, SMALL
    b, s, l, _ = oracle_mod.centerpoint_postprocess(
        head["hm"], head["reg"], head["height"], head["dim"], head["vel"], head["rot"], cfg["voxel_size"][:2],
        cfg["point_cloud_range"], tc["post_center_limit_range"], pipe.label_off, tc["down_ratio"], tc["score_threshold"],
        tc["nms_iou_threshold"], tc["nms_pre_max_size"], tc["nms_post_max_size"], True)
    k = int(out["counts"][-1].item())
    assert k == len(l)
    np.testing.assert_array_equal(out["labels"][:k].cpu().numpy(), l)
    np.testing.assert_allclose(out["scores"][:k].cpu().numpy(), s, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(out["boxes"][:k].cpu().numpy(), b, rtol=1e-4, atol=1e-4)
    assert int(out["status"].item()) == 0


def _same(a, b):
    import torch
    return all(torch.equal(x, y) for x, y in zip(a, b))


def test_graph_sweep_and_lanes_are_bit_identical(cuda):
    import torch
    from paddle3d_b200.ops import sparse_nn as sp
    from paddle3d_b200.pipeline import CenterPointPillarsHotPath, CenterPointSweep
    cfg = synth.CP_PILLARS
    frames = [torch.from_numpy(synth.lidar_cloud(cfg, 20 + i, num_points=100000)).pin_memory() for i in range(4)]
    kw = dict(cfg=cfg, device=cuda, seed=3, num_points=100000)
    sp.status_tensor(cuda).zero_()
    eager = CenterPointPillarsHotPath(**kw)
    eager.calibrate_head(frames[0].to(cuda))
    want = [tuple(t.clone() for t in eager.infer(f)) for f in frames]
    assert len({len(w[2]) for w in want}) > 1 or len(want[0][2]) > 6  # the frames differ / detect something
    graph = CenterPointPillarsHotPath(**kw)
    graph.dense = eager.dense  # calibrated biases
    graph.points.copy_(frames[0])
    graph.capture(count_nodes=True)
    for f, w in zip(frames, want):
        assert _same(graph.infer(f), w)
    got = list(graph.infer_many(iter(frames)))
    assert len(got) == len(want) and all(_same(g, w) for g, w in zip(got, want))
    sweep = CenterPointSweep(2, pipeline_cls=CenterPointPillarsHotPath, **kw)
    assert sweep.lanes[1].net is sweep.lanes[0].net and sweep.lanes[1].dense is sweep.lanes[0].dense
    sweep.calibrate_head(frames[0].to(cuda))
    sweep.capture(frames[0].to(cuda))
    got = list(sweep.infer_many(iter(frames)))
    assert len(got) == len(want) and all(_same(g, w) for g, w in zip(got, want))
    print("pillar frame graph nodes: %s" % graph.graph_nodes)


def test_full_size_frame(cuda):
    import torch
    cfg = synth.CP_PILLARS
    pipe = _pipe(cuda, cfg)
    pts = torch.from_numpy(synth.lidar_cloud(cfg, 0)).pin_memory()
    pipe.calibrate_head(pts.to(cuda))
    pipe.points.copy_(pts)
    pipe.capture()
    boxes, scores, labels = pipe.infer(pts)
    counts = pipe.h_counts.clone()
    assert int(pipe.h_status[0]) == 0
    assert all(int(c) >= 1 for c in counts[:-1]) and int(counts[-1]) == len(labels)
    nv = int(pipe.out["num_voxels"][0].item())
    print("full-size pillar frame: %d occupied pillars of the %d cap (%s), %d boxes" % (
        nv, cfg["max_voxels"], "cap reached" if nv >= cfg["max_voxels"] else "cap not reached", len(labels)))


def test_deploy_predictor_pillars(cuda):
    import torch
    from paddle3d_b200 import deploy
    from paddle3d_b200.pipeline import CenterPointPillarsHotPath
    N = 40000
    pts = synth.lidar_cloud(synth.CP_PILLARS, 21, num_points=30000)
    pred = deploy.Predictor(device=cuda, max_points=N, seed=3, pipeline_cls=CenterPointPillarsHotPath)
    assert pred.cfg["name"] == "centerpoint_pillar_02"
    b, l, s = pred.run(pts)
    ref = _pipe(cuda, synth.CP_PILLARS, num_points=N)
    full = np.full((N, 5), np.nan, np.float32)
    full[:len(pts)] = pts
    rb, rs, rl = ref.infer(torch.from_numpy(full).pin_memory())
    assert np.array_equal(b, rb.numpy()) and np.array_equal(l, rl.numpy()) and np.array_equal(s, rs.numpy())
