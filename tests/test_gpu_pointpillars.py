"""GPU tests of PointPillars (KITTI car): p3d_anchor_head_postprocess against the composed device path it replaces (torch
decode + nms_utils.rotate_nms_pcdet over p3d_nms + direction fix + range filter) and against the numpy restatement, the
trunk + SSD conv against the CPU arm, the whole PointPillarsHotPath frame against the CPU frame, and its eager, graph,
sweep and deploy forms."""
import numpy as np
import pytest

from paddle3d_b200 import anchor_head as ah
from paddle3d_b200 import synth
from parity import rel_check

pytestmark = pytest.mark.gpu

CFG = synth.PP_KITTI_CAR
TC = CFG["test_cfg"]
GAIN = 6.0 ** 0.5


def _head_tensors(cuda, seed, mu, H=248, W=216, A=2, C=1, quant=None):
    import torch
    rng = np.random.default_rng(seed)
    cls = rng.normal(mu, 1.0, (1, A * C, H, W))
    if quant:
        cls = np.round(cls * quant) / quant  # many equal logits: equal scores, ties by ascending anchor index
    box = np.concatenate([rng.normal(0, 0.5, (1, A, 3, H, W)), rng.normal(0, 0.2, (1, A, 3, H, W)),
                          rng.normal(0, 1.0, (1, A, 1, H, W))], 2).reshape(1, 7 * A, H, W)
    dir = rng.normal(0, 1, (1, 2 * A, H, W))
    return [torch.from_numpy(x.astype(np.float32)).to(cuda) for x in (cls, box, dir)]


def _frame_pillars(cuda, seed=2):
    """coors / num_voxels of a frame for the anchor mask: points spread uniformly over the near half of C2's range
    (x < 34.56 m), so that the mask keeps about half of the anchors (55 534 of 107 136 for seed 2) and drops the rest."""
    import torch
    from paddle3d_b200.ops import voxelize as vox
    half = dict(synth.C2, point_cloud_range=[0.0, -39.68, -3.0, 34.56, 39.68, 1.0])
    pts = torch.from_numpy(synth.uniform_cloud(half, seed, num_points=60000, margin=0.0)).to(cuda)
    _, coords, _, nv = vox.hard_voxelize(pts, CFG["voxel_size"], CFG["point_cloud_range"], CFG["max_points"], CFG["max_voxels"])
    return torch.nn.functional.pad(coords, (1, 0), value=0), nv


def _kernel(cls, box, dir, anchors, cells, coors, nv, tc, ny=496, nx=432):
    from paddle3d_b200.ops import anchor_head as oah
    b, s, l, idx, cnt = oah.anchor_head_postprocess_device(
        cls, box, dir, anchors, cells, coors, nv, ny, nx, tc["anchor_area_threshold"], tc["score_threshold"],
        tc["nms_iou_threshold"], tc["nms_pre_max_size"], tc["nms_post_max_size"], tc["post_center_range"])
    k = int(cnt[1])
    return b[:k], s[:k], l[:k], idx[:k].long(), int(cnt[0])


def _composed(cls, box, dir, anchors, keep, tc):
    """The device path the kernel replaces: torch elementwise decode (separate launches, no FMA contraction),
    nms_utils.rotate_nms_pcdet over p3d_nms (with its host syncs), direction fix and range filter."""
    import torch
    from paddle3d_b200.ops import nms_utils
    A = box.shape[1] // 7
    C = cls.shape[1] // A
    H, W = cls.shape[2], cls.shape[3]

    def per_anchor(x, k):
        return x[0].reshape(A, k, H * W).permute(2, 0, 1).reshape(-1, k)
    lg, bt, dt = per_anchor(cls, C), per_anchor(box, 7), per_anchor(dir, 2)
    sig = torch.sigmoid(lg)
    score = sig.amax(1)
    ar = torch.arange(C, device=cls.device).expand_as(sig)
    label = torch.where(sig == score[:, None], ar, C).amin(1)  # first maximal class
    cand = score >= torch.tensor(tc["score_threshold"], dtype=torch.float32)
    if keep is not None:
        cand &= keep
    idx = torch.nonzero(cand).reshape(-1)
    t, an = bt[idx], anchors[idx]
    xa, ya, za, wa, la, ha, ra = [an[:, k] for k in range(7)]
    za = za + ha / 2
    diag = torch.sqrt(la ** 2 + wa ** 2)
    xg = t[:, 0] * diag + xa
    yg = t[:, 1] * diag + ya
    zg = t[:, 2] * ha + za
    wg = torch.exp(t[:, 3]) * wa
    lg_ = torch.exp(t[:, 4]) * la
    hg = torch.exp(t[:, 5]) * ha
    rg = t[:, 6] + ra
    zg = zg - hg / 2
    boxes = torch.stack([xg, yg, zg, wg, lg_, hg, rg], 1)
    if len(idx):
        sel = nms_utils.rotate_nms_pcdet(boxes, score[idx], tc["nms_iou_threshold"], tc["nms_pre_max_size"],
                                         tc["nms_post_max_size"])
    else:
        sel = torch.zeros(0, dtype=torch.long, device=cls.device)
    b = boxes[sel].clone()
    d = dt[idx][sel]
    opp = (b[:, 6] > 0) ^ (d[:, 1] > d[:, 0])
    b[:, 6] = b[:, 6] + torch.where(opp, torch.tensor(np.pi).to(b), torch.tensor(0.0).to(b))
    m = torch.ones(len(b), dtype=torch.bool, device=b.device)
    if tc["post_center_range"] is not None:
        r = torch.tensor(tc["post_center_range"], dtype=torch.float32, device=b.device)
        m = (b[:, :3] >= r[:3]).all(1) & (b[:, :3] <= r[3:]).all(1)
    s = sel[m]
    return b[m], score[idx][s], label[idx][s].long(), idx[s], len(idx)


def _race(cuda, h, anchors, cells, coors, nv, tc, ny=496, nx=432):
    import torch
    keep = None
    if cells is not None and tc["anchor_area_threshold"] >= 0:
        keep = torch.from_numpy(ah.anchors_area(ah.occupancy(coors.cpu().numpy(), int(nv.item()), ny, nx),
                                                cells.cpu().numpy()) > tc["anchor_area_threshold"]).to(cuda)
    got = _kernel(*h, anchors, cells, coors, nv, tc, ny, nx)
    want = _composed(*h, anchors, keep, tc)
    assert got[4] == want[4], "candidate count"
    for name, g, w in zip(("boxes", "scores", "labels", "anchor index"), got[:4], want[:4]):
        assert g.shape == w.shape and torch.equal(g, w), name
    return got


@pytest.fixture(scope="module")
def car(cuda):
    import torch
    a = ah.create_anchors_3d_stride(**CFG["anchors"])
    cells = ah.anchor_cells(a, CFG["voxel_size"], CFG["point_cloud_range"], (432, 496))
    coors, nv = _frame_pillars(cuda)
    return torch.from_numpy(a).to(cuda), torch.from_numpy(cells).to(cuda), coors, nv


@pytest.mark.parametrize("mu,quant,mask,rng,what", [
    (-5.54, None, True, True, "a few hundred candidates, mask and range on"),
    (-4.5, None, True, True, "about 3000 (the top-1000 cut)"),
    (-4.5, None, False, True, "about 6000, mask off"),
    (-4.5, None, True, False, "about 3000, range off"),
    (-30.0, None, True, True, "none"),
    (6.0, None, False, True, "all 107 136 anchors"),
    (-4.5, 4, True, True, "quantised logits: score ties"),
])
def test_kernel_matches_composed_path(cuda, car, mu, quant, mask, rng, what):
    anchors, cells, coors, nv = car
    h = _head_tensors(cuda, 7, mu, quant=quant)
    tc = dict(TC, anchor_area_threshold=TC["anchor_area_threshold"] if mask else -1,
              post_center_range=TC["post_center_range"] if rng else None)
    b, s, l, idx, ncand = _race(cuda, h, anchors, cells if mask else None, coors, nv, tc)
    if mu < -20:
        assert ncand == 0 and len(b) == 0  # no fake row
    if mu > 5:
        assert ncand == 107136 and len(b) > 0
    if mu == -4.5 and quant is None:
        assert ncand > TC["nms_pre_max_size"]
    print("%s: %d candidates, %d boxes" % (what, ncand, len(b)))


def test_kernel_matches_composed_path_multiclass(cuda):
    """A = 6 (3 sizes x 2 rotations), C = 3 on a 20 x 24 map, no mask, range on."""
    import torch
    an = ah.create_anchors_3d_stride((20, 24), (1.6, 3.9, 1.56, 0.6, 0.8, 1.73, 0.6, 1.76, 1.73), (0.32, 0.32, 0.0),
                                     (0.16, -3.0, -1.0), (0, 1.57))
    h = _head_tensors(cuda, 9, -2.0, H=20, W=24, A=6, C=3)
    tc = dict(TC, anchor_area_threshold=-1, nms_pre_max_size=300, nms_post_max_size=50)
    b, s, l, idx, ncand = _race(cuda, h, torch.from_numpy(an).to(cuda), None, None, None, tc)
    assert ncand > 300 and set(l.tolist()) == {0, 1, 2}


def test_kernel_matches_numpy_restatement(cuda, oracle_mod, car):
    """Logits quantised so that numpy's and the device's sigmoid rank the candidates identically: order and labels exact,
    boxes and scores within the parity tolerance."""
    from cpu_pointpillars_frame import anchor_postprocess_np
    anchors, cells, coors, nv = car
    for mu, mask in ((-4.5, True), (-5.54, False)):
        h = _head_tensors(cuda, 11, mu, quant=16)
        tc = dict(TC, anchor_area_threshold=TC["anchor_area_threshold"] if mask else -1)
        b, s, l, idx, ncand = _kernel(*h, anchors, cells if mask else None, coors, nv, tc)
        hn = [t.cpu().numpy() for t in h]
        r = anchor_postprocess_np(*hn, anchors.cpu().numpy(), cells.cpu().numpy() if mask else None, coors.cpu().numpy(),
                                  int(nv.item()), 496, 432, tc["anchor_area_threshold"], tc["score_threshold"],
                                  tc["nms_iou_threshold"], tc["nms_pre_max_size"], tc["nms_post_max_size"],
                                  tc["post_center_range"], oracle_mod.nms)
        assert ncand == r["candidates"]
        np.testing.assert_array_equal(idx.cpu().numpy(), r["index"])
        np.testing.assert_array_equal(l.cpu().numpy(), r["labels"])
        rel_check("anchor postprocess boxes", b.cpu().numpy(), r["boxes"])
        rel_check("anchor postprocess scores", s.cpu().numpy(), r["scores"])


def test_trunk_and_ssd_conv_match_cpu(cuda, oracle_mod):
    """SecondRPN (1x1, k = s = 2 and 4 transposed deblocks, 384-channel concat) + the 20-plane SSD conv on a 64 x 64 x 64
    input against the CPU arm, the bar of test_pillar_dense_head_matches_cpu_head; the pixel-image path equals NCHW."""
    import torch
    from cpu_pointpillars_frame import CpuPointPillarsFrame
    from paddle3d_b200.dense_head import SecondRPN
    from paddle3d_b200.ops import dense_conv as dc
    rpn = SecondRPN(**CFG["backbone"]).init_weight(seed=2, device=cuda, bn_gain=GAIN)
    ssd = ah.SSDHead(rpn.fpn_channels, 1, dict(CFG["anchors"], feature_size=(32, 32))).init_weight(seed=3, device=cuda)
    x = np.maximum(np.random.default_rng(0).normal(size=(1, 64, 64, 64)), 0).astype(np.float32)
    xt = torch.from_numpy(x).to(cuda)
    got = ssd(*rpn(xt))
    g16 = ssd(*rpn(dc.nchw_to_pixel_h16(xt), (1, 64, 64, 64)))
    torch.cuda.synchronize()
    cpu = CpuPointPillarsFrame(CFG, dict(dense=rpn.export_numpy(), ssd=ssd.export_numpy(), pfn=None), TC, None)
    want = cpu.head(x)
    assert want.shape == (1, 20, 32, 32)
    w = [want[:, :2], want[:, 2:16], want[:, 16:]]
    for g, gg, wv in zip(got, g16, w):
        assert g.shape == wv.shape
        assert np.abs(g.cpu().numpy() - wv).max() <= 1e-4 * max(1.0, np.abs(wv).max())
        assert torch.equal(g, gg)


def _pipe(cuda, **kw):
    from paddle3d_b200.ops import sparse_nn as sp
    from paddle3d_b200.pipeline import PointPillarsHotPath
    sp.status_tensor(cuda).zero_()  # the device's status word is sticky: start these frames from a clean one
    return PointPillarsHotPath(CFG, cuda, seed=3, **kw)


def test_frame_matches_cpu_frame(cuda, oracle_mod):
    """Full-size C2 cloud: voxel count, canvas, head planes (CPU head on the GPU's canvas) and the post-processing of the
    GPU's own planes (numpy restatement: keep order and labels exact, boxes within tolerance)."""
    import torch
    from cpu_pointpillars_frame import CpuPointPillarsFrame
    pipe = _pipe(cuda)
    pts = synth.lidar_cloud(synth.C2, 11)
    pipe.calibrate_head(torch.from_numpy(pts).to(cuda))
    pipe.points.copy_(torch.from_numpy(pts).to(cuda))
    with torch.cuda.stream(pipe.stream):
        out = pipe.forward_device()
    pipe.stream.synchronize()
    pipe.out = out
    pipe.check_status(out["status"].cpu())
    cpu = CpuPointPillarsFrame(CFG, pipe.export_weights_numpy(), pipe.test_cfg, pipe.ssd.cells)
    ref = cpu.run(pts, head=False)
    assert int(out["num_voxels"][0].item()) == ref["num_voxels"]
    bev = pipe.bev_nchw().cpu().numpy()
    assert bev.shape == ref["bev"].shape == (1, 64, 496, 432)
    rel_check("pointpillars frame canvas", bev, ref["bev"])
    planes = cpu.head(bev)
    h = out["head"]
    got = np.concatenate([h["cls"].cpu().numpy(), h["box"].cpu().numpy(), h["dir"].cpu().numpy()], 1)
    assert got.shape == planes.shape == (1, 20, 248, 216)
    assert np.abs(got - planes).max() <= 1e-4 * max(1.0, np.abs(planes).max())
    r = cpu.postprocess(got, ref["coors"], ref["num_voxels"])
    counts = out["counts"].cpu().numpy()
    k = int(counts[1])
    print("pointpillars frame: %d pillars, %d candidates, %d boxes" % (ref["num_voxels"], counts[0], k))
    assert counts[0] == r["candidates"] > TC["nms_pre_max_size"] and k == len(r["index"]) > 0
    np.testing.assert_array_equal(out["anchor_index"][:k].cpu().numpy(), r["index"])
    np.testing.assert_array_equal(out["labels"][:k].cpu().numpy(), r["labels"])
    rel_check("pointpillars frame boxes", out["boxes"][:k].cpu().numpy(), r["boxes"])
    rel_check("pointpillars frame scores", out["scores"][:k].cpu().numpy(), r["scores"])


def _same(a, b):
    import torch
    return all(torch.equal(x, y) for x, y in zip(a, b))


def test_graph_sweep_lanes_and_predictor_are_bit_identical(cuda):
    import torch
    from paddle3d_b200 import deploy
    from paddle3d_b200.pipeline import CenterPointSweep, PointPillarsHotPath
    frames = [torch.from_numpy(synth.lidar_cloud(synth.C2, 20 + i)).pin_memory() for i in range(4)]
    kw = dict(cfg=CFG, device=cuda, seed=3)
    eager = _pipe(cuda)
    eager.calibrate_head(frames[0].to(cuda))
    want = [tuple(t.clone() for t in eager.infer(f)) for f in frames]
    assert all(w[0].shape[1] == 7 for w in want) and len(want[0][2]) > 10
    assert len({len(w[2]) for w in want}) > 1 or not _same(want[0], want[1])  # the frames differ
    graph = _pipe(cuda)
    graph.ssd = eager.ssd  # calibrated biases
    graph.points.copy_(frames[0])
    graph.capture(count_nodes=True)  # a host synchronisation inside the frame would fail the capture
    for f, w in zip(frames, want):
        assert _same(graph.infer(f), w)
    got = list(graph.infer_many(iter(frames)))
    assert len(got) == len(want) and all(_same(g, w) for g, w in zip(got, want))
    sweep = CenterPointSweep(2, pipeline_cls=PointPillarsHotPath, **kw)
    assert sweep.lanes[1].ssd is sweep.lanes[0].ssd and sweep.lanes[1].dense is sweep.lanes[0].dense
    sweep.calibrate_head(frames[0].to(cuda))
    sweep.capture(frames[0].to(cuda))
    got = list(sweep.infer_many(iter(frames)))
    assert len(got) == len(want) and all(_same(g, w) for g, w in zip(got, want))
    print("pointpillars frame graph nodes: %s" % graph.graph_nodes)
    # deploy: a Predictor defaults to the car configuration; uncalibrated seeded weights, compared with a pipeline
    N = 30000
    pts = synth.lidar_cloud(synth.C2, 21)
    pred = deploy.Predictor(device=cuda, max_points=N, seed=3, pipeline_cls=PointPillarsHotPath)
    assert pred.cfg["name"] == "pointpillars_kitti_car"
    b, l, s = pred.run(pts)
    ref = _pipe(cuda, num_points=N)
    full = np.full((N, 4), np.nan, np.float32)
    full[:len(pts)] = pts
    rb, rs, rl = ref.infer(torch.from_numpy(full).pin_memory())
    assert np.array_equal(b, rb.numpy()) and np.array_equal(l, rl.numpy()) and np.array_equal(s, rs.numpy())
    assert b.shape[1] == 7 and all(line.count(" ") >= 10 for line in deploy.format_result(b, l, s))
