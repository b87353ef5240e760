"""CPU arm of the PointPillars frame for the tests (pipeline.PointPillarsHotPath): chains the oracle's existing functions -
voxelizer, pillar_feature_net, pillar_scatter, conv2d / deconv2d / bn2d_relu (through CpuDenseHead's layer helper) and the
rotated NMS - and adds a numpy restatement of the SSD head's post-processing (anchor_postprocess_np).  oracle/ stays the
fixed yardstick of the suite, so the frame that composes it lives here, beside the tests that use it."""
import time

import numpy as np

from oracle.cpu_reference import CpuDenseHead
from paddle3d_b200 import anchor_head as ah

F32 = np.float32


def decode_np(t, an):
    """second_box_decode in fp32, operation by operation (numpy does not contract into FMAs)."""
    xa, ya, za, wa, la, ha, ra = [an[:, k] for k in range(7)]
    xt, yt, zt, wt, lt, ht, rt = [t[:, k] for k in range(7)]
    za = za + ha / F32(2)
    diag = np.sqrt(la * la + wa * wa)
    xg = xt * diag + xa
    yg = yt * diag + ya
    zg = zt * ha + za
    wg = np.exp(wt) * wa
    lg = np.exp(lt) * la
    hg = np.exp(ht) * ha
    rg = rt + ra
    zg = zg - hg / F32(2)
    return np.stack([xg, yg, zg, wg, lg, hg, rg], 1).astype(F32)


def anchor_postprocess_np(cls, box, dir, anchors, cells, coors, num_voxels, ny, nx, area_thr, score_thr, iou_thr, pre_max,
                          post_max, post_center_range, nms_fn):
    """Restatement of steps 1-8 of csrc/anchor_postprocess.cu (SECOND's predict + rotate_nms_pcdet, batch 1).  cls / box /
    dir: NCHW fp32 numpy planes; nms_fn(boxes [n, 7], thr) -> (keep, num_keep) (oracle.nms).  Returns dict(boxes, scores,
    labels, index, candidates)."""
    A = box.shape[1] // 7
    C = cls.shape[1] // A
    H, W = cls.shape[2], cls.shape[3]

    def per_anchor(x, k):  # [1, A * k, H, W] -> [H * W * A, k], anchor (y * W + x) * A + a
        return np.ascontiguousarray(x[0].reshape(A, k, H * W).transpose(2, 0, 1).reshape(-1, k))
    lg, bt, dt = per_anchor(cls, C), per_anchor(box, 7), per_anchor(dir, 2)
    keep = np.ones(len(lg), bool)
    if cells is not None and area_thr >= 0:                                      # 1. anchor mask
        keep = ah.anchors_area(ah.occupancy(coors, num_voxels, ny, nx), cells) > area_thr
    with np.errstate(over="ignore"):                                             # 2. scores (first max wins)
        sig = (F32(1) / (F32(1) + np.exp(-lg))).astype(F32)
    label = sig.argmax(1)
    score = sig.max(1)
    idx = np.nonzero(keep & (score >= F32(score_thr)))[0]
    order = idx[np.argsort(-score[idx], kind="stable")][:pre_max]                # 4. descending, ties ascending index
    boxes = decode_np(bt[order], anchors[order])                                 # 3. decode
    nb = boxes[:, [0, 1, 2, 4, 3, 5, 6]].copy()                                  # 5. rotate_nms_pcdet's layout
    nb[:, 6] = -nb[:, 6] - F32(np.pi / 2)
    k, nk = nms_fn(nb, iou_thr) if len(nb) else (np.zeros(0, np.int32), 0)
    sel = np.asarray(k[:nk][:post_max], np.int64)
    b = boxes[sel].copy()
    dl = dt[order[sel]].argmax(1)                                                # 6. direction fix
    flip = (b[:, 6] > 0) ^ (dl != 0)
    b[flip, 6] = b[flip, 6] + F32(np.pi)
    m = np.ones(len(b), bool)
    if post_center_range is not None:                                            # 7. range filter
        r = np.asarray(post_center_range, F32)
        m = (b[:, :3] >= r[:3]).all(1) & (b[:, :3] <= r[3:]).all(1)
    s = sel[m]
    return dict(boxes=b[m], scores=score[order[s]], labels=label[order[s]].astype(np.int64), index=order[s],
                candidates=len(idx))


class CpuPointPillarsFrame:
    """CPU arm of pipeline.PointPillarsHotPath through the oracle.  weights: export_weights_numpy() of the pipeline."""

    def __init__(self, cfg, weights, test_cfg, cells, use_ref_voxelizer=True):
        import oracle
        self.o = oracle
        self.cfg, self.w, self.tc, self.cells = cfg, weights, test_cfg, cells
        self.layers = CpuDenseHead(weights["dense"])
        self.use_ref = use_ref_voxelizer and oracle.ref_lib("cpu") is not None
        g = oracle.grid_size(cfg["voxel_size"], cfg["point_cloud_range"])
        self.nx, self.ny = g[0], g[1]

    def head(self, bev):
        """SecondBackbone + SecondFPN + the SSD conv: [1, A * (C + 9), H, W] fp32 planes."""
        w, x, feats = self.w["dense"], bev, []
        for blk in w["blocks"]:
            for l in blk:
                x = self.layers._conv(l, x)
            feats.append(x)
        cat = np.concatenate([self.layers._conv(l, f) for l, f in zip(w["deblocks"], feats)], axis=1)
        c = self.w["ssd"]["conv"]
        return self.o.conv2d(cat, c["weight"], c["bias"], 1, 0)

    def run(self, points, head=True):
        """head=False: voxelizer and canvas only (a test can run the head on another canvas)."""
        cfg, o, p = self.cfg, self.o, self.w["pfn"]
        t = {}
        t0 = time.perf_counter()
        vox = o.ref_hard_voxelize_cpu if self.use_ref else o.hard_voxelize
        v, c, n, nv = vox(points, cfg["voxel_size"], cfg["point_cloud_range"], cfg["max_points"], cfg["max_voxels"])
        k = int(nv[0])
        coors = np.concatenate([np.zeros((k, 1), np.int32), c[:k]], 1)
        t["voxelize"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        feats = o.pillar_feature_net(v[:k], n[:k], coors, p["weight"], p["gamma"], p["beta"], p["mean"], p["var"], p["eps"],
                                     cfg["voxel_size"], cfg["point_cloud_range"])
        bev = o.pillar_scatter(feats, coors, 1, self.ny, self.nx)
        t["pillar_encoder"] = time.perf_counter() - t0
        if not head:
            return dict(bev=bev, num_voxels=k, coors=coors, times=t)
        t0 = time.perf_counter()
        planes = self.head(bev)
        t["trunk_and_ssd_conv"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        r = self.postprocess(planes, coors, k)
        t["postprocess"] = time.perf_counter() - t0
        r.update(bev=bev, planes=planes, num_voxels=k, coors=coors, times=t)
        return r

    def postprocess(self, planes, coors, num_voxels):
        s, tc = self.w["ssd"], self.tc
        A, C = s["num_anchors"], s["num_classes"]
        cls, box, dir = planes[:, :A * C], planes[:, A * C:A * (C + 7)], planes[:, A * (C + 7):]
        return anchor_postprocess_np(cls, box, dir, s["anchors"], self.cells, coors, num_voxels, self.ny, self.nx,
                                     tc["anchor_area_threshold"], tc["score_threshold"], tc["nms_iou_threshold"],
                                     tc["nms_pre_max_size"], tc["nms_post_max_size"], tc["post_center_range"], self.o.nms)
