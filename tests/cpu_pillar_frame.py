"""CPU arm of the CenterPoint-pillars frame for the tests: chains the oracle's existing functions (oracle/ stays the
fixed yardstick of the suite, so the pillar frame that composes them lives here, beside the tests that use it)."""
import time

import numpy as np

from oracle.cpu_reference import CpuDenseHead


class CpuPillarFrame:
    """CPU arm of the CenterPoint-pillars frame (pipeline.CenterPointPillarsHotPath) through the oracle: the reference's
    CPU voxelizer (oracle.hard_voxelize when oracle/_ref was not built), PillarFeatureNet, PointPillarsScatter, the dense
    RPN / neck / CenterHead (CpuDenseHead) and centerpoint_postprocess.  weights: export_weights_numpy() of the pipeline."""

    def __init__(self, cfg, weights, test_cfg, label_offsets, use_ref_voxelizer=True):
        import oracle
        self.o = oracle
        self.cfg, self.w, self.tc, self.off = cfg, weights, test_cfg, label_offsets
        self.dense = CpuDenseHead(weights["dense"])
        self.use_ref = use_ref_voxelizer and oracle.ref_lib("cpu") is not None
        g = oracle.grid_size(cfg["voxel_size"], cfg["point_cloud_range"])
        self.nx, self.ny = g[0], g[1]

    def run(self, points):
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
        t0 = time.perf_counter()
        h = self.dense.run(bev)
        t["dense_head"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        tc = self.tc
        boxes, scores, labels, _ = o.centerpoint_postprocess(
            h["hm"], h["reg"], h["height"], h["dim"], h["vel"], h["rot"], cfg["voxel_size"][:2], cfg["point_cloud_range"],
            tc["post_center_limit_range"], self.off, tc["down_ratio"], tc["score_threshold"], tc["nms_iou_threshold"],
            tc["nms_pre_max_size"], tc["nms_post_max_size"], True)
        t["postprocess"] = time.perf_counter() - t0
        return dict(bev=bev, boxes=boxes, scores=scores, labels=labels, times=t, num_voxels=k, head=h)
