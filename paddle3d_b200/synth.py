"""Seeded synthetic inputs for the hot path (numpy only; no datasets exist offline).

Shapes follow SURVEY.md §8 / BASELINE.json configs:
  C1 1k pts (C2 geometry)   C2 PointPillars KITTI 20k x 4   C3 CenterPoint-voxel nuScenes 300k x 5
  C4 bev_pool_v2 (6 cams, 16x44 feature maps, D=118, C=80, 128x128 / 200x200 BEV grid)
Config values cite the reference YAMLs they come from.
"""
import math

import numpy as np

# configs/pointpillars/pointpillars_xyres16_kitti_car.yml:87-108
C2 = dict(name="pointpillars_kitti", num_points=20000, point_dim=4, voxel_size=[0.16, 0.16, 4.0],
          point_cloud_range=[0.0, -39.68, -3.0, 69.12, 39.68, 1.0], max_points=32, max_voxels=40000)
# configs/centerpoint/centerpoint_voxels_0075voxel_nuscenes_10sweep.yml:111-172
C3 = dict(name="centerpoint_voxel_0075", num_points=300000, point_dim=5, voxel_size=[0.075, 0.075, 0.2],
          point_cloud_range=[-54.0, -54.0, -5.0, 54.0, 54.0, 3.0], max_points=10, max_voxels=160000)
# 0.1 m variant named by BASELINE.json.metric: same 1440x1440x40 grid over a 144 m square
C3_01 = dict(name="centerpoint_voxel_01", num_points=300000, point_dim=5, voxel_size=[0.1, 0.1, 0.2],
             point_cloud_range=[-72.0, -72.0, -5.0, 72.0, 72.0, 3.0], max_points=10, max_voxels=160000)
C1 = dict(C2, name="c1_cpu", num_points=1000)
# LiDAR branch of BEVFusion (configs/bevfusion/bevf_pp_2x8_1x_nusc.yaml:87-105): 0.25 m pillars on a 400 x 400 grid
C4_LIDAR = dict(name="bevfusion_lidar_pillars", num_points=300000, point_dim=4, voxel_size=[0.25, 0.25, 8.0],
                point_cloud_range=[-50.0, -50.0, -5.0, 50.0, 50.0, 3.0], max_points=64, max_voxels=40000)

CENTERPOINT_TASKS = [1, 2, 2, 1, 2, 2]  # classes per task (yml:139-151)
CENTERPOINT_TEST_CFG = dict(  # yml:163-172
    post_center_limit_range=[-61.2, -61.2, -10.0, 61.2, 61.2, 10.0], nms_pre_max_size=1000, nms_post_max_size=83,
    nms_iou_threshold=0.2, score_threshold=0.1, down_ratio=8)
# configs/centerpoint/centerpoint_pillars_02voxel_nuscenes_10sweep.yml: 0.2 m pillars on a 512 x 512 grid, one PFN layer
# of 64 channels, SecondBackbone 64/128/256 (layer_nums 3/5/5, strides 2/2/2), SecondFPN 128 x 3 with upsample_strides
# [0.5, 1, 2] (concat 384 channels at 128 x 128), CenterHead as the voxel model's; head maps at stride 4
CP_PILLARS = dict(name="centerpoint_pillar_02", num_points=300000, point_dim=5, voxel_size=[0.2, 0.2, 8.0],
                  point_cloud_range=[-51.2, -51.2, -5.0, 51.2, 51.2, 3.0], max_points=20, max_voxels=40000,
                  pfn_channels=64, backbone=dict(in_channels=64, out_channels=(64, 128, 256), layer_nums=(3, 5, 5),
                                                 downsample_strides=(2, 2, 2), fpn_out_channels=(128, 128, 128),
                                                 upsample_strides=(0.5, 1, 2), share_conv_channel=64, bev_depth=1))
CP_PILLARS_TEST_CFG = dict(CENTERPOINT_TEST_CFG, down_ratio=4)
# PointPillars, KITTI car (C2's voxelizer): one PFN layer of 64 channels, SecondBackbone 64/128/256 (layer_nums 3/5/5,
# strides 2/2/2), SecondFPN 128 x 3 with upsample_strides [1, 2, 4] (concat 384 channels at 248 x 216), SSD head with 2
# anchors per location and 1 class.  The anchor and test values are the standard PointPillars car ones (second.pytorch
# car config); they were NOT re-read from the reference yml (DESIGN.md, known gaps).
PP_KITTI_CAR = dict(C2, name="pointpillars_kitti_car", pfn_channels=64,
                    backbone=dict(in_channels=64, out_channels=(64, 128, 256), layer_nums=(3, 5, 5),
                                  downsample_strides=(2, 2, 2), fpn_out_channels=(128, 128, 128), upsample_strides=(1, 2, 4),
                                  bev_depth=1),
                    num_classes=1,
                    # create_anchors_3d_stride: feature map (ny, nx), (w, l, h), x / y / z strides and offsets; rotations as
                    # written in the config (1.57, not pi / 2)
                    anchors=dict(feature_size=(248, 216), sizes=(1.6, 3.9, 1.56), strides=(0.32, 0.32, 0.0),
                                 offsets=(0.16, -39.52, -1.78), rotations=(0, 1.57)),
                    test_cfg=dict(score_threshold=0.05, nms_pre_max_size=1000, nms_post_max_size=300, nms_iou_threshold=0.5,
                                  anchor_area_threshold=1, post_center_range=[0, -39.68, -5, 69.12, 39.68, 5]))


def uniform_cloud(cfg, seed, num_points=None, margin=0.02):
    """Worst case for hashing: x,y,z ~ U(range, slightly overshooting so some points fall outside)."""
    rng = np.random.default_rng(seed)
    n = cfg["num_points"] if num_points is None else num_points
    lo = np.asarray(cfg["point_cloud_range"][:3], np.float64)
    hi = np.asarray(cfg["point_cloud_range"][3:], np.float64)
    span = hi - lo
    xyz = rng.uniform(lo - margin * span, hi + margin * span, size=(n, 3))
    extra = rng.uniform(0.0, 1.0, size=(n, cfg["point_dim"] - 3))
    return np.concatenate([xyz, extra], 1).astype(np.float32)


def lidar_cloud(cfg, seed, num_points=None, sweeps=10, beams=32):
    """LiDAR-like occupancy (SURVEY.md §8d): `sweeps` x `beams` rings hitting the ground plane
    z=-1.8 m or one of 64 seeded boxes; sigma = 2 cm noise; intensity U(0,1); time lag = sweep*0.05."""
    rng = np.random.default_rng(seed)
    n = cfg["num_points"] if num_points is None else num_points
    pcr = cfg["point_cloud_range"]
    rmax = min(pcr[3], pcr[4])
    az_steps = int(math.ceil(n / (sweeps * beams))) + 8
    elev = np.deg2rad(np.linspace(-30.67, 10.67, beams))
    # boxes: centre (x,y), half sizes, height
    nb = 64
    bc = rng.uniform(-0.8 * rmax, 0.8 * rmax, size=(nb, 2))
    bs = rng.uniform(0.75, 5.0, size=(nb, 2))
    bh = rng.uniform(1.0, 3.5, size=(nb,))
    pts = []
    for s in range(sweeps):
        az = rng.uniform(0, 2 * np.pi) + np.linspace(0, 2 * np.pi, az_steps, endpoint=False)
        a, e = np.meshgrid(az, elev, indexing="ij")
        dx, dy, dz = np.cos(e) * np.cos(a), np.cos(e) * np.sin(a), np.sin(e)
        # ground hit
        with np.errstate(divide="ignore", invalid="ignore"):
            tg = np.where(dz < -1e-3, -1.8 / dz, np.inf)
        t = np.minimum(tg, rmax * 1.2)
        # box hits (slab test in xy, then height check)
        for k in range(nb):
            with np.errstate(divide="ignore", invalid="ignore"):
                tx1, tx2 = (bc[k, 0] - bs[k, 0]) / dx, (bc[k, 0] + bs[k, 0]) / dx
                ty1, ty2 = (bc[k, 1] - bs[k, 1]) / dy, (bc[k, 1] + bs[k, 1]) / dy
            tn = np.maximum(np.minimum(tx1, tx2), np.minimum(ty1, ty2))
            tf = np.minimum(np.maximum(tx1, tx2), np.maximum(ty1, ty2))
            hit = (tn > 0.5) & (tn < tf)
            zh = -1.8 + bh[k]
            zz = tn * dz
            hit &= (zz < zh - 1.8 + 1.8) & (zz > -1.8)
            t = np.where(hit & (tn < t), tn, t)
        ok = np.isfinite(t) & (t < rmax * 1.1)
        x, y, z = (t * dx)[ok], (t * dy)[ok], (t * dz)[ok]
        p = np.stack([x, y, z], 1) + rng.normal(0, 0.02, size=(ok.sum(), 3))
        cols = [p]
        if cfg["point_dim"] >= 4:
            cols.append(rng.uniform(0, 1, size=(len(p), 1)))
        if cfg["point_dim"] >= 5:
            cols.append(np.full((len(p), 1), s * 0.05))
        pts.append(np.concatenate(cols, 1))
    pts = np.concatenate(pts, 0)
    rng.shuffle(pts, axis=0)
    if len(pts) < n:  # pad by jittered repeats
        rep = pts[rng.integers(0, len(pts), size=n - len(pts))].copy()
        rep[:, :3] += rng.normal(0, 0.05, size=(len(rep), 3))
        pts = np.concatenate([pts, rep], 0)
    return pts[:n].astype(np.float32)


def random_boxes(n, seed, extent=40.0, clustered=True):
    """[x,y,z,dx,dy,dz,heading] boxes; clustered centres so that rotated overlaps are common."""
    rng = np.random.default_rng(seed)
    if clustered:
        centres = rng.uniform(-extent, extent, size=(max(n // 8, 1), 2))
        xy = centres[rng.integers(0, len(centres), size=n)] + rng.normal(0, 1.2, size=(n, 2))
    else:
        xy = rng.uniform(-extent, extent, size=(n, 2))
    z = rng.normal(-1.0, 0.5, size=(n, 1))
    dims = np.abs(rng.normal([4.2, 1.9, 1.6], [1.0, 0.4, 0.3], size=(n, 3))) + 0.2
    heading = rng.uniform(-np.pi, np.pi, size=(n, 1))
    return np.concatenate([xy, z, dims, heading], 1).astype(np.float32)


def centerpoint_head_outputs(seed, tasks=CENTERPOINT_TASKS, H=180, W=180, hm_mean=-5.5, hm_std=1.5,
                             with_velocity=True):
    """Per-task head tensors (NCHW, batch 1) with the statistics of SURVEY.md §8d."""
    rng = np.random.default_rng(seed)
    out = dict(hm=[], reg=[], height=[], dim=[], vel=[], rot=[])
    for c in tasks:
        out["hm"].append(rng.normal(hm_mean, hm_std, size=(1, c, H, W)).astype(np.float32))
        out["reg"].append(rng.uniform(0, 1, size=(1, 2, H, W)).astype(np.float32))
        out["height"].append(rng.normal(-1, 1, size=(1, 1, H, W)).astype(np.float32))
        out["dim"].append(rng.normal(0.5, 0.4, size=(1, 3, H, W)).astype(np.float32))
        out["rot"].append(rng.normal(0, 1, size=(1, 2, H, W)).astype(np.float32))
        out["vel"].append(rng.normal(0, 1, size=(1, 2, H, W)).astype(np.float32) if with_velocity else out["reg"][-1])
    return out


def label_offsets(tasks=CENTERPOINT_TASKS):
    """num_classes attr as built by CenterHead.predict_by_custom_op (center_head.py:306-309):
    prefix sums; only the first T entries are used by the op."""
    off, flag = [], 0
    for c in tasks:
        off.append(flag)
        flag += c
    return off


def bev_pool_inputs(seed, n_cams=6, D=118, H=16, W=44, C=80, grid=(128, 128, 1), bounds=((-51.2, 51.2), (-51.2, 51.2), (-5.0, 3.0)),
                    depth_range=(1.0, 60.0)):
    """Restatement of LSSViewTransformer.voxel_pooling_prepare_v2
    (paddle3d/models/transformers/bevdet_transformer.py:230-274) on a synthetic 6-camera rig:
    pinhole cameras at 60-degree yaw steps, frustum points -> ego frame -> voxel ranks, argsort, run lengths."""
    rng = np.random.default_rng(seed)
    B, N = 1, n_cams
    gx, gy, gz = grid
    lower = np.array([b[0] for b in bounds], np.float32)
    interval = np.array([(bounds[0][1] - bounds[0][0]) / gx, (bounds[1][1] - bounds[1][0]) / gy,
                         (bounds[2][1] - bounds[2][0]) / gz], np.float32)
    fx = 1266.0 * (704.0 / 1600.0) / 16.0  # focal in feature-map pixels
    cx, cy = W / 2.0, H / 2.0
    d = np.linspace(depth_range[0], depth_range[1], D, dtype=np.float32)
    u = (np.arange(W, dtype=np.float32) + 0.5)
    v = (np.arange(H, dtype=np.float32) + 0.5)
    dd, vv, uu = np.meshgrid(d, v, u, indexing="ij")  # D,H,W
    xc = (uu - cx) / fx * dd
    yc = (vv - cy) / fx * dd
    zc = dd
    coor = np.zeros((B, N, D, H, W, 3), np.float32)
    for n in range(N):
        yaw = n * (2 * np.pi / N)
        # camera: z forward, x right, y down  ->  ego: x forward, y left, z up
        fwd = np.array([np.cos(yaw), np.sin(yaw), 0.0], np.float32)
        right = np.array([np.sin(yaw), -np.cos(yaw), 0.0], np.float32)
        up = np.array([0.0, 0.0, 1.0], np.float32)
        p = zc[..., None] * fwd + xc[..., None] * right - yc[..., None] * up
        p[..., 2] += 1.5
        coor[0, n] = p
    num_points = B * N * D * H * W
    ranks_depth = np.arange(num_points, dtype=np.int64)
    ranks_feat = np.arange(num_points // D, dtype=np.int64).reshape(B, N, 1, H, W)
    ranks_feat = np.broadcast_to(ranks_feat, (B, N, D, H, W)).reshape(-1)
    c = ((coor - lower) / interval).astype(np.int64).reshape(num_points, 3)  # trunc toward 0 (:241-243)
    batch_idx = np.repeat(np.arange(B), num_points // B)
    kept = (c[:, 0] >= 0) & (c[:, 0] < gx) & (c[:, 1] >= 0) & (c[:, 1] < gy) & (c[:, 2] >= 0) & (c[:, 2] < gz)
    c, ranks_depth, ranks_feat, batch_idx = c[kept], ranks_depth[kept], ranks_feat[kept], batch_idx[kept]
    ranks_bev = batch_idx * (gz * gy * gx) + c[:, 2] * (gy * gx) + c[:, 1] * gx + c[:, 0]
    order = np.argsort(ranks_bev, kind="stable")
    ranks_bev, ranks_depth, ranks_feat = ranks_bev[order], ranks_depth[order], ranks_feat[order]
    first = np.ones(len(ranks_bev), bool)
    first[1:] = ranks_bev[1:] != ranks_bev[:-1]
    interval_starts = np.nonzero(first)[0].astype(np.int32)
    interval_lengths = np.zeros_like(interval_starts)
    interval_lengths[:-1] = interval_starts[1:] - interval_starts[:-1]
    interval_lengths[-1] = len(ranks_bev) - interval_starts[-1]
    logits = rng.normal(0, 1, size=(B * N, D, H, W)).astype(np.float32)
    e = np.exp(logits - logits.max(1, keepdims=True))
    depth = (e / e.sum(1, keepdims=True)).astype(np.float32)
    feat = rng.normal(0, 1, size=(B * N, H, W, C)).astype(np.float32)
    return dict(depth=depth, feat=feat, ranks_depth=ranks_depth.astype(np.int32), ranks_feat=ranks_feat.astype(np.int32),
                ranks_bev=ranks_bev.astype(np.int32), interval_starts=interval_starts,
                interval_lengths=interval_lengths.astype(np.int32), bev_feat_shape=(B, gy, gx, C),
                coor=coor, grid_lower_bound=lower, grid_interval=interval, grid_size=(gx, gy, gz))


def kaiming_uniform(rng, shape, fan_in):
    bound = math.sqrt(6.0 / fan_in) / math.sqrt(1 + 5.0)  # a = sqrt(5), as reset_parameters does
    return rng.uniform(-bound, bound, size=shape).astype(np.float32)
