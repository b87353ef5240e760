#!/usr/bin/env python
"""Deploy-style CLI (mirrors deploy/centerpoint/python/infer.py:54-201): one `.bin` sweep in, detections out.

    python tools/infer.py --lidar_file sweep.bin --num_point_dim 5 [--use_timelag 1] [--model voxel|pillars] [--out results.txt]
    python tools/infer.py --lidar_file kitti.bin --num_point_dim 4 --use_timelag 0 --model pointpillars

No checkpoints exist offline: the model runs with the seeded weights of the benchmark (same architecture)."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from paddle3d_b200 import deploy  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lidar_file", required=True, help="path of a float32 .bin point file")
    ap.add_argument("--num_point_dim", type=int, default=5, help="values per point in the file (infer.py:61-65)")
    ap.add_argument("--use_timelag", type=int, default=1, help="append the time-lag column (infer.py:66-70)")
    ap.add_argument("--gpu_id", type=int, default=0)
    ap.add_argument("--max_points", type=int, default=300000)
    ap.add_argument("--no_head", action="store_true", help="voxel model only: resident synthetic head tensors")
    ap.add_argument("--model", default="voxel", choices=["voxel", "pillars", "pointpillars"],
                    help="CenterPoint-voxel (0.075 m), CenterPoint-pillars (0.2 m) or PointPillars (KITTI car, 7-column "
                         "boxes; points x, y, z, intensity: --num_point_dim 4 --use_timelag 0)")
    ap.add_argument("--out", default=None, help="also write the detections to this text file")
    args = ap.parse_args()
    points = deploy.preprocess(args.lidar_file, args.num_point_dim, bool(args.use_timelag))
    from paddle3d_b200.pipeline import CenterPointHotPath, CenterPointPillarsHotPath, PointPillarsHotPath
    cls = {"voxel": CenterPointHotPath, "pillars": CenterPointPillarsHotPath, "pointpillars": PointPillarsHotPath}[args.model]
    pred = deploy.Predictor(device="cuda:%d" % args.gpu_id, max_points=max(args.max_points, len(points)),
                            with_head=not args.no_head, pipeline_cls=cls)
    box3d_lidar, label_preds, scores = pred.run(points)
    deploy.parse_result(box3d_lidar, label_preds, scores)
    if args.out:
        deploy.write_results(args.out, box3d_lidar, label_preds, scores)


if __name__ == "__main__":
    main()
