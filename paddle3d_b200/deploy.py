"""Deploy-style runner and result output (SURVEY.md §8f-4), mirroring `deploy/centerpoint/python/infer.py`:

    preprocess(file, num_point_dim, use_timelag)   infer.py:86-104   read a `.bin` sweep, keep x, y, z, intensity, add the lag column
    Predictor(...).run(points)                      infer.py:163-189  -> (box3d_lidar [K, 9], label_preds [K], scores [K]) on the host
    parse_result(box3d_lidar, label_preds, scores)  infer.py:139-160  the reference's text format, fake rows (score -1) skipped

The predictor is `CenterPointHotPath` (or, with pipeline_cls, `CenterPointPillarsHotPath` / `PointPillarsHotPath`) behind the reference's three-output contract (the exported model's outputs are
box3d_lidar, label_preds, scores in that order, infer.py:180-188).  A frame may hold fewer points than the capacity the
pipeline was captured for: the tail of the device buffer is filled with NaN rows, which `hard_voxelize` drops exactly
like the reference drops out-of-range points (voxelize_op.cc:37-45 -> csrc/voxelize.cu cell_of).  Host code, as in the
reference; the CLI is tools/infer.py.
"""
import sys

import numpy as np


def read_point(file_path, num_point_dim):
    points = np.fromfile(file_path, np.float32).reshape(-1, num_point_dim)
    return points[:, :4]


def insert_time_to_points(points):
    return np.hstack([points, np.zeros((points.shape[0], 1), dtype=points.dtype)])


def preprocess(file_path, num_point_dim, use_timelag):
    points = read_point(file_path, num_point_dim)
    return insert_time_to_points(points) if use_timelag else points


def format_result(box3d_lidar, label_preds, scores):
    """The lines parse_result prints (infer.py:139-160), as a list of strings."""
    box3d_lidar, label_preds, scores = np.asarray(box3d_lidar), np.asarray(label_preds), np.asarray(scores)
    num_bbox3d, dims = box3d_lidar.shape
    lines = []
    for i in range(num_bbox3d):
        if scores[i] < 0:  # fake row of an empty task (postprocess.cu:190-202)
            continue
        b = box3d_lidar[i]
        if dims == 9:
            lines.append("Score: {} Label: {} Box(x_c, y_c, z_c, w, l, h, vec_x, vec_y, -rot): {} {} {} {} {} {} {} {} {}".format(
                scores[i], label_preds[i], b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7], b[8]))
        elif dims == 7:
            lines.append("Score: {} Label: {} Box(x_c, y_c, z_c, w, l, h, -rot): {} {} {} {} {} {} {}".format(
                scores[i], label_preds[i], b[0], b[1], b[2], b[3], b[4], b[5], b[6]))
    return lines


def parse_result(box3d_lidar, label_preds, scores, file=None):
    for line in format_result(box3d_lidar, label_preds, scores):
        print(line, file=file or sys.stdout)


def write_results(path, box3d_lidar, label_preds, scores):
    """Same lines into a text file (one detection per line)."""
    with open(path, "w") as f:
        parse_result(box3d_lidar, label_preds, scores, file=f)


class Predictor:
    """`init_predictor` + `run` of the reference's deploy script over the B200 pipeline."""

    def __init__(self, cfg=None, device="cuda:0", max_points=None, seed=0, precision=None, with_head=True, weights=None,
                 pipeline_cls=None):
        """pipeline_cls: CenterPointHotPath (default), CenterPointPillarsHotPath or PointPillarsHotPath; cfg defaults to the
        class's default_cfg (synth.C3, synth.CP_PILLARS, synth.PP_KITTI_CAR).  precision and with_head apply to the voxel
        model only: the pillar models always run their fp16-pair dense heads."""
        import torch
        from .ops import sparse_nn as sp
        from .pipeline import CenterPointHotPath
        self.torch = torch
        pipeline_cls = pipeline_cls or CenterPointHotPath
        self.cfg = dict(cfg or pipeline_cls.default_cfg)
        if pipeline_cls is CenterPointHotPath:
            self.pipe = CenterPointHotPath(self.cfg, device, precision=sp.F16X3 if precision is None else precision,
                                           seed=seed, num_points=max_points, with_head=with_head)
        else:
            self.pipe = pipeline_cls(self.cfg, device, seed=seed, num_points=max_points)
        self.host = torch.empty((self.pipe.n, self.pipe.F), dtype=torch.float32).pin_memory()
        self.captured = False

    def run(self, points):
        """points [n, F] fp32 (n <= capacity) -> (box3d_lidar, label_preds, scores) numpy arrays."""
        points = np.ascontiguousarray(points, dtype=np.float32)
        n, f = points.shape
        if f != self.pipe.F:
            raise ValueError("expected %d values per point, got %d" % (self.pipe.F, f))
        if n > self.pipe.n:
            raise ValueError("%d points exceed the capacity %d this predictor was built for" % (n, self.pipe.n))
        h = self.host.numpy()
        h[:n] = points
        h[n:] = np.nan  # dropped by the voxelizer like any point outside the range
        if not self.captured:
            self.pipe.points.copy_(self.host)
            self.pipe.capture()
            self.captured = True
        boxes, scores, labels = self.pipe.infer(self.host)
        return boxes.numpy().copy(), labels.numpy().copy(), scores.numpy().copy()
