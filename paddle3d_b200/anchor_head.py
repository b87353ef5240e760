"""PointPillars' anchor-based SSD head (SURVEY.md §8 C2): the cls / box / dir 1x1 convolutions on the SecondFPN concat, the
anchors they regress against, and the static per-anchor cell bounds of the anchor mask.

The anchor functions are restatements of the standard PointPillars / SECOND ones (second.pytorch box_np_ops:
create_anchors_3d_stride, rbbox2d_to_near_bbox, fused_get_anchors_area); they were NOT re-read from the reference tree
(PARITY UNPINNED, DESIGN.md §4).  numpy only, evaluated in fp32 like the numpy / numba originals.  The post-processing
that consumes all of this is ops.anchor_head (csrc/anchor_postprocess.cu)."""
import numpy as np

BOX_CODE = 7  # (x, y, z, w, l, h, r)


def create_anchors_3d_stride(feature_size, sizes, strides, offsets, rotations):
    """feature_size (ny, nx) -> anchors [ny * nx * A, 7] fp32, A = len(sizes) * len(rotations); anchor
    (y * nx + x) * A + s * len(rotations) + r has centre (x * stride_x + offset_x, y * stride_y + offset_y, offset_z),
    size sizes[s] = (w, l, h) and yaw rotations[r] (create_anchors_3d_stride's [z, y, x, size, rot, 7] order, z = 1)."""
    f32 = np.float32
    ny, nx = [int(v) for v in feature_size]
    xs = np.arange(nx, dtype=f32) * f32(strides[0]) + f32(offsets[0])
    ys = np.arange(ny, dtype=f32) * f32(strides[1]) + f32(offsets[1])
    z = f32(0) * f32(strides[2]) + f32(offsets[2])
    sizes = np.asarray(sizes, f32).reshape(-1, 3)
    rots = np.asarray(rotations, f32).reshape(-1)
    S, R = len(sizes), len(rots)
    out = np.empty((ny, nx, S, R, BOX_CODE), f32)
    out[..., 0] = xs.reshape(1, nx, 1, 1)
    out[..., 1] = ys.reshape(ny, 1, 1, 1)
    out[..., 2] = z
    out[..., 3:6] = sizes.reshape(1, 1, S, 1, 3)
    out[..., 6] = rots.reshape(1, 1, 1, R)
    return out.reshape(-1, BOX_CODE)


def _limit_period(val, offset=0.5, period=np.pi):
    return val - np.floor(val / np.float32(period) + np.float32(offset)) * np.float32(period)


def rbbox2d_to_near_bbox(rbboxes):
    """[N, 5] (x, y, xdim, ydim, rad) -> [N, 4] (xmin, ymin, xmax, ymax) of the nearest standing or lying box: the dims
    swap when |limit_period(rad, 0.5, pi)| > pi / 4."""
    rb = np.asarray(rbboxes, np.float32)
    cond = (np.abs(_limit_period(rb[:, 4])) > np.float32(np.pi / 4))[:, None]
    c = np.where(cond, rb[:, [0, 1, 3, 2]], rb[:, :4])
    half = c[:, 2:] / np.float32(2)
    return np.concatenate([c[:, :2] - half, c[:, :2] + half], 1)


def anchor_cells(anchors, voxel_size, point_cloud_range, grid_size):
    """Static cell bounds of the anchor mask: [N, 4] int32 (x0, y0, x1, y1) = floor((near_bbox - offset) / voxel) with the
    min corner clipped at 0 and the max corner at grid - 1, as fused_get_anchors_area computes them.  grid_size (nx, ny)."""
    bv = rbbox2d_to_near_bbox(np.asarray(anchors, np.float32)[:, [0, 1, 3, 4, 6]])
    st = np.asarray(voxel_size[:2], np.float32)
    off = np.asarray(point_cloud_range[:2], np.float32)
    c = np.floor((bv - np.concatenate([off, off])) / np.concatenate([st, st])).astype(np.int32)
    c[:, 0] = np.maximum(c[:, 0], 0)
    c[:, 1] = np.maximum(c[:, 1], 0)
    c[:, 2] = np.minimum(c[:, 2], int(grid_size[0]) - 1)
    c[:, 3] = np.minimum(c[:, 3], int(grid_size[1]) - 1)
    return np.ascontiguousarray(c)


def occupancy(coors, num_voxels, ny, nx):
    """Pillar occupancy [ny, nx] int32 of coors [:, 4] (b, z, y, x) (sparse_sum_for_anchors_mask; one pillar per cell)."""
    occ = np.zeros((ny, nx), np.int32)
    c = np.asarray(coors)[:int(num_voxels)]
    ok = (c[:, 2] >= 0) & (c[:, 2] < ny) & (c[:, 3] >= 0) & (c[:, 3] < nx)
    occ[c[ok, 2], c[ok, 3]] = 1
    return occ


def anchors_area(occ, cells):
    """fused_get_anchors_area on the integral image of occ: I[y1, x1] - I[y1, x0] - I[y0, x1] + I[y0, x0]."""
    I = np.asarray(occ, np.int64).cumsum(0).cumsum(1)
    x0, y0, x1, y1 = [cells[:, k] for k in range(4)]
    return I[y1, x1] - I[y1, x0] - I[y0, x1] + I[y0, x0]


class SSDHead:
    """cls (A * C), box (7A) and dir (2A) 1x1 convolutions on the FPN concat, run as ONE fp16-pair 1x1 convolution of
    in_channels -> A * (C + 9) with fp32 NCHW planes out; forward returns views (cls, box, dir) into them.  The dense
    kernel's epilogue writes exactly cout planes for any cout >= 16 (its N tile is zero-padded above cout).
    anchor_cfg: create_anchors_3d_stride's arguments (feature_size, sizes, strides, offsets, rotations)."""

    def __init__(self, in_channels, num_classes, anchor_cfg):
        from .dense_head import _Conv
        self.anchor_cfg = dict(anchor_cfg)
        self.A = len(np.asarray(anchor_cfg["sizes"]).reshape(-1, 3)) * len(anchor_cfg["rotations"])
        self.C = int(num_classes)
        self.planes = self.A * (self.C + 2 + BOX_CODE)
        if self.planes < 16:
            raise ValueError("SSDHead: A * (C + 9) = %d output planes; the fp16-pair 1x1 conv needs >= 16" % self.planes)
        self.conv = _Conv(in_channels, self.planes, 1, 1, 0, bias=True, relu=False, f16=True)
        self.anchors = create_anchors_3d_stride(**self.anchor_cfg)
        self.cells = None
        self.anchors_dev = self.cells_dev = None

    @property
    def num_anchors(self):
        return len(self.anchors)

    def init_weight(self, seed=0, device="cuda"):
        self.conv.init(np.random.default_rng(seed), device)
        self._device = device
        if device is not None:
            import torch
            self.anchors_dev = torch.from_numpy(self.anchors).to(device)
        return self

    def set_mask_grid(self, voxel_size, point_cloud_range, grid_size):
        """Static cell bounds of the anchor mask on the pillar grid (grid_size (nx, ny))."""
        self.cells = anchor_cells(self.anchors, voxel_size, point_cloud_range, grid_size)
        if getattr(self, "_device", None) is not None:
            import torch
            self.cells_dev = torch.from_numpy(self.cells).to(self._device)
        return self

    def split(self, planes):
        """[B, A * (C + 9), H, W] -> the (cls, box, dir) plane groups (views)."""
        a, c = self.A, self.C
        return planes[:, :a * c], planes[:, a * c:a * (c + BOX_CODE)], planes[:, a * (c + BOX_CODE):]

    def forward(self, cat, shape):
        """cat: pixel fp16-pair rows of the FPN concat, shape (B, H, W, in_channels) -> (cls, box, dir) fp32 NCHW views."""
        _, planes, _ = self.conv(cat, shape, want_nchw=True)
        return self.split(planes)

    __call__ = forward

    def export_numpy(self):
        return dict(conv=self.conv.np, num_anchors=self.A, num_classes=self.C, anchors=self.anchors)

    def calibrate_cls_bias(self, cat, shape, score_threshold, keep=None, target_frac=0.014):
        """Seeded random weights score anchors arbitrarily; a trained PointPillars fires on a few hundred.  This shifts every
        cls bias by one common amount so that round(target_frac * num_anchors) anchors (1 500 of the car model's 107 136,
        more than nms_pre_max_size) score at or above `score_threshold` on this frame.  keep: the frame's anchor mask
        (bool [num_anchors]); the count is taken among the kept anchors.  Weights stay seeded; the new bias is exported."""
        import torch
        cls, _, _ = self.forward(cat, shape)
        b, ac, h, w = cls.shape
        # logits per anchor (y, x, a) and class, the max over classes ranks the anchor (sigmoid is monotone)
        lg = cls[0].reshape(self.A, self.C, h * w).permute(2, 0, 1).reshape(-1, self.C).amax(1).double().cpu().numpy()
        if keep is not None:
            lg = lg[np.asarray(keep, bool)]
        k = max(1, min(len(lg), int(round(target_frac * self.num_anchors))))
        q = np.sort(lg)[len(lg) - k]  # the k-th largest logit
        logit_thr = float(np.log(score_threshold / (1.0 - score_threshold)))
        # shift so that q lands a little above the threshold logit (fp32 rounding of the conv must not drop it)
        shift = np.float32(logit_thr - q + 1e-3)
        bias = self.conv.np["bias"]
        bias[:self.A * self.C] = (bias[:self.A * self.C] + shift).astype(np.float32)
        self.conv.dev["shift"] = torch.from_numpy(bias.astype(np.float32)).to(cls.device)
        return self
