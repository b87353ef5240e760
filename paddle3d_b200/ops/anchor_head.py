"""Post-processing of PointPillars' anchor-based SSD head on the device (csrc/anchor_postprocess.cu): anchor mask,
sigmoid scores, top-k by score, second_box_decode, rotated NMS with rotate_nms_pcdet's semantics, direction fix and the
post_center_range filter, with no host synchronisation (the reference runs this as Python over Paddle ops,
pointpillars.py:105-129).  Batch size 1."""
import torch

from .._lib import check, host_floats, lib
from .._mem import ptr, require_cuda, stream, workspace


def anchor_head_postprocess_device(cls, box, dir, anchors, anchor_cells, coors, num_voxels, grid_ny, grid_nx,
                                   anchor_area_threshold, score_threshold, nms_iou_threshold, nms_pre_max_size,
                                   nms_post_max_size, post_center_range=None):
    """Sync-free form.  cls [1, A*C, H, W], box [1, 7A, H, W], dir [1, 2A, H, W] fp32; anchors [H*W*A, 7] fp32;
    anchor_cells [H*W*A, 4] int32 or None (no anchor mask; also when anchor_area_threshold < 0); coors [n, 4] (b, z, y, x)
    int32 and num_voxels [1] int32 of the frame's pillars.  Returns worst-case-sized (boxes [post_max, 7], scores, labels
    int64, anchor indices int32) plus counts [2] = (candidates, rows) on the device."""
    cls = require_cuda(cls, "cls", torch.float32)
    box = require_cuda(box, "box", torch.float32)
    dir = require_cuda(dir, "dir", torch.float32)
    anchors = require_cuda(anchors, "anchors", torch.float32)
    if cls.dim() != 4 or cls.shape[0] != 1:
        raise ValueError("cls must be [1, A*C, H, W]: batch size 1")
    _, AC, H, W = [int(v) for v in cls.shape]
    A = int(box.shape[1]) // 7
    if A < 1 or box.shape[1] != 7 * A or dir.shape[1] != 2 * A or AC % A or tuple(box.shape[2:]) != (H, W) or \
            tuple(dir.shape[2:]) != (H, W):
        raise ValueError("box must have 7A, dir 2A and cls A*C planes of one H x W")
    C = AC // A
    N = H * W * A
    if tuple(anchors.shape) != (N, 7):
        raise ValueError("anchors must be [H*W*A, 7] = [%d, 7], got %s" % (N, tuple(anchors.shape)))
    use_mask = anchor_cells is not None and anchor_area_threshold >= 0
    if use_mask:
        anchor_cells = require_cuda(anchor_cells, "anchor_cells", torch.int32)
        coors = require_cuda(coors, "coors", torch.int32)
        num_voxels = require_cuda(num_voxels, "num_voxels", torch.int32)
        if tuple(anchor_cells.shape) != (N, 4) or coors.dim() != 2 or coors.shape[1] != 4:
            raise ValueError("anchor_cells must be [H*W*A, 4] and coors [n, 4] (b, z, y, x)")
    else:
        anchor_cells = coors = num_voxels = None
        grid_ny = grid_nx = 0
    dev = cls.device
    rows = max(int(nms_post_max_size), 1)
    boxes = torch.empty((rows, 7), dtype=torch.float32, device=dev)
    scores = torch.empty((rows,), dtype=torch.float32, device=dev)
    labels = torch.empty((rows,), dtype=torch.int64, device=dev)
    index = torch.empty((rows,), dtype=torch.int32, device=dev)
    counts = torch.empty((2,), dtype=torch.int32, device=dev)
    L = lib()
    nbytes = L.p3d_anchor_head_postprocess_workspace_bytes(N, int(grid_ny), int(grid_nx), int(nms_pre_max_size))
    if not nbytes:
        raise ValueError("anchor_head_postprocess: unsupported sizes (anchors %d, grid %s x %s, pre_max %s)" % (
            N, grid_ny, grid_nx, nms_pre_max_size))
    ws = workspace(nbytes, dev, "anchor_head")
    rng = host_floats(post_center_range) if post_center_range is not None else None
    check(L.p3d_anchor_head_postprocess(ptr(cls), ptr(box), ptr(dir), H, W, A, C, ptr(anchors), ptr(anchor_cells),
                                        ptr(coors), ptr(num_voxels), int(grid_ny), int(grid_nx),
                                        float(anchor_area_threshold), float(score_threshold), float(nms_iou_threshold),
                                        int(nms_pre_max_size), int(nms_post_max_size), rng, ptr(boxes), ptr(scores),
                                        ptr(labels), ptr(index), ptr(counts), ptr(ws), ws.numel(), stream(dev)),
          "anchor_head_postprocess")
    return boxes, scores, labels, index, counts


def anchor_head_postprocess(cls, box, dir, anchors, anchor_cells, coors, num_voxels, grid_ny, grid_nx,
                            anchor_area_threshold, score_threshold, nms_iou_threshold, nms_pre_max_size,
                            nms_post_max_size, post_center_range=None):
    """(boxes [K, 7] fp32, scores [K] fp32, labels [K] int64) as SECOND's predict returns them (box3d_lidar, scores,
    label_preds).  The only host sync is the read of K needed to give the outputs their dynamic shape."""
    boxes, scores, labels, _, counts = anchor_head_postprocess_device(
        cls, box, dir, anchors, anchor_cells, coors, num_voxels, grid_ny, grid_nx, anchor_area_threshold,
        score_threshold, nms_iou_threshold, nms_pre_max_size, nms_post_max_size, post_center_range)
    k = int(counts[-1].item())
    return boxes[:k], scores[:k], labels[:k]
