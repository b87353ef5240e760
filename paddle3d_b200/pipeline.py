"""CenterPoint hot-path frames on one B200: the public API a user calls (bench.py `e2e`).  CenterPointHotPath is the voxel
model (below); CenterPointPillarsHotPath the 0.2 m pillar model (hard_voxelize -> PillarFeatureNet into the pixel fp16-pair
BEV image -> the same dense RPN / neck / CenterHead -> centerpoint_postprocess); PointPillarsHotPath the PointPillars KITTI
car model (same pillar front end -> SecondRPN -> SSD head -> anchor_head_postprocess).  All share their frame I/O
(_FramePipeline) and run side by side in CenterPointSweep lanes.

    voxelize (+ VoxelMean fused)  ->  SparseResNet3D (21 sparse convs)  ->  dense BEV [1,256,180,180]
    -> dense 2-D RPN + neck + CenterHead (with_head=True; otherwise resident synthetic head tensors)
    -> centerpoint_postprocess -> boxes

Everything between the H2D copy of the points and the D2H copy of the boxes is captured once in a
CUDA graph (data-dependent row counts live in device scalars, buffers are sized by capacity), so a
frame is: cudaMemcpyAsync H2D, one graph launch, cudaMemcpyAsync D2H.
Call sites mirrored: CenterPoint.extract_feat (centerpoint.py:126-138) and
CenterHead.predict_by_custom_op (center_head.py:294-339).
"""
import numpy as np
import torch

from . import synth
from .layers import SparseResNet3D
from .ops import centerpoint_postprocess as cpp
from .ops import sparse_nn as sp
from .ops import voxelize as vox

# BatchNorm gamma of the seeded pillar model (PillarFeatureNet and dense head): keeps the activations O(1) through the
# 1 + 16 + 3 + 1 + 36 layers of the frame (see DESIGN.md §1)
PILLARS_BN_GAIN = 6.0 ** 0.5


def _count_graph_nodes(raw_graph):
    """Node counts of a cudaGraph_t by type, through libcudart (ctypes)."""
    import ctypes as C
    rt = C.CDLL("libcudart.so")
    n = C.c_size_t(0)
    g = C.c_void_p(int(raw_graph))
    if rt.cudaGraphGetNodes(g, None, C.byref(n)) != 0:
        return None
    nodes = (C.c_void_p * n.value)()
    if rt.cudaGraphGetNodes(g, nodes, C.byref(n)) != 0:
        return None
    names = {0: "kernel", 1: "memcpy", 2: "memset"}  # cudaGraphNodeType
    out = {"kernel": 0, "memcpy": 0, "memset": 0, "other": 0}
    for i in range(n.value):
        t = C.c_int(0)
        rt.cudaGraphNodeGetType(C.c_void_p(nodes[i]), C.byref(t))
        out[names.get(t.value, "other")] += 1
    return out


class _FramePipeline:
    """Frame I/O shared by the CenterPoint pipelines: the static device input, the pipeline stream, the CUDA graph of
    one frame and the pinned result buffers; infer / infer_many / capture / launch around the subclass's
    forward_device() (one frame enqueued on the current stream, returning a dict with at least boxes, scores, labels,
    counts and status) and check_status() (raises on a non-zero device status word)."""

    # attributes a CenterPointSweep lane shares with lane 0 (one model); default_cfg: the configuration a Predictor uses
    shared_attrs = ("net", "dense")
    default_cfg = None

    def _init_io(self, status_words, rows=None, box_dim=9, count_words=None):
        """Needs self.n, self.F, self.device, and (for the defaults of rows / count_words: one block of result rows and
        one count per task, then the total) self.label_off and self.test_cfg.  The total row count is the last count."""
        self.points = torch.zeros((self.n, self.F), dtype=torch.float32, device=self.device)  # static input
        self.graph = None
        self.out = None
        self.stream = torch.cuda.Stream(self.device)
        if rows is None:
            rows = len(self.label_off) * self.test_cfg["nms_post_max_size"]
        if count_words is None:
            count_words = len(self.label_off) + 1
        self.h_boxes = torch.empty((rows, box_dim), dtype=torch.float32).pin_memory()
        self.h_scores = torch.empty((rows,), dtype=torch.float32).pin_memory()
        self.h_labels = torch.empty((rows,), dtype=torch.int64).pin_memory()
        self.h_counts = torch.empty((count_words,), dtype=torch.int32).pin_memory()
        self.h_status = torch.zeros((status_words,), dtype=torch.int32).pin_memory()

    def capture(self, warmup=2, count_nodes=False):
        """Warm up (sizes the workspaces) on the side stream, then capture the frame into a CUDA graph.  count_nodes:
        keep the cudaGraph_t and store its node counts (cudaGraphGetNodes / cudaGraphNodeGetType) in self.graph_nodes =
        {"kernel": .., "memset": .., "memcpy": .., "other": ..}."""
        with torch.cuda.stream(self.stream):
            for _ in range(warmup):
                self.out = self.forward_device()
            self.stream.synchronize()
            self.graph = torch.cuda.CUDAGraph(keep_graph=True) if count_nodes else torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=self.stream):
                self.out = self.forward_device()
            self.graph_nodes = None
            if count_nodes:
                try:
                    self.graph_nodes = _count_graph_nodes(self.graph.raw_cuda_graph())
                except Exception:  # noqa: BLE001  (a debugging aid must not take the pipeline down)
                    self.graph_nodes = None
        self.stream.synchronize()
        return self

    def launch(self):
        """Replay the captured frame on the pipeline stream (inputs already in self.points)."""
        with torch.cuda.stream(self.stream):
            self.graph.replay()

    # ---- public end-to-end call: host points in, host boxes out
    def infer(self, points_host):
        """points_host: pinned [n, F] fp32 tensor.  Returns (boxes [K,9], scores [K], labels [K]) on the host."""
        with torch.cuda.stream(self.stream):
            self.points.copy_(points_host, non_blocking=True)
            if self.graph is not None:
                self.graph.replay()
            else:
                self.out = self.forward_device()
            o = self.out
            self.h_counts.copy_(o["counts"], non_blocking=True)
            self.h_status.copy_(o["status"], non_blocking=True)
            self.h_boxes.copy_(o["boxes"], non_blocking=True)
            self.h_scores.copy_(o["scores"], non_blocking=True)
            self.h_labels.copy_(o["labels"], non_blocking=True)
        self.stream.synchronize()
        self.check_status(self.h_status)
        k = int(self.h_counts[-1])
        return self.h_boxes[:k], self.h_scores[:k], self.h_labels[:k]

    # ---- public end-to-end call for a sweep of frames: same per-frame work, copies overlapped with compute
    def prepare_sweep(self):
        """Copy stream, staging buffers, pinned result slots and events of infer_many (allocated once; pinned allocations
        cost milliseconds, so callers that time a sweep call this first)."""
        if getattr(self, "_copy_stream", None) is not None:
            return self
        self._copy_stream = torch.cuda.Stream(self.device)
        self._staging = [torch.empty_like(self.points) for _ in range(2)]
        self._slots = [dict(boxes=torch.empty_like(self.h_boxes).pin_memory(),
                            scores=torch.empty_like(self.h_scores).pin_memory(),
                            labels=torch.empty_like(self.h_labels).pin_memory(),
                            counts=torch.empty_like(self.h_counts).pin_memory(),
                            status=torch.zeros_like(self.h_status).pin_memory()) for _ in range(2)]
        self._staged = [torch.cuda.Event() for _ in range(2)]    # H2D into staging[k] done
        self._consumed = [torch.cuda.Event() for _ in range(2)]  # staging[k] copied into the graph's input
        self._done = [torch.cuda.Event() for _ in range(2)]      # results of slot k are on the host
        return self

    def _submit(self, pts, k, first_use):
        """Enqueue one frame of a sweep into slot k: H2D on the copy stream, graph replay, D2H of the results."""
        cs, st = self._copy_stream, self.stream
        with torch.cuda.stream(cs):
            if not first_use:
                cs.wait_event(self._consumed[k])
            self._staging[k].copy_(pts, non_blocking=True)
            self._staged[k].record(cs)
        with torch.cuda.stream(st):
            st.wait_event(self._staged[k])
            self.points.copy_(self._staging[k], non_blocking=True)
            self._consumed[k].record(st)
            self.graph.replay()
            o, sl = self.out, self._slots[k]
            sl["counts"].copy_(o["counts"], non_blocking=True)
            sl["status"].copy_(o["status"], non_blocking=True)
            sl["boxes"].copy_(o["boxes"], non_blocking=True)
            sl["scores"].copy_(o["scores"], non_blocking=True)
            sl["labels"].copy_(o["labels"], non_blocking=True)
            self._done[k].record(st)

    def _result(self, k):
        self._done[k].synchronize()
        sl = self._slots[k]
        self.check_status(sl["status"])
        n = int(sl["counts"][-1])
        return sl["boxes"][:n].clone(), sl["scores"][:n].clone(), sl["labels"][:n].clone()

    def infer_many(self, frames_host):
        """frames_host: iterable of pinned [n, F] fp32 tensors.  Yields (boxes, scores, labels) per frame, in order.

        Every frame still pays its own H2D copy and its own D2H read-back; the H2D of frame i+1 runs on a copy
        stream while frame i computes (two device staging buffers, two pinned result slots), and the host reads the
        results of frame i after it has submitted frame i+1.  CenterPointSweep runs several such lanes side by side."""
        if self.graph is None:
            raise RuntimeError("infer_many needs a captured pipeline: call capture() first")
        self.prepare_sweep()
        i = -1
        for i, pts in enumerate(frames_host):
            self._submit(pts, i & 1, i < 2)
            if i >= 1:
                yield self._result((i - 1) & 1)
        if i >= 0:
            yield self._result(i & 1)

    def bytes_per_frame(self):
        h2d = self.n * self.F * 4
        d2h = (self.h_boxes.numel() * 4 + self.h_scores.numel() * 4 + self.h_labels.numel() * 8 + self.h_counts.numel() * 4 +
               self.h_status.numel() * 4)
        return h2d, d2h


class CenterPointHotPath(_FramePipeline):
    default_cfg = synth.C3

    def __init__(self, cfg=None, device="cuda:0", precision=sp.FP32, seed=0, num_points=None, level_caps=None,
                 head_seed=0, with_head=False, keep_bev=True, bn_gain=1.0):
        self.cfg = dict(cfg or synth.C3)
        self.device = torch.device(device)
        self.n = int(num_points or self.cfg["num_points"])
        self.F = self.cfg["point_dim"]
        self.test_cfg = dict(synth.CENTERPOINT_TEST_CFG)
        self.label_off = synth.label_offsets()
        self.net = SparseResNet3D(self.F, self.cfg["voxel_size"], self.cfg["point_cloud_range"])
        self.net.init_weight(seed=seed, device=self.device, bn_gain=bn_gain).set_precision(precision)
        V = self.cfg["max_voxels"]
        self.net.set_level_caps(level_caps or [3 * V, 3 * V, 2 * V, V])
        h = synth.centerpoint_head_outputs(head_seed)
        self.head_host = h
        self.head = {k: [torch.from_numpy(x).to(self.device) for x in v] for k, v in h.items()}
        # with_head: run the dense RPN / neck / CenterHead (dense_head.DenseRPNHead, SURVEY §8f-1) on the BEV tensor and
        # feed ITS outputs to the postprocess instead of the resident synthetic head tensors (parity-green per layer and
        # as a small network; this whole-frame composition has not been timed yet, hence off by default)
        self.dense = None
        if with_head:
            from .dense_head import DenseRPNHead
            self.dense = DenseRPNHead(in_channels=128 * 2).init_weight(seed=seed + 1, device=self.device, bn_gain=bn_gain)
        # keep_bev=False (with the fp16-pair dense head): the sparse rows go straight into the pixel fp16-pair image the RPN
        # reads; the reference's fp32 NCHW BEV tensor is then not materialised in the frame (bev_nchw() rebuilds it on demand)
        self.keep_bev = keep_bev or self.dense is None or not self.dense.f16
        self._init_io(5)

    # ---- one frame, enqueued on the current stream, device in / device out
    def forward_device(self):
        cfg, tc = self.cfg, self.test_cfg
        mean, coors, npv, nv = vox.voxelize_mean(self.points, cfg["voxel_size"], cfg["point_cloud_range"],
                                                 cfg["max_points"], cfg["max_voxels"], 0)
        bev, bev_h16 = None, None
        if self.keep_bev:
            bev = self.net(mean, coors, 1, num=nv)
            h = self.dense(bev) if self.dense is not None else self.head
        else:
            bev_h16 = self.net(mean, coors, 1, num=nv, pixel_h16=True)
            h = self.dense.forward_h16(*bev_h16)
        # frame status word (ADVICE r1): [fp16-range overflow of the pair-row kernels, overflow flag of each strided level]
        status = torch.stack([sp.status_tensor(self.device)[0]] + [c[1] for c in self.net.level_counters])
        boxes, scores, labels, counts = cpp.centerpoint_postprocess_device(
            h["hm"], h["reg"], h["height"], h["dim"], h["vel"], h["rot"], cfg["voxel_size"][:2],
            cfg["point_cloud_range"], tc["post_center_limit_range"], self.label_off, tc["down_ratio"],
            tc["score_threshold"], tc["nms_iou_threshold"], tc["nms_pre_max_size"], tc["nms_post_max_size"], True)
        return dict(bev=bev, bev_h16=bev_h16, boxes=boxes, scores=scores, labels=labels, counts=counts, num_voxels=nv,
                    coors=coors, mean=mean, status=status)

    def bev_nchw(self):
        """The dense BEV tensor [1, 256, H, W] fp32 of the last frame (rebuilt from the pixel fp16-pair image when the
        frame did not materialise it)."""
        if self.out["bev"] is not None:
            self.stream.synchronize()
            return self.out["bev"]
        from .ops import dense_conv as dc
        rows, shape = self.out["bev_h16"]
        with torch.cuda.stream(self.stream):
            out = dc.pixel_h16_to_nchw(rows, shape)
            # pixel rows hold (z, c)-ordered channels (to_pixel_h16); the reference tensor is (c, z)-ordered
            b, h, w, cd = shape
            D = self.dense.bev_depth
            out = out.view(b, D, cd // D, h, w).transpose(1, 2).reshape(b, cd, h, w).contiguous()
        self.stream.synchronize()  # callers read it from other streams
        return out

    def calibrate_head(self, points_dev):
        """Shift the heat-map biases of the (randomly initialised) dense head so that ~1.4 % of the BEV cells of this frame
        score above the threshold, as SURVEY.md §8d specifies for the synthetic workload (see
        DenseRPNHead.calibrate_heatmap_bias).  Call before capture()."""
        if self.dense is None:
            return self
        cfg = self.cfg
        with torch.cuda.stream(self.stream):
            self.points.copy_(points_dev)
            mean, coors, npv, nv = vox.voxelize_mean(self.points, cfg["voxel_size"], cfg["point_cloud_range"],
                                                     cfg["max_points"], cfg["max_voxels"], 0)
            bev = self.net(mean, coors, 1, num=nv)
            self.dense.calibrate_heatmap_bias(bev, self.test_cfg["score_threshold"])
        self.stream.synchronize()
        return self

    @staticmethod
    def check_status(status_host):
        """Raise when the frame's device status word reports dropped work (never a silent wrong result)."""
        st = [int(v) for v in status_host]
        if st[0]:
            raise RuntimeError("sparse backbone: an activation left fp16's range (|x| >= 65504) on the fp16-pair path; "
                               "run this model with precision TF32X3_SPLIT")
        for lvl, v in enumerate(st[1:]):
            if v:
                raise RuntimeError("sparse backbone: strided level %d overflowed its row capacity (set_level_caps); "
                                   "output sites were dropped" % (lvl + 1))

    def export_weights_numpy(self):
        """Weights as plain numpy dicts for the CPU arm (oracle.cpu_reference.CpuFrame)."""
        def conv(l):
            return dict(weight=l.weight.cpu().numpy(), bias=None if l.bias is None else l.bias.cpu().numpy(),
                        stride=l.stride, padding=l.padding)

        def bn(l):
            return dict(gamma=l.weight.cpu().numpy(), beta=l.bias.cpu().numpy(), mean=l._mean.cpu().numpy(),
                        var=l._variance.cpu().numpy(), eps=l.epsilon)

        def block(b):
            return dict(conv1=conv(b.conv1), bn1=bn(b.bn1), conv2=conv(b.conv2), bn2=bn(b.bn2))

        n = self.net
        return dict(conv_input=dict(conv=conv(n.conv_input[0]), bn=bn(n.conv_input[1])),
                    blocks0=[block(b) for b in n.blocks0],
                    stages=[dict(down=dict(conv=conv(d[0]), bn=bn(d[1])), blocks=[block(b) for b in bl]) for d, bl in n.stages],
                    extra=dict(conv=conv(n.extra_conv[0]), bn=bn(n.extra_conv[1])))


class _PillarFramePipeline(_FramePipeline):
    """Pillar front end shared by the pillar models: hard_voxelize + PillarFeatureNet written straight into the pixel
    fp16-pair BEV image (needs self.cfg, self.net, self.ny, self.nx); status word [fp16-range overflow]."""

    def _front(self):
        """hard_voxelize + the pillar encoder into the pixel fp16-pair image: (rows, shape), num_voxels, coors."""
        cfg = self.cfg
        voxels, coords, npv, nv = vox.hard_voxelize(self.points, cfg["voxel_size"], cfg["point_cloud_range"],
                                                    cfg["max_points"], cfg["max_voxels"])
        coors = torch.nn.functional.pad(coords, (1, 0), value=0)  # (b, z, y, x), batch 0 (voxelize.py:51-57)
        img = self.net.forward_pixel_h16(voxels, npv, coors, 1, self.ny, self.nx, num=nv)
        return img, nv, coors

    def bev_nchw(self):
        """The pillar canvas [1, C, ny, nx] fp32 of the last frame, rebuilt from its pixel fp16-pair image."""
        from .ops import dense_conv as dc
        with torch.cuda.stream(self.stream):
            out = dc.pixel_h16_to_nchw(*self.out["bev_h16"])
        self.stream.synchronize()  # callers read it from other streams
        return out

    @staticmethod
    def check_status(status_host):
        """Raise when the frame's device status word reports a saturated value (never a silent wrong result)."""
        if int(status_host[0]):
            raise RuntimeError("pillar frame: an activation left fp16's range (|x| > 65504) on the fp16-pair path and "
                               "was saturated")


class CenterPointPillarsHotPath(_PillarFramePipeline):
    """CenterPoint-pillars hot-path frame (centerpoint_pillars_02voxel_nuscenes_10sweep.yml, synth.CP_PILLARS):

        hard_voxelize -> PillarFeatureNet written straight into the pixel fp16-pair BEV image [1, 512, 512, 64]
        -> SecondBackbone + SecondFPN (down-sampling, 1x1 and up-sampling deblocks) + CenterHead -> centerpoint_postprocess

    captured as one CUDA graph, with the same public calls as CenterPointHotPath.  No fp32 NCHW canvas exists in the frame
    (bev_nchw() rebuilds it on demand).  Status word: [fp16-range overflow of the pair-image kernels]."""
    default_cfg = synth.CP_PILLARS

    def __init__(self, cfg=None, device="cuda:0", seed=0, num_points=None, bn_gain=PILLARS_BN_GAIN, test_cfg=None):
        from .dense_head import DenseRPNHead
        from .layers import PillarFeatureNet, _grid
        self.cfg = dict(cfg or synth.CP_PILLARS)
        cfg = self.cfg
        self.device = torch.device(device)
        self.n = int(num_points or cfg["num_points"])
        self.F = cfg["point_dim"]
        self.test_cfg = dict(test_cfg or synth.CP_PILLARS_TEST_CFG)
        self.label_off = synth.label_offsets()
        g = _grid(cfg["point_cloud_range"], cfg["voxel_size"])
        self.nx, self.ny = int(g[0]), int(g[1])
        self.net = PillarFeatureNet(self.F, (cfg["pfn_channels"],), False, cfg["max_points"], cfg["voxel_size"],
                                    cfg["point_cloud_range"])
        self.net.init_weight(seed=seed, device=self.device, bn_gain=bn_gain)
        self.dense = DenseRPNHead(**cfg["backbone"]).init_weight(seed=seed + 1, device=self.device, bn_gain=bn_gain)
        self._init_io(1)

    # ---- one frame, enqueued on the current stream, device in / device out
    def forward_device(self):
        cfg, tc = self.cfg, self.test_cfg
        bev_h16, nv, coors = self._front()
        h = self.dense.forward_h16(*bev_h16)
        status = sp.status_tensor(self.device).clone()
        boxes, scores, labels, counts = cpp.centerpoint_postprocess_device(
            h["hm"], h["reg"], h["height"], h["dim"], h["vel"], h["rot"], cfg["voxel_size"][:2],
            cfg["point_cloud_range"], tc["post_center_limit_range"], self.label_off, tc["down_ratio"],
            tc["score_threshold"], tc["nms_iou_threshold"], tc["nms_pre_max_size"], tc["nms_post_max_size"], True)
        return dict(bev=None, bev_h16=bev_h16, head=h, boxes=boxes, scores=scores, labels=labels, counts=counts,
                    num_voxels=nv, coors=coors, status=status)

    def calibrate_head(self, points_dev):
        """As CenterPointHotPath.calibrate_head: shift the heat-map biases so that ~1.4 % of the cells of this frame score
        above the threshold.  Call before capture()."""
        from .ops import dense_conv as dc
        with torch.cuda.stream(self.stream):
            self.points.copy_(points_dev)
            img, _, _ = self._front()
            self.dense.calibrate_heatmap_bias(dc.pixel_h16_to_nchw(*img), self.test_cfg["score_threshold"])
        self.stream.synchronize()
        return self

    def export_weights_numpy(self):
        """Weights as plain numpy dicts for the CPU arm (oracle.cpu_reference.CpuPillarFrame)."""
        return dict(pfn=dict(self.net.np), dense=self.dense.export_numpy())


class PointPillarsHotPath(_PillarFramePipeline):
    """PointPillars, KITTI car (synth.PP_KITTI_CAR; the reference's detection/pointpillars):

        hard_voxelize -> PillarFeatureNet written straight into the pixel fp16-pair BEV image [1, 496, 432, 64]
        -> SecondBackbone + SecondFPN (dense_head.SecondRPN: concat of 384 channels at 248 x 216)
        -> SSD head (anchor_head.SSDHead: cls / box / dir as one 1x1 conv, 20 fp32 planes)
        -> anchor_head_postprocess (anchor mask, scores, top-k, decode, rotated NMS, direction fix, range filter)

    captured as one CUDA graph, with the same public calls as the CenterPoint pipelines.  Results: boxes [K, 7] (x, y, z,
    w, l, h, r), scores [K], labels [K] (class index).  Status word: [fp16-range overflow of the pair-image kernels]."""
    shared_attrs = ("net", "dense", "ssd")
    default_cfg = synth.PP_KITTI_CAR

    def __init__(self, cfg=None, device="cuda:0", seed=0, num_points=None, bn_gain=PILLARS_BN_GAIN, test_cfg=None):
        from .anchor_head import SSDHead
        from .dense_head import SecondRPN
        from .layers import PillarFeatureNet, _grid
        self.cfg = dict(cfg or synth.PP_KITTI_CAR)
        cfg = self.cfg
        self.device = torch.device(device)
        self.n = int(num_points or cfg["num_points"])
        self.F = cfg["point_dim"]
        self.test_cfg = dict(test_cfg or cfg["test_cfg"])
        g = _grid(cfg["point_cloud_range"], cfg["voxel_size"])
        self.nx, self.ny = int(g[0]), int(g[1])
        self.net = PillarFeatureNet(self.F, (cfg["pfn_channels"],), False, cfg["max_points"], cfg["voxel_size"],
                                    cfg["point_cloud_range"])
        self.net.init_weight(seed=seed, device=self.device, bn_gain=bn_gain)
        self.dense = SecondRPN(**cfg["backbone"]).init_weight(seed=seed + 1, device=self.device, bn_gain=bn_gain)
        fh, fw = self.dense.out_hw(self.ny, self.nx)
        if tuple(cfg["anchors"]["feature_size"]) != (fh, fw):
            raise ValueError("anchor feature_size %s does not match the FPN output %s" % (cfg["anchors"]["feature_size"],
                                                                                         (fh, fw)))
        self.ssd = SSDHead(self.dense.fpn_channels, cfg["num_classes"], cfg["anchors"]).init_weight(seed + 2, self.device)
        self.ssd.set_mask_grid(cfg["voxel_size"], cfg["point_cloud_range"], (self.nx, self.ny))
        self._init_io(1, rows=max(int(self.test_cfg["nms_post_max_size"]), 1), box_dim=7, count_words=2)

    def _head(self, img):
        """SecondRPN + the SSD conv on the pixel image: (cls, box, dir) fp32 NCHW views."""
        cat, shape = self.dense(*img)
        return self.ssd(cat, shape)

    def _postprocess(self, head, coors, nv):
        from .ops import anchor_head as ah
        tc = self.test_cfg
        return ah.anchor_head_postprocess_device(
            head[0], head[1], head[2], self.ssd.anchors_dev, self.ssd.cells_dev, coors, nv, self.ny, self.nx,
            tc["anchor_area_threshold"], tc["score_threshold"], tc["nms_iou_threshold"], tc["nms_pre_max_size"],
            tc["nms_post_max_size"], tc["post_center_range"])

    # ---- one frame, enqueued on the current stream, device in / device out
    def forward_device(self):
        bev_h16, nv, coors = self._front()
        head = self._head(bev_h16)
        status = sp.status_tensor(self.device).clone()
        boxes, scores, labels, index, counts = self._postprocess(head, coors, nv)
        return dict(bev=None, bev_h16=bev_h16, head=dict(cls=head[0], box=head[1], dir=head[2]), boxes=boxes,
                    scores=scores, labels=labels, anchor_index=index, counts=counts, num_voxels=nv, coors=coors,
                    status=status)

    def anchor_mask(self, coors, num_voxels):
        """The anchor mask of a frame on the host (bool [num_anchors]; None when the test config disables it)."""
        from . import anchor_head
        thr = self.test_cfg["anchor_area_threshold"]
        if thr < 0:
            return None
        occ = anchor_head.occupancy(coors, num_voxels, self.ny, self.nx)
        return anchor_head.anchors_area(occ, self.ssd.cells) > thr

    def calibrate_head(self, points_dev):
        """Shift the cls biases of the (seeded) SSD head so that ~1.4 % of the anchors score above the threshold on this
        frame (SSDHead.calibrate_cls_bias; about 1 500 candidates, more than nms_pre_max_size).  Call before capture()."""
        with torch.cuda.stream(self.stream):
            self.points.copy_(points_dev)
            img, nv, coors = self._front()
            cat, shape = self.dense(*img)
            keep = self.anchor_mask(coors.cpu().numpy(), int(nv.item()))
            self.ssd.calibrate_cls_bias(cat, shape, self.test_cfg["score_threshold"], keep=keep)
        self.stream.synchronize()
        return self

    def export_weights_numpy(self):
        """Weights as plain numpy dicts for the CPU arm (tests/cpu_pointpillars_frame.py)."""
        return dict(pfn=dict(self.net.np), dense=self.dense.export_numpy(), ssd=self.ssd.export_numpy())


class CenterPointSweep:
    """Several frames of a sweep in flight on ONE GPU.

    `lanes` CenterPointHotPath instances share the model (weights, packed images) but own their buffers, workspaces,
    CUDA graph and stream; frames are dealt round-robin.  A frame is a chain of ~70 kernels of very different shapes -
    persistent tensor-core kernels that fill the GPU, and latency-bound ones (voxel hashing, rulebooks, post-processing,
    the tails of every layer) that leave most SMs idle: with a second frame in flight those gaps are filled by the other
    frame's kernels.  Measured on the C3 frame (tools/two_in_flight.py): 602 -> 713 frames/s with two lanes.  The latency
    of one frame does not improve (use CenterPointHotPath.infer for that); results are those of the single-lane pipeline.
    """

    def __init__(self, lanes=2, pipeline_cls=CenterPointHotPath, **kw):
        """pipeline_cls: CenterPointHotPath, CenterPointPillarsHotPath or PointPillarsHotPath; kw go to its constructor."""
        if lanes < 1:
            raise ValueError("lanes >= 1")
        first = pipeline_cls(**kw)
        self.lanes = [first]
        for _ in range(lanes - 1):
            p = pipeline_cls(**kw)
            for name in pipeline_cls.shared_attrs:  # one model: calibration / weight loading happens once, on lane 0
                setattr(p, name, getattr(first, name))
            self.lanes.append(p)
        self.device = first.device

    def __len__(self):
        return len(self.lanes)

    def calibrate_head(self, points_dev):
        self.lanes[0].calibrate_head(points_dev)
        return self

    def capture(self, points_dev, **kw):
        for p in self.lanes:
            p.points.copy_(points_dev)
            p.capture(**kw)
        return self

    def prepare_sweep(self):
        for p in self.lanes:
            p.prepare_sweep()
        return self

    def launch(self, i, points_dev):
        """Frame i of a device-resident sweep: copy into lane i % lanes and replay its graph (asynchronous)."""
        p = self.lanes[i % len(self.lanes)]
        with torch.cuda.stream(p.stream):
            p.points.copy_(points_dev, non_blocking=True)
            p.graph.replay()
        return p

    def synchronize(self):
        for p in self.lanes:
            p.stream.synchronize()

    @staticmethod
    def _lane_slot(i, lanes):
        return i % lanes, (i // lanes) & 1

    @staticmethod
    def plan(n_frames, lanes):
        """The order of operations of infer_many for a sweep of n_frames: ("submit", frame, lane, slot) / ("result", frame,
        lane, slot) tuples.  Frame i runs on lane i % lanes, slot (i // lanes) & 1; at most lanes + 1 frames are
        outstanding, and the result of a frame is always read before its (lane, slot) is submitted again
        (tests/test_sweep_plan.py checks these invariants without a GPU)."""
        import collections
        pending = collections.deque()
        for i in range(n_frames):
            pending.append((i,) + CenterPointSweep._lane_slot(i, lanes))
            yield ("submit",) + pending[-1]
            if len(pending) > lanes:
                yield ("result",) + pending.popleft()
        while pending:
            yield ("result",) + pending.popleft()

    def infer_many(self, frames_host):
        """As CenterPointHotPath.infer_many (pinned host frames in, host results out, in order), with len(self) frames
        computing concurrently: frame i runs on lane i % lanes, slot (i // lanes) & 1 (see plan())."""
        import collections
        L = len(self.lanes)
        for p in self.lanes:
            if p.graph is None:
                raise RuntimeError("infer_many needs captured lanes: call capture() first")
            p.prepare_sweep()
        pending = collections.deque()
        for i, pts in enumerate(frames_host):
            li, k = self._lane_slot(i, L)
            lane = self.lanes[li]
            lane._submit(pts, k, i < 2 * L)
            pending.append((lane, k))
            if len(pending) > L:
                pl, pk = pending.popleft()
                yield pl._result(pk)
        while pending:
            pl, pk = pending.popleft()
            yield pl._result(pk)
