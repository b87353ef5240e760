"""PointPillars (KITTI car) without a GPU: the anchors and their (y, x, a) order, the static cell bounds of the anchor mask
against a brute-force restatement of fused_get_anchors_area, the integral-image area against a direct count, the trunk /
SSD head geometry, the numpy post-processing at a tiny size, and the host-side checks of p3d_anchor_head_postprocess
(every call below is rejected before any CUDA call)."""
import ctypes as C
import math

import numpy as np
import pytest

from paddle3d_b200 import anchor_head as ah
from paddle3d_b200 import synth

CFG = synth.PP_KITTI_CAR
GRID = (432, 496)  # (nx, ny) of C2's 0.16 m pillars


def _anchors():
    return ah.create_anchors_3d_stride(**CFG["anchors"])


def test_anchor_count_values_and_order():
    a = _anchors()
    assert a.shape == (248 * 216 * 2, 7) == (107136, 7) and a.dtype == np.float32
    f32 = np.float32
    for y, x, r in ((0, 0, 0), (0, 0, 1), (0, 1, 0), (1, 0, 1), (123, 77, 1), (247, 215, 0), (247, 215, 1)):
        i = (y * 216 + x) * 2 + r
        want = [f32(x) * f32(0.32) + f32(0.16), f32(y) * f32(0.32) + f32(-39.52), f32(-1.78), f32(1.6), f32(3.9), f32(1.56),
                f32((0, 1.57)[r])]
        assert a[i].tolist() == [float(v) for v in want], (y, x, r)
    assert a[-1, 0] == pytest.approx(68.96, abs=1e-4) and a[-1, 1] == pytest.approx(39.52, abs=1e-4)


def _near_bbox_one(x, y, w, l, r):
    """rbbox2d_to_near_bbox for one box, scalar fp32 arithmetic."""
    f32 = np.float32
    r = f32(r)
    lim = r - f32(math.floor(float(r / f32(np.pi) + f32(0.5)))) * f32(np.pi)
    if abs(lim) > f32(np.pi / 4):
        w, l = l, w
    return (f32(x) - f32(w) / f32(2), f32(y) - f32(l) / f32(2), f32(x) + f32(w) / f32(2), f32(y) + f32(l) / f32(2))


def _fused_cells_one(bv, vs, off, grid):
    """fused_get_anchors_area's corner computation for one anchor (numba-style scalar loop, fp32)."""
    f32 = np.float32
    c = [int(math.floor(float((f32(bv[0]) - f32(off[0])) / f32(vs[0])))),
         int(math.floor(float((f32(bv[1]) - f32(off[1])) / f32(vs[1])))),
         int(math.floor(float((f32(bv[2]) - f32(off[0])) / f32(vs[0])))),
         int(math.floor(float((f32(bv[3]) - f32(off[1])) / f32(vs[1]))))]
    return [max(c[0], 0), max(c[1], 0), min(c[2], grid[0] - 1), min(c[3], grid[1] - 1)]


def test_cell_bounds_against_brute_force():
    a = _anchors()
    cells = ah.anchor_cells(a, CFG["voxel_size"], CFG["point_cloud_range"], GRID)
    assert cells.shape == (len(a), 4) and cells.dtype == np.int32
    rng = np.random.default_rng(0)
    idx = set(rng.integers(0, len(a), 300).tolist())
    for y in (0, 247):            # anchors clipped at the y edges ...
        for x in (0, 1, 107, 214, 215):
            idx.update({(y * 216 + x) * 2, (y * 216 + x) * 2 + 1})
    for x in (0, 215):            # ... and at the x edges
        for y in (0, 5, 130, 246):
            idx.update({(y * 216 + x) * 2, (y * 216 + x) * 2 + 1})
    for i in sorted(idx):
        x, y, _, w, l, _, r = a[i]
        want = _fused_cells_one(_near_bbox_one(x, y, w, l, r), CFG["voxel_size"], CFG["point_cloud_range"], GRID)
        assert cells[i].tolist() == want, i
    # all four edges clip somewhere, and the 1.57 rotation swaps w and l (3.9 m along x, 1.6 m along y)
    assert (cells[:, 0] == 0).any() and (cells[:, 1] == 0).any()
    assert (cells[:, 2] == GRID[0] - 1).any() and (cells[:, 3] == GRID[1] - 1).any()
    mid = (100 * 216 + 100) * 2
    span = cells[mid:mid + 2, 2:] - cells[mid:mid + 2, :2]
    assert span[0, 0] < span[0, 1] and span[1, 0] > span[1, 1]


def test_integral_area_against_direct_count():
    rng = np.random.default_rng(1)
    ny, nx = 37, 29
    for p in (0.0, 0.1, 0.6):
        occ = (rng.random((ny, nx)) < p).astype(np.int32)
        cells = np.stack([rng.integers(0, nx, 200), rng.integers(0, ny, 200)], 1)
        cells = np.concatenate([cells, np.minimum(cells + rng.integers(0, 9, (200, 2)), [nx - 1, ny - 1])], 1).astype(np.int32)
        got = ah.anchors_area(occ, cells)
        # the exclusive-min corner: rows y0 + 1 .. y1 and columns x0 + 1 .. x1
        want = [occ[y0 + 1:y1 + 1, x0 + 1:x1 + 1].sum() for x0, y0, x1, y1 in cells]
        assert got.tolist() == want
    coors = np.array([[0, 0, 3, 4], [0, 0, 36, 28], [0, 0, 40, 1], [0, 0, 0, 0]], np.int32)
    occ = ah.occupancy(coors, 3, ny, nx)
    assert occ.sum() == 2 and occ[3, 4] == 1 and occ[36, 28] == 1  # outside rows skipped, rows >= num_voxels ignored


def test_trunk_and_ssd_geometry():
    from paddle3d_b200.dense_head import SecondRPN
    rpn = SecondRPN(**CFG["backbone"]).init_weight(seed=1, device=None)
    assert [len(b) for b in rpn.blocks] == [4, 6, 6]
    assert [(d.k, d.stride, d.up, d.cin, d.cout) for d in rpn.deblocks] == [(1, 1, 1, 64, 128), (2, 2, 2, 128, 128),
                                                                            (4, 4, 4, 256, 128)]
    assert rpn.out_hw(496, 432) == (248, 216) and rpn.fpn_channels == 384
    head = ah.SSDHead(rpn.fpn_channels, CFG["num_classes"], CFG["anchors"]).init_weight(seed=2, device=None)
    assert (head.A, head.C, head.planes) == (2, 1, 20) and head.num_anchors == 107136
    assert head.conv.np["weight"].shape == (20, 384, 1, 1) and head.conv.np["bias"].shape == (20,)
    planes = np.arange(20 * 6).reshape(1, 20, 2, 3)
    cls, box, dir = head.split(planes)
    assert cls.shape[1] == 2 and box.shape[1] == 14 and dir.shape[1] == 4
    assert cls[0, 0, 0, 0] == 0 and box[0, 0, 0, 0] == 12 and dir[0, 0, 0, 0] == 96
    multi = ah.SSDHead(384, 3, dict(CFG["anchors"], sizes=(1.6, 3.9, 1.56, 0.6, 0.8, 1.73, 0.6, 1.76, 1.73),
                                    feature_size=(4, 5)))
    assert (multi.A, multi.C, multi.planes, multi.num_anchors) == (6, 3, 72, 4 * 5 * 6)
    with pytest.raises(ValueError):
        ah.SSDHead(384, 1, dict(CFG["anchors"], rotations=(0,)))  # 10 planes: below the fp16-pair conv's 16


def test_numpy_postprocess_tiny(oracle_mod):
    """The numpy restatement end to end on a 6 x 5 map with A = 2: threshold, order, NMS, direction fix, range filter."""
    from cpu_pointpillars_frame import anchor_postprocess_np
    rng = np.random.default_rng(3)
    H, W, A = 6, 5, 2
    anchors = ah.create_anchors_3d_stride((H, W), (1.6, 3.9, 1.56), (2.0, 2.0, 0.0), (1.0, -5.0, -1.78), (0, 1.57))
    cls = rng.normal(0, 2, (1, A, H, W)).astype(np.float32)
    box = rng.normal(0, 0.3, (1, 7 * A, H, W)).astype(np.float32)
    dir = rng.normal(0, 1, (1, 2 * A, H, W)).astype(np.float32)
    r = anchor_postprocess_np(cls, box, dir, anchors, None, None, 0, 0, 0, -1, 0.3, 0.5, 1000, 300, None, oracle_mod.nms)
    s = 1 / (1 + np.exp(-cls[0].reshape(A, -1).T.reshape(-1)))
    assert r["candidates"] == int((s >= np.float32(0.3)).sum()) > 0
    assert np.all(np.diff(r["scores"]) <= 0) and len(r["index"]) <= r["candidates"]
    r2 = anchor_postprocess_np(cls, box, dir, anchors, None, None, 0, 0, 0, -1, 0.3, 0.5, 1000, 300,
                               [0, -5, -5, 5, 5, 5], oracle_mod.nms)
    assert np.all(r2["boxes"][:, 0] >= 0) and np.all(r2["boxes"][:, 0] <= 5) and set(r2["index"]) <= set(r["index"])
    none = anchor_postprocess_np(cls - 100, box, dir, anchors, None, None, 0, 0, 0, -1, 0.3, 0.5, 1000, 300, None,
                                 oracle_mod.nms)
    assert none["candidates"] == 0 and len(none["boxes"]) == 0


def test_anchor_postprocess_argument_checks():
    from paddle3d_b200 import _lib
    L = _lib.lib()
    q = L.p3d_anchor_head_postprocess_workspace_bytes
    assert q(107136, 496, 432, 1000) > 107136 * 16
    assert q(107136, 0, 0, 1000) > 0  # no anchor mask: no occupancy image
    assert q(0, 496, 432, 1000) == 0 and q(-5, 496, 432, 1000) == 0 and q(107136, -1, 432, 1000) == 0
    assert q(107136, 496, 432, 0) == 0 and q(1 << 30, 1, 1, 10) == 0
    f = L.p3d_anchor_head_postprocess
    p = C.c_void_p(256)
    odd = C.c_void_p(260)

    def call(cls=p, H=248, W=216, A=2, Cc=1, cells=p, coors=p, nv=p, ny=496, nx=432, thr=1.0, pre=1000, post=300, out=p,
             ws=p, nbytes=1 << 40):
        return f(cls, p, p, H, W, A, Cc, p, cells, coors, nv, ny, nx, thr, 0.05, 0.5, pre, post, None, out, p, p, None, p,
                 ws, nbytes, None)

    assert call(cls=None) == -1
    assert call(out=None) == -1
    assert call(ws=None) == -1
    assert call(H=0) == -1 and call(A=0) == -1 and call(Cc=0) == -1
    assert call(pre=0) == -1 and call(post=-1) == -1
    assert call(coors=None) == -1 and call(nv=None) == -1 and call(ny=0) == -1  # the mask needs the frame's pillars
    assert call(coors=odd) == -1 and call(cells=odd) == -1
    assert call(nbytes=1024) == -2
    assert call(H=1 << 14, W=1 << 14, A=4) == -4


def test_host_mirror_rejects_cpu_tensors():
    import torch
    from paddle3d_b200 import _lib
    from paddle3d_b200.ops import anchor_head as oah
    z = torch.zeros
    with pytest.raises(_lib.P3DError):
        oah.anchor_head_postprocess(z(1, 2, 4, 4), z(1, 14, 4, 4), z(1, 4, 4, 4), z(32, 7), None, None, None, 0, 0, -1,
                                    0.05, 0.5, 100, 10)
