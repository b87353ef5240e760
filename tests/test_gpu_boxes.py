"""GPU parity: iou3d_nms, centerpoint_postprocess, bev_pool_v2 through the C ABI.
Keep lists / labels / indices: bit-exact.  Float outputs: bit-exact against the reference's own CUDA
kernels (their outputs on these seeded inputs: tests/golden/ref_kernels.npz) and within 1e-4 relative of the CPU oracle."""
import ctypes as C

import numpy as np
import pytest

from conftest import golden
from paddle3d_b200 import synth
from parity import digest

pytestmark = pytest.mark.gpu
RTOL = 1e-4  # BASELINE.json north_star tolerance for fp32 quantities


def _t(cuda, a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda)


def _ref_kernel_output(key, *inputs):
    """What the reference's CUDA kernel returned for `key` on `inputs` (tests/golden/make_golden.py
    make_ref_kernels_golden)."""
    g = golden("ref_kernels.npz")
    assert digest(*inputs) == g[key + "_inputs"], "%s: the seeded inputs changed; the stored reference output does not apply" % key
    return g[key]


def test_iou_golden_and_oracle(cuda, oracle_mod):
    from paddle3d_b200.ops import iou3d_nms
    g = golden("iou_bev.npz")
    got = iou3d_nms.boxes_iou_bev_gpu(_t(cuda, g["boxes_a"]), _t(cuda, g["boxes_b"])).cpu().numpy()
    np.testing.assert_allclose(got, g["iou"], rtol=RTOL, atol=1e-6)
    a, b = synth.random_boxes(517, 1), synth.random_boxes(333, 2)
    b[:100] = a[:100] + np.random.default_rng(0).normal(0, 0.3, (100, 7)).astype(np.float32)
    got = iou3d_nms.boxes_iou_bev_gpu(_t(cuda, a), _t(cuda, b)).cpu().numpy()
    np.testing.assert_allclose(got, oracle_mod.boxes_iou_bev(a, b), rtol=RTOL, atol=1e-6)
    got = iou3d_nms.boxes_overlap_bev_gpu(_t(cuda, a), _t(cuda, b)).cpu().numpy()
    np.testing.assert_allclose(got, oracle_mod.boxes_overlap_bev(a, b), rtol=RTOL, atol=1e-5)
    assert iou3d_nms.boxes_iou_bev_gpu(_t(cuda, a[:0]), _t(cuda, b)).shape == (0, 333)


def test_iou_bit_exact_vs_reference_kernels(cuda):
    from paddle3d_b200.ops import iou3d_nms
    a, b = synth.random_boxes(400, 3), synth.random_boxes(400, 3)
    b[:, :2] += 0.4
    ta, tb = _t(cuda, a), _t(cuda, b)
    for mine, theirs in ((iou3d_nms.boxes_iou_bev_gpu, "boxes_iou_bev"), (iou3d_nms.boxes_overlap_bev_gpu, "boxes_overlap_bev")):
        want = _ref_kernel_output(theirs, a, b)
        got = mine(ta, tb).cpu().numpy()
        assert np.array_equal(got, want), "not bit-identical to the reference kernel"


@pytest.mark.parametrize("n,thr,normal", [(1, 0.1, False), (63, 0.2, False), (64, 0.2, False), (65, 0.2, True),
                                          (1000, 0.2, False), (1000, 0.01, False), (1000, 0.7, True), (4096, 0.2, False)])
def test_nms_keep_bit_exact(cuda, oracle_mod, n, thr, normal):
    from paddle3d_b200.ops import iou3d_nms
    boxes = synth.random_boxes(n, 100 + n)
    fn = iou3d_nms.nms_normal_gpu if normal else iou3d_nms.nms_gpu
    keep, num = fn(_t(cuda, boxes), thr)
    want_keep, want_num = oracle_mod.nms(boxes, thr, normal)
    assert keep.dtype.is_floating_point is False and not keep.is_cuda  # CPU int32 like the reference
    assert int(num[0]) == want_num
    assert np.array_equal(keep.numpy()[:want_num], want_keep[:want_num])


def test_nms_mask_bit_exact_vs_reference_kernel(cuda, oracle_mod):
    """Upper-triangle words of our bit-matrix == the reference nms_kernel's, via the greedy result on both."""
    from paddle3d_b200.ops import iou3d_nms
    n = 1000
    boxes = synth.random_boxes(n, 77)
    tb = _t(cuda, boxes)
    m = _ref_kernel_output("nms_mask_1000", boxes)
    keep_ref = np.zeros(n, np.int32)
    nk = oracle_mod.lib().orc_nms_reduce(m.ctypes.data_as(C.c_void_p), n, keep_ref.ctypes.data_as(C.c_void_p))
    keep, num = iou3d_nms.nms_gpu(tb, 0.2)
    assert int(num[0]) == nk and np.array_equal(keep.numpy()[:nk], keep_ref[:nk])
    assert np.array_equal(m, oracle_mod.nms_mask(boxes, 0.2))  # oracle restatement pinned on the reference kernel


def test_nms_normal_mask_vs_reference_kernel(cuda, oracle_mod):
    """nms_normal (axis-aligned IoU, iou3d_nms_kernel.cu:380-434): the reference kernel's bit-matrix equals the
    oracle's, and its greedy reduction equals our nms_normal_gpu keep list."""
    from paddle3d_b200.ops import iou3d_nms
    for n, thr in ((1000, 0.3), (257, 0.05)):
        boxes = synth.random_boxes(n, 500 + n)
        tb = _t(cuda, boxes)
        m = _ref_kernel_output("nms_normal_mask_%d" % n, boxes)
        assert np.array_equal(m, oracle_mod.nms_mask(boxes, thr, True))
        keep_ref = np.zeros(n, np.int32)
        nk = oracle_mod.lib().orc_nms_reduce(m.ctypes.data_as(C.c_void_p), n, keep_ref.ctypes.data_as(C.c_void_p))
        keep, num = iou3d_nms.nms_normal_gpu(tb, thr)
        assert int(num[0]) == nk and np.array_equal(keep.numpy()[:nk], keep_ref[:nk])


@pytest.mark.parametrize("dims", [9, 7])
def test_postprocess_indexed_nms_vs_reference_kernel(cuda, oracle_mod, dims):
    """The indexed NMS of centerpoint_postprocess (centerpoint_postprocess/iou3d_nms_kernel.cu:274-352: boxes fetched
    through index[sorted_index[i]], w/l swapped, angle -theta - pi/2 evaluated in double): the reference kernel's
    bit-matrix must equal the oracle's restatement (orc_cpp_nms_mask), which is what our postprocess is checked against,
    and the greedy reduction of it must equal our p3d_nms on the same re-laid boxes."""
    from paddle3d_b200.ops import iou3d_nms
    rng = np.random.default_rng(dims)
    M, n_sel, n_for = 3000, 1500, 1000
    b7 = synth.random_boxes(M, 11)
    boxes = np.zeros((M, dims), np.float32)
    boxes[:, :6] = b7[:, :6]
    boxes[:, dims - 1] = b7[:, 6]
    if dims == 9:
        boxes[:, 6:8] = rng.normal(size=(M, 2)).astype(np.float32)
    index = rng.choice(M, n_sel, replace=False).astype(np.int32)          # compacted candidate -> cell
    sorted_index = rng.permutation(n_sel).astype(np.int64)                # score order -> candidate
    m = _ref_kernel_output("cpp_nms_mask_%d" % dims, boxes, index, sorted_index)
    want = oracle_mod.cpp_nms_mask(boxes, index, sorted_index, n_for, 0.2)
    assert np.array_equal(m, want), "oracle restatement of the indexed NMS differs from the reference kernel"
    keep_ref = np.zeros(n_for, np.int32)
    nk = oracle_mod.lib().orc_nms_reduce(m.ctypes.data_as(C.c_void_p), n_for, keep_ref.ctypes.data_as(C.c_void_p))
    sel = boxes[index[sorted_index[:n_for]]]
    relaid = np.stack([sel[:, 0], sel[:, 1], sel[:, 2], sel[:, 4], sel[:, 3], sel[:, 5],
                       (-sel[:, dims - 1].astype(np.float64) - 3.141592653589793 / 2).astype(np.float32)], 1)
    keep, num = iou3d_nms.nms_gpu(_t(cuda, relaid), 0.2)
    assert int(num[0]) == nk and np.array_equal(keep.numpy()[:nk], keep_ref[:nk])


def _cpp_args(h, with_velocity=True):
    cfg = synth.CENTERPOINT_TEST_CFG
    return [h["hm"], h["reg"], h["height"], h["dim"], h["vel"], h["rot"], [0.075, 0.075], synth.C3["point_cloud_range"],
            cfg["post_center_limit_range"], synth.label_offsets(), cfg["down_ratio"], cfg["score_threshold"],
            cfg["nms_iou_threshold"], cfg["nms_pre_max_size"], cfg["nms_post_max_size"], with_velocity]


@pytest.mark.parametrize("seed,hm_mean,with_vel", [(0, -5.5, True), (1, -4.0, True), (2, -5.5, False), (3, -20.0, True)])
def test_centerpoint_postprocess(cuda, oracle_mod, seed, hm_mean, with_vel):
    """hm_mean -5.5: ~450 candidates/task; -4.0: ~3.7k (exercises the top-1000 cut); -20: empty tasks (fake rows)."""
    from paddle3d_b200.ops import centerpoint_postprocess as cpp
    h = synth.centerpoint_head_outputs(seed, hm_mean=hm_mean, with_velocity=with_vel)
    args = _cpp_args(h, with_vel)
    wb, ws, wl, wc = oracle_mod.centerpoint_postprocess(*args)
    targs = [[_t(cuda, x) for x in a] if i < 6 else a for i, a in enumerate(args)]
    gb, gs, gl = cpp.centerpoint_postprocess(*targs)
    assert gl.dtype.is_floating_point is False and gl.element_size() == 8  # labels int64
    assert gb.shape == wb.shape
    assert np.array_equal(gl.cpu().numpy(), wl)                     # labels / keep set / order: bit exact
    np.testing.assert_allclose(gs.cpu().numpy(), ws, rtol=RTOL)      # scores (sigmoid): fp32 tolerance
    np.testing.assert_allclose(gb.cpu().numpy(), wb, rtol=RTOL, atol=1e-5)
    _, _, _, counts = cpp.centerpoint_postprocess_device(*targs)
    assert np.array_equal(counts.cpu().numpy()[:-1], wc) and int(counts[-1]) == len(wl)
    if hm_mean < -10:
        assert (ws == -1).all() and (wl == 0).all() and len(wl) == 6


def test_bev_pool_v2(cuda, oracle_mod):
    from paddle3d_b200.ops import bev_pool_v2, bev_pool_v2_backward
    for grid in ((128, 128, 1), (200, 200, 1)):
        b = (-51.2, 51.2) if grid[0] == 128 else (-50.0, 50.0)
        d = synth.bev_pool_inputs(5, grid=grid, bounds=(b, b, (-5.0, 3.0)))
        keys = ["depth", "feat", "ranks_depth", "ranks_feat", "ranks_bev", "interval_lengths", "interval_starts"]
        targs = [_t(cuda, d[k]) for k in keys]
        got = bev_pool_v2.bev_pool_v2(*targs, d["bev_feat_shape"])
        nargs = [d[k] for k in keys]
        want_fma = oracle_mod.bev_pool_v2(*nargs, d["bev_feat_shape"], use_fma=True)
        want = oracle_mod.bev_pool_v2(*nargs, d["bev_feat_shape"], use_fma=False)
        assert np.array_equal(got.cpu().numpy(), want_fma)  # same FMA chain as the reference GPU kernel
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=RTOL, atol=1e-5)
        assert digest(got.cpu().numpy()) == _ref_kernel_output("bev_pool_v2_%d" % grid[0], *nargs), \
            "not bit-identical to the reference bev_pool_v2 kernel"
    # backward: intervals grouped by ranks_feat (QuickCumsumCuda.backward, bevdet_transformer.py:54-66)
    order = np.argsort(d["ranks_feat"], kind="stable")
    rf, rd, rb = d["ranks_feat"][order], d["ranks_depth"][order], d["ranks_bev"][order]
    first = np.ones(len(rf), bool)
    first[1:] = rf[1:] != rf[:-1]
    starts = np.nonzero(first)[0].astype(np.int32)
    lens = np.diff(np.append(starts, len(rf))).astype(np.int32)
    og = np.random.default_rng(1).normal(size=d["bev_feat_shape"]).astype(np.float32)
    dg, fg = bev_pool_v2_backward.bev_pool_v2_bkwd(_t(cuda, og), _t(cuda, d["depth"]), _t(cuda, d["feat"]), _t(cuda, rd),
                                                   _t(cuda, rf), _t(cuda, rb), _t(cuda, lens), _t(cuda, starts))
    wdg, wfg = oracle_mod.bev_pool_v2_bkwd(og, d["depth"], d["feat"], rd, rf, rb, lens, starts, use_fma=True)
    assert np.array_equal(dg.cpu().numpy(), wdg) and np.array_equal(fg.cpu().numpy(), wfg)
    # ... and bit-identical to the reference's own bev_pool_grad_kernel (bev_pool_cuda.cu:46-96) on the entries it
    # writes (it leaves untouched entries of its caller-zeroed outputs alone; ours writes zeros there)
    want = _ref_kernel_output("bev_pool_v2_grad", og, d["depth"], d["feat"], rd, rf, rb, lens, starts)
    assert digest(dg.cpu().numpy(), fg.cpu().numpy()) == want, "not bit-identical to the reference bev_pool_grad_kernel"
    # odd channel count -> scalar path; empty interval list -> zeros
    d2 = synth.bev_pool_inputs(6, C=7, D=20)
    targs = [_t(cuda, d2[k]) for k in keys]
    got = bev_pool_v2.bev_pool_v2(*targs, d2["bev_feat_shape"])
    assert np.array_equal(got.cpu().numpy(), oracle_mod.bev_pool_v2(*[d2[k] for k in keys], d2["bev_feat_shape"], use_fma=True))
    e = [targs[0], targs[1]] + [t[:0] for t in targs[2:]]
    assert not bev_pool_v2.bev_pool_v2(*e, d2["bev_feat_shape"]).any()


def test_nms_callers_on_device(cuda, oracle_mod):
    """rotate_nms_pcdet / class_agnostic_nms / boxes_iou3d_gpu (SURVEY §8a-12) with the real GPU ops underneath; the
    index logic itself is covered on the CPU with the oracle's NMS injected (tests/test_nms_utils.py)."""
    import torch
    from paddle3d_b200.ops import nms_utils
    rng = np.random.default_rng(0)
    boxes = synth.random_boxes(300, 5)
    scores = rng.uniform(size=300).astype(np.float32)
    got = nms_utils.rotate_nms_pcdet(_t(cuda, boxes), _t(cuda, scores), 0.2, 200, 50)
    b = boxes[:, [0, 1, 2, 4, 3, 5, 6]].copy()
    b[:, -1] = -b[:, -1] - np.float32(np.pi / 2)
    order = np.argsort(-scores, kind="stable")[:200]
    keep, n = oracle_mod.nms(b[order], 0.2)
    assert np.array_equal(got.cpu().numpy(), order[keep[:n]][:50])
    a, c = synth.random_boxes(40, 7), synth.random_boxes(30, 8)
    iou = nms_utils.boxes_iou3d_gpu(_t(cuda, a), _t(cuda, c)).cpu().numpy()
    assert iou.shape == (40, 30) and (iou >= 0).all() and (iou <= 1 + 1e-5).all()


def test_voxel_pooling_prepare_v2_on_device(cuda, oracle_mod):
    """a-10 / f-3: frustum points -> sorted ranks + run lengths, bit-exact against the numpy restatement of
    bevdet_transformer.py:230-274 (stable tie order), then chained into bev_pool_v2 (identical BEV tensor)."""
    import torch
    from paddle3d_b200.ops import bev_pool_v2 as bp
    for grid, b in (((128, 128, 1), (-51.2, 51.2)), ((200, 200, 1), (-50.0, 50.0))):
        d = synth.bev_pool_inputs(9, grid=grid, bounds=(b, b, (-5.0, 3.0)))
        coor = d["coor"].copy()
        coor[0, 0, 0, 0, :3] = [[np.nan, 0, 0], [1e30, 0, 0], [-0.3 * d["grid_interval"][0] + d["grid_lower_bound"][0], 0.0, 0.0]]
        want = oracle_mod.voxel_pooling_prepare_v2(coor, d["grid_lower_bound"], d["grid_interval"], d["grid_size"])
        prep = bp.voxel_pooling_prepare_v2(_t(cuda, coor), d["grid_lower_bound"], d["grid_interval"], d["grid_size"])
        got = bp.trim(prep)
        for g, w, name in zip(got, want, ("ranks_bev", "ranks_depth", "ranks_feat", "interval_starts", "interval_lengths")):
            assert np.array_equal(g.cpu().numpy(), w), name
        assert not prep[0][len(want[0]):].any() and not prep[4][len(want[3]):].any()  # capacity tails are zero
        rb, rd, rf, st, ln = got
        bev = bp.bev_pool_v2(_t(cuda, d["depth"]), _t(cuda, d["feat"]), rd, rf, rb, ln, st, d["bev_feat_shape"])
        ref = oracle_mod.bev_pool_v2(d["depth"], d["feat"], want[1], want[2], want[0], want[4], want[3], d["bev_feat_shape"], use_fma=True)
        assert np.array_equal(bev.cpu().numpy(), ref)
    # nothing inside the grid -> the reference's five Nones
    far = np.full((1, 1, 2, 2, 2, 3), 1e6, np.float32)
    assert bp.trim(bp.voxel_pooling_prepare_v2(_t(cuda, far), [-50, -50, -5], [0.5, 0.5, 8], [200, 200, 1])) == (None,) * 5


def test_bev_pool_round1_kernel_still_bit_exact(cuda, oracle_mod, monkeypatch):
    """The float4-per-thread kernel (odd channel counts, C > 256) is still reachable and exact: C = 7 takes the scalar
    path, C = 260 the float4 path."""
    from paddle3d_b200.ops import bev_pool_v2
    keys = ["depth", "feat", "ranks_depth", "ranks_feat", "ranks_bev", "interval_lengths", "interval_starts"]
    for C_ in (7, 260):
        d = synth.bev_pool_inputs(4, C=C_, D=12, H=8, W=10, grid=(32, 32, 1), bounds=((-20, 20), (-20, 20), (-5, 3)))
        got = bev_pool_v2.bev_pool_v2(*[_t(cuda, d[k]) for k in keys], d["bev_feat_shape"])
        want = oracle_mod.bev_pool_v2(*[d[k] for k in keys], d["bev_feat_shape"], use_fma=True)
        assert np.array_equal(got.cpu().numpy(), want)
