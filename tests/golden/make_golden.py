"""Generate the committed golden fixtures from the REFERENCE ITSELF (run in the build container only;
/root/reference does not exist on the GPU box, the .npz files do).

  voxelize_*.npz   outputs of the reference's own hard_voxelize_cpu (voxelize_op.cc:84-146, compiled
                   unmodified into oracle/_ref/libp3d_ref_cpu.so) AND of the reference's numba
                   points_to_voxel (paddle3d/transforms/functional.py:118-150, AST-extracted and exec'd —
                   importing the package would import paddle) on seeded inputs; the two must agree.
  iou_bev.npz      boxes_iou_bev_cpu (iou3d_cpu.cpp:241-264, compiled unmodified).
  sweeps.npz       LoadPointCloud.__call__ (paddle3d/transforms/reader.py:116-167, AST-extracted: importing the module
                   would import paddle) on three seeded .bin files; stores the files' contents, the transforms, the
                   sweep order the reference's np.random.choice drew and the merged cloud.
  ref_kernels.npz  what the reference's own CUDA kernels returned on the seeded inputs of tests/test_gpu_boxes.py (see
                   make_ref_kernels_golden); written separately, on a machine with a GPU.

Usage: python tests/golden/make_golden.py [ref_kernels]
"""
import ast
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from paddle3d_b200 import synth  # noqa: E402

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))


def numba_points_to_voxel():
    import numba  # noqa: F401
    src = open(os.path.join(REF, "paddle3d/transforms/functional.py")).read()
    tree = ast.parse(src)
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "points_to_voxel"][0]
    code = ast.get_source_segment(src, fn)
    ns = {"numba": __import__("numba"), "np": np}
    exec(code, ns)
    return ns["points_to_voxel"]


def run_numba(fn, pts, cfg, P, V):
    vs = np.asarray(cfg["voxel_size"], np.float32)
    pcr = np.asarray(cfg["point_cloud_range"], np.float32)
    grid = np.round((pcr[3:] - pcr[:3]) / vs).astype(np.int32)
    voxels = np.zeros((V, P, pts.shape[1]), np.float32)
    coords = np.zeros((V, 3), np.int32)
    npv = np.zeros((V,), np.int32)
    g2v = np.full(tuple(grid[::-1]), -1, np.int32)
    nv = fn(pts, vs, pcr, grid, voxels, coords, npv, g2v, P, V)
    return voxels, coords, npv, np.array([nv], np.int32)


def reference_load_point_cloud():
    """The reference's LoadPointCloud class body (methods only), exec'd without its paddle-importing module."""
    src = open(os.path.join(REF, "paddle3d/transforms/reader.py")).read()
    tree = ast.parse(src)
    cls = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "LoadPointCloud"][0]
    code = "class LoadPointCloud:\n" + "\n".join(
        "    " + line for fn in cls.body if isinstance(fn, ast.FunctionDef)
        for line in ast.get_source_segment(src, fn).splitlines())
    import typing
    ns = {"np": np, "Union": typing.Union, "List": typing.List, "Sample": object, "PointCloud": lambda x: x}
    exec(code, ns)
    return ns["LoadPointCloud"]


def make_sweeps_golden():
    import tempfile
    from types import SimpleNamespace as NS
    rng = np.random.default_rng(21)
    clouds = [np.concatenate([rng.uniform(-3, 3, size=(n, 3)), rng.uniform(0, 255, size=(n, 1)),
                              rng.integers(0, 32, size=(n, 1))], 1).astype(np.float32) for n in (500, 400, 300, 350)]
    mats, lags = [], [0.05, 0.1, 0.15]
    for k in range(3):
        a = 0.01 * (k + 1)
        m = np.eye(4)
        m[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
        m[:3, 3] = [0.3 * (k + 1), -0.1 * k, 0.02]
        mats.append(m)
    mats[1] = None  # a sweep without transform
    with tempfile.TemporaryDirectory() as d:
        paths = []
        for i, c in enumerate(clouds):
            paths.append(os.path.join(d, "c%d.bin" % i))
            c.tofile(paths[-1])
        sweeps = [NS(path=paths[i + 1], meta=NS(ref_from_curr=mats[i], time_lag=lags[i])) for i in range(3)]
        sample = NS(modality="lidar", data=None, path=paths[0], sweeps=sweeps)
        cls = reference_load_point_cloud()
        np.random.seed(1)
        order = np.random.choice(3, 3, replace=False)  # what the call below will draw
        np.random.seed(1)
        out = cls(dim=5, use_dim=[0, 1, 2, 4], use_time_lag=True, sweep_remove_radius=1)(sample).data
    np.savez_compressed(os.path.join(HERE, "sweeps.npz"), cloud0=clouds[0], cloud1=clouds[1], cloud2=clouds[2],
                        cloud3=clouds[3], mat0=mats[0], mat2=mats[2], lags=np.asarray(lags), order=order, merged=out)
    print("sweeps", out.shape, out.dtype, "order", order)


def main():
    oracle.build(ref=True)
    make_sweeps_golden()
    p2v = numba_points_to_voxel()
    cases = {
        # name: (cfg, generator, seed, num_points, max_points, max_voxels)
        "c1_uniform": (synth.C1, synth.uniform_cloud, 0, 1000, 32, 40000),
        "c1_dense": (synth.C1, "dense", 5, 1000, 5, 120),                      # many points per cell, cap, P overflow
        "c1_cap": (synth.C1, synth.uniform_cloud, 1, 1000, 2, 300),            # hits the max_voxels cap
        "c2_lidar_small": (synth.C2, synth.lidar_cloud, 2, 4000, 4, 1500),     # over-full cells + cap
        "c3_lidar_small": (synth.C3, synth.lidar_cloud, 3, 6000, 3, 5000),
    }
    for name, (cfg, gen, seed, n, P, V) in cases.items():
        if gen == "dense":
            rng = np.random.default_rng(seed)
            pts = np.concatenate([rng.normal([30, 0, -1], [1.0, 1.0, 0.5], size=(n, 3)), rng.uniform(0, 1, (n, 1))], 1).astype(np.float32)
        else:
            pts = gen(cfg, seed, num_points=n)
        if name == "c2_lidar_small":
            pts = pts[(pts[:, 0] > 0)][:n]
        ref = oracle.ref_hard_voxelize_cpu(pts, cfg["voxel_size"], cfg["point_cloud_range"], P, V)
        nb = run_numba(p2v, pts, cfg, P, V)
        for a, b in zip(ref, nb):
            assert np.array_equal(a, b), "reference C++ and numba voxelizers disagree on %s" % name
        np.savez_compressed(os.path.join(HERE, "voxelize_%s.npz" % name), points=pts,
                            voxel_size=np.asarray(cfg["voxel_size"], np.float32),
                            point_cloud_range=np.asarray(cfg["point_cloud_range"], np.float32),
                            max_points=P, max_voxels=V, voxels=ref[0], coords=ref[1], num_points_per_voxel=ref[2],
                            num_voxels=ref[3])
        print(name, "num_voxels", int(ref[3][0]), "max npv", int(ref[2].max()))
    a = synth.random_boxes(96, 11)
    rng = np.random.default_rng(12)
    b = a[rng.permutation(96)[:80]].copy()
    b[:, :2] += rng.normal(0, 0.8, size=(80, 2)).astype(np.float32)
    b[:, 6] += rng.normal(0, 0.4, size=80).astype(np.float32)
    b[:8] = a[:8]  # identical boxes
    b[8:16] = a[8:16]
    b[8:16, 6] += 1e-3  # nearly identical
    iou = oracle.ref_boxes_iou_bev_cpu(a, b)
    np.savez_compressed(os.path.join(HERE, "iou_bev.npz"), boxes_a=a, boxes_b=b, iou=iou)
    print("iou_bev", iou.shape, "nonzero", float((iou > 0).mean()))


def make_ref_kernels_golden():
    """ref_kernels.npz: the outputs of the reference's CUDA kernels (iou3d_nms_kernel.cu, centerpoint_postprocess/
    iou3d_nms_kernel.cu, bev_pool_cuda.cu; compiled unmodified into oracle/_ref) on the seeded inputs of
    tests/test_gpu_boxes.py, so that those tests need no reference build.  Each entry `k` comes with `k_inputs`, the
    parity.digest of the inputs it was computed from; bev_pool_v2 outputs (megabytes) are stored as digests too.

    The values are written from the two implementations that the GPU suite found bit-identical to the reference kernels
    on exactly these inputs (commit d310766 on a B200: 144 passed, none skipped, every oracle/_ref build loaded): the
    oracle for the NMS bit-matrices and bev_pool_v2 forward / backward, and this repository's boxes_iou_bev /
    boxes_overlap_bev kernels for the IoU matrices.  Regenerate only from code that still passes against the reference
    build."""
    import torch
    sys.path.insert(0, os.path.dirname(HERE))
    from parity import digest
    from paddle3d_b200.ops import iou3d_nms
    oracle.build(ref=False)
    out = {}

    def case(key, value, *inputs):
        out[key] = value
        out[key + "_inputs"] = np.array(digest(*inputs))

    a, b = synth.random_boxes(400, 3), synth.random_boxes(400, 3)
    b[:, :2] += 0.4
    ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    case("boxes_iou_bev", iou3d_nms.boxes_iou_bev_gpu(ta, tb).cpu().numpy(), a, b)
    case("boxes_overlap_bev", iou3d_nms.boxes_overlap_bev_gpu(ta, tb).cpu().numpy(), a, b)
    boxes = synth.random_boxes(1000, 77)
    case("nms_mask_1000", oracle.nms_mask(boxes, 0.2), boxes)
    for n, thr in ((1000, 0.3), (257, 0.05)):
        boxes = synth.random_boxes(n, 500 + n)
        case("nms_normal_mask_%d" % n, oracle.nms_mask(boxes, thr, True), boxes)
    for dims in (9, 7):  # the indexed NMS of centerpoint_postprocess
        rng = np.random.default_rng(dims)
        M, n_sel, n_for = 3000, 1500, 1000
        b7 = synth.random_boxes(M, 11)
        boxes = np.zeros((M, dims), np.float32)
        boxes[:, :6] = b7[:, :6]
        boxes[:, dims - 1] = b7[:, 6]
        if dims == 9:
            boxes[:, 6:8] = rng.normal(size=(M, 2)).astype(np.float32)
        index = rng.choice(M, n_sel, replace=False).astype(np.int32)
        sorted_index = rng.permutation(n_sel).astype(np.int64)
        case("cpp_nms_mask_%d" % dims, oracle.cpp_nms_mask(boxes, index, sorted_index, n_for, 0.2), boxes, index, sorted_index)
    keys = ["depth", "feat", "ranks_depth", "ranks_feat", "ranks_bev", "interval_lengths", "interval_starts"]
    for grid in ((128, 128, 1), (200, 200, 1)):
        bd = (-51.2, 51.2) if grid[0] == 128 else (-50.0, 50.0)
        d = synth.bev_pool_inputs(5, grid=grid, bounds=(bd, bd, (-5.0, 3.0)))
        nargs = [d[k] for k in keys]
        case("bev_pool_v2_%d" % grid[0], np.array(digest(oracle.bev_pool_v2(*nargs, d["bev_feat_shape"], use_fma=True))),
             *nargs)
    # backward on the 200 x 200 inputs, intervals grouped by ranks_feat
    order = np.argsort(d["ranks_feat"], kind="stable")
    rf, rd, rb = d["ranks_feat"][order], d["ranks_depth"][order], d["ranks_bev"][order]
    first = np.ones(len(rf), bool)
    first[1:] = rf[1:] != rf[:-1]
    starts = np.nonzero(first)[0].astype(np.int32)
    lens = np.diff(np.append(starts, len(rf))).astype(np.int32)
    og = np.random.default_rng(1).normal(size=d["bev_feat_shape"]).astype(np.float32)
    dg, fg = oracle.bev_pool_v2_bkwd(og, d["depth"], d["feat"], rd, rf, rb, lens, starts, use_fma=True)
    case("bev_pool_v2_grad", np.array(digest(dg, fg)), og, d["depth"], d["feat"], rd, rf, rb, lens, starts)
    np.savez_compressed(os.path.join(HERE, "ref_kernels.npz"), **out)
    print("ref_kernels", sorted(k for k in out if not k.endswith("_inputs")))


if __name__ == "__main__":
    if sys.argv[1:] == ["ref_kernels"]:
        make_ref_kernels_golden()
    else:
        main()
