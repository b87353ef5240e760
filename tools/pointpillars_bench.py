#!/usr/bin/env python
"""PointPillars, KITTI car, on one GPU (pipeline.PointPillarsHotPath, synth.PP_KITTI_CAR: C2's 20k x 4 points, 0.16 m
pillars on a 496 x 432 grid, 107 136 anchors), measured in one run:

  * frames/s with 1 and 4 lanes: a device-resident pool of 32 distinct frames, CUDA-graph replay per frame
    (bench.measure, the timing of bench.py's `value`);
  * e2e frames/s through infer_many (pinned host frames, H2D + graph + D2H per frame) and the one-frame latency of infer;
  * the split of one frame into voxelize, PFN -> pixel image, trunk + SSD conv and anchor post-processing (CUDA events
    around an eager frame, the host enqueues the whole frame before the GPU starts);
  * p3d_anchor_head_postprocess against the composed path it replaces (torch decode + nms_utils.rotate_nms_pcdet over
    p3d_nms + direction fix + range filter, with that path's host synchronisations) on the same head tensors: the
    calibrated frame's, and the worst case where every anchor is a candidate;
  * the algorithmic FLOPs of the dense part, from the layer geometry.

    python tools/pointpillars_bench.py [--steps 400] [--warmup 40] [--out profiles/r04_pointpillars_bench.json]

Prints one JSON line (and writes it to --out).  Needs a CUDA device."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from pillars_bench import gpu_info  # noqa: E402


def dense_flops(rpn, ssd, H, W):
    """Algorithmic FLOPs (2 x MACs) of SecondBackbone + SecondFPN and of the SSD conv on an H x W image:
    (trunk, head)."""
    total, h, w, shapes = 0.0, H, W, []
    for blk in rpn.blocks:
        for c in blk:
            h, w = (h + 2 * c.padding - c.k) // c.stride + 1, (w + 2 * c.padding - c.k) // c.stride + 1
            total += 2.0 * h * w * c.cin * c.cout * c.k * c.k
        shapes.append((1, h, w, blk[-1].cout))
    for (_, h, w, _), de in zip(shapes, rpn.deblocks):
        oh, ow = rpn.deblock_out_hw(de, h, w)
        total += 2.0 * oh * ow * de.cin * de.cout * (1 if de.up > 1 else de.k * de.k)
    oh, ow = rpn.fpn_out_hw(shapes)
    return total, 2.0 * oh * ow * ssd.conv.cin * ssd.conv.cout


def stage_split(pipe, frame, reps):
    """Per-stage device times (ms, median over reps) of one eager frame."""
    import torch
    from paddle3d_b200.ops import voxelize as vox
    cfg, st = pipe.cfg, pipe.stream
    names = ["voxelize", "pfn_to_pixel_image", "trunk_and_ssd_conv", "anchor_postprocess"]
    runs = {k: [] for k in names}
    for rep in range(reps + 1):
        with torch.cuda.stream(st):
            pipe.points.copy_(frame)
            torch.cuda._sleep(int(2e7))  # the host enqueues the whole frame first: events bracket back-to-back kernels
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record(st)
            voxels, coords, npv, nv = vox.hard_voxelize(pipe.points, cfg["voxel_size"], cfg["point_cloud_range"],
                                                        cfg["max_points"], cfg["max_voxels"])
            coors = torch.nn.functional.pad(coords, (1, 0), value=0)
            ev[1].record(st)
            img = pipe.net.forward_pixel_h16(voxels, npv, coors, 1, pipe.ny, pipe.nx, num=nv)
            ev[2].record(st)
            head = pipe._head(img)
            ev[3].record(st)
            pipe._postprocess(head, coors, nv)
            ev[4].record(st)
        ev[4].synchronize()
        if rep:  # the first pass warms the allocator
            for k in range(4):
                runs[names[k]].append(ev[k].elapsed_time(ev[k + 1]))
    return {k: statistics.median(v) for k, v in runs.items()}, int(nv.item())


def postprocess_race(pipe, head, coors, nv, rounds, iters):
    """The fused post-processing (graph of `iters` launches, device time) against the composed path (host clock around
    `iters` synchronised calls: it reads counts back to the host and cannot be captured), alternately, `rounds` times.
    Returns medians in us and whether the two give the same boxes, scores, labels and anchor indices."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_pointpillars import _composed
    tc, st = pipe.test_cfg, pipe.stream
    keep = torch.from_numpy(pipe.anchor_mask(coors.cpu().numpy(), int(nv.item()))).to(pipe.device)

    def fused():
        return pipe._postprocess(head, coors, nv)

    def composed():
        return _composed(*head, pipe.ssd.anchors_dev, keep, tc)

    with torch.cuda.stream(st):
        b, s, l, idx, cnt = fused()
        k = int(cnt[1])
        got = (b[:k], s[:k], l[:k], idx[:k].long())
        want = composed()
        equal = all(torch.equal(g, w) for g, w in zip(got, want[:4]))
        cand = int(cnt[0])
    t_f, t_c = [], []
    for _ in range(rounds):
        t_f.append(1e3 * bench.graph_time_ms(fused, st, iters))
        with torch.cuda.stream(st):
            composed()
            st.synchronize()
            t0 = time.perf_counter()
            for _ in range(iters):
                composed()
            st.synchronize()
        t_c.append(1e6 * (time.perf_counter() - t0) / iters)
    return {"fused_us": statistics.median(t_f), "composed_us": statistics.median(t_c), "fused_us_all": t_f,
            "composed_us_all": t_c, "outputs_bit_equal": equal, "candidates": cand, "boxes": k, "rounds": rounds,
            "calls_per_round": iters}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--lanes", default="1,4")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    from paddle3d_b200 import synth
    from paddle3d_b200.pipeline import PILLARS_BN_GAIN, CenterPointSweep, PointPillarsHotPath
    if not torch.cuda.is_available():
        raise SystemExit("pointpillars_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    cfg = synth.PP_KITTI_CAR
    frames = bench.frame_pool(cfg, bench.POOL)
    dev_frames = [torch.from_numpy(f).to(dev) for f in frames]
    host_frames = [torch.from_numpy(f).pin_memory() for f in frames]
    res = {"model": "PointPillars KITTI car (synth.PP_KITTI_CAR): 20k x 4 points, 496 x 432 pillars, max 40000, P 32, "
                    "107136 anchors",
           "gpu": gpu_info(), "torch_device_name": torch.cuda.get_device_name(dev), "bn_gain": PILLARS_BN_GAIN,
           "frames_in_pool": bench.POOL, "l2": "input pool 10 MB (fits the 126 MB L2); no explicit flush",
           "steps": args.steps, "warmup": args.warmup, "sweep": {}}
    first = None
    for L in [int(x) for x in args.lanes.split(",")]:
        sweep = CenterPointSweep(L, pipeline_cls=PointPillarsHotPath, cfg=cfg, device=dev, seed=0)
        sweep.calibrate_head(dev_frames[0])
        sweep.capture(dev_frames[0], count_nodes=True)
        m = bench.measure(sweep, dev_frames, host_frames, argparse.Namespace(steps=args.steps, warmup=args.warmup), 1, None,
                          False, 0)
        res["sweep"]["lanes_%d" % L] = {"frames_per_s": m["value"], "ms_per_frame": m["ms_per_step"],
                                        "e2e_infer_many_frames_per_s": m["e2e_value"],
                                        "infer_one_frame_latency_ms": 1e3 / m["e2e_sync_value"]}
        if first is None:
            first = sweep.lanes[0]
            res["graph_nodes"] = first.graph_nodes
        else:
            del sweep
    pipe = first
    res["stage_ms"], res["num_voxels_frame0"] = stage_split(pipe, dev_frames[0], 20)
    res["stage_note"] = "eager frame, CUDA events between stages, median of 20; the graph replays the same kernels"
    with torch.cuda.stream(pipe.stream):
        pipe.points.copy_(dev_frames[0])
        img, nv, coors = pipe._front()
        head = pipe._head(img)
    res["postprocess_frame"] = postprocess_race(pipe, head, coors, nv, 7, 20)
    # worst case: every anchor a candidate (logits far above the threshold), no anchor mask
    worst = tuple(t.clone() for t in head)
    worst[0].fill_(6.0)
    tc0 = pipe.test_cfg
    pipe.test_cfg = dict(tc0, anchor_area_threshold=-1)
    res["postprocess_all_anchors"] = postprocess_race(pipe, worst, coors, nv, 3, 5)
    pipe.test_cfg = tc0
    res["postprocess_note"] = ("fused: CUDA graph of the kernel chain, device time per call; composed: torch decode + "
                               "rotate_nms_pcdet over p3d_nms + direction fix + range filter, host clock around "
                               "synchronised calls (it synchronises with the host, so it cannot be captured)")
    trunk, ssd = dense_flops(pipe.dense, pipe.ssd, pipe.ny, pipe.nx)
    ms = bench.graph_time_ms(lambda: pipe._head(img), pipe.stream, 5)
    res["dense"] = {"algorithmic_gflop_trunk": trunk / 1e9, "algorithmic_gflop_ssd_conv": ssd / 1e9, "ms_graph": ms,
                    "achieved_tflops": (trunk + ssd) / (ms * 1e-3) / 1e12,
                    "note": "2 x MACs of the convolutions from the layer geometry; the fp16-pair kernels execute 3 fp16 "
                            "MMAs per product"}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
