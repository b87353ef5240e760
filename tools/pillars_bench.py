#!/usr/bin/env python
"""CenterPoint-pillars on one GPU (pipeline.CenterPointPillarsHotPath, synth.CP_PILLARS: 300k x 5 points, 0.2 m pillars on
a 512 x 512 grid), measured in one run:

  * frames/s with 1 and 4 lanes: a device-resident pool of 32 distinct frames (32 x 6 MB, more than the 126 MB L2),
    CUDA-graph replay per frame (bench.measure, the timing of bench.py's `value`);
  * e2e frames/s through infer_many (pinned host frames, H2D + graph + D2H per frame) and the one-frame latency of infer;
  * the split of one frame into voxelize, PFN -> pixel image, dense RPN / neck / head and postprocess (CUDA events around
    an eager frame, the host enqueues the whole frame before the GPU starts);
  * the fused encoder against the three launches it replaces (pillar_feature_net + pillar_scatter + nchw_to_pixel_h16),
    each captured in a CUDA graph and timed alternately;
  * the algorithmic FLOPs of the dense part, from the layer geometry.

    python tools/pillars_bench.py [--steps 400] [--warmup 40] [--out profiles/r03_pillars_bench.json]

Prints one JSON line (and writes it to --out).  Needs a CUDA device."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def dense_flops(head, H, W):
    """Algorithmic FLOPs (2 x MACs) of the dense RPN / neck / CenterHead on an H x W BEV image, from each layer's
    geometry (down-sampling, 1x1 and transposed deblocks alike)."""
    total, h, w, shapes = 0.0, H, W, []
    for blk in head.blocks:
        for c in blk:
            h, w = (h + 2 * c.padding - c.k) // c.stride + 1, (w + 2 * c.padding - c.k) // c.stride + 1
            total += 2.0 * h * w * c.cin * c.cout * c.k * c.k
        shapes.append((1, h, w, blk[-1].cout))
    for (_, h, w, _), de in zip(shapes, head.deblocks):
        oh, ow = head.deblock_out_hw(de, h, w)
        # a transposed conv with kernel = stride: every output pixel takes one tap; a conv: k x k taps
        total += 2.0 * oh * ow * de.cin * de.cout * (1 if de.up > 1 else de.k * de.k)
    oh, ow = head.fpn_out_hw(shapes)
    total += 2.0 * oh * ow * head.shared.cin * head.shared.cout * 9
    for hs in head.heads:
        for _, a, f in hs:
            total += 2.0 * oh * ow * (a.cin * a.cout + f.cin * f.cout) * 9
    return total


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001  (the torch name below still identifies the card)
        return {"error": repr(e)}


def stage_split(pipe, frame, reps):
    """Per-stage device times (ms, median over reps) of one eager frame."""
    import torch
    from paddle3d_b200.ops import centerpoint_postprocess as cpp
    from paddle3d_b200.ops import voxelize as vox
    cfg, tc, st = pipe.cfg, pipe.test_cfg, pipe.stream
    names = ["voxelize", "pfn_to_pixel_image", "dense_rpn_neck_head", "postprocess"]
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
            h = pipe.dense.forward_h16(*img)
            ev[3].record(st)
            cpp.centerpoint_postprocess_device(h["hm"], h["reg"], h["height"], h["dim"], h["vel"], h["rot"],
                                               cfg["voxel_size"][:2], cfg["point_cloud_range"], tc["post_center_limit_range"],
                                               pipe.label_off, tc["down_ratio"], tc["score_threshold"],
                                               tc["nms_iou_threshold"], tc["nms_pre_max_size"], tc["nms_post_max_size"], True)
            ev[4].record(st)
        ev[4].synchronize()
        if rep:  # the first pass warms the allocator
            for k in range(4):
                runs[names[k]].append(ev[k].elapsed_time(ev[k + 1]))
    return {k: statistics.median(v) for k, v in runs.items()}, int(nv.item())


def encoder_race(pipe, frame, rounds, iters):
    """Fused encoder vs the chain it replaces on the voxels of `frame`; the two are timed alternately, `rounds` times,
    each a CUDA graph of `iters` launches (bench.graph_time_ms).  Returns medians in us and whether the images are equal."""
    import torch
    from paddle3d_b200.ops import dense_conv as dc
    from paddle3d_b200.ops import pillar_scatter as ps
    from paddle3d_b200.ops import voxelize as vox
    cfg, net, st = pipe.cfg, pipe.net, pipe.stream
    with torch.cuda.stream(st):
        voxels, coords, npv, nv = vox.hard_voxelize(frame, cfg["voxel_size"], cfg["point_cloud_range"], cfg["max_points"],
                                                    cfg["max_voxels"])
        coors = torch.nn.functional.pad(coords, (1, 0), value=0)

    def fused():
        return net.forward_pixel_h16(voxels, npv, coors, 1, pipe.ny, pipe.nx, num=nv)[0]

    def chain():
        return dc.nchw_to_pixel_h16(ps.pillar_scatter(net(voxels, npv, coors, num=nv), coors, 1, pipe.ny, pipe.nx, num=nv))

    with torch.cuda.stream(st):
        equal = bool(torch.equal(fused(), chain()))
    t_f, t_c = [], []
    for _ in range(rounds):
        t_f.append(1e3 * bench.graph_time_ms(fused, st, iters))
        t_c.append(1e3 * bench.graph_time_ms(chain, st, iters))
    return {"fused_us": statistics.median(t_f), "chain_us": statistics.median(t_c), "fused_us_all": t_f, "chain_us_all": t_c,
            "images_bit_equal": equal, "rounds": rounds, "launches_per_graph": iters}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--lanes", default="1,4")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    from paddle3d_b200 import synth
    from paddle3d_b200.pipeline import PILLARS_BN_GAIN, CenterPointPillarsHotPath, CenterPointSweep
    if not torch.cuda.is_available():
        raise SystemExit("pillars_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    cfg = synth.CP_PILLARS
    frames = bench.frame_pool(cfg, bench.POOL)
    dev_frames = [torch.from_numpy(f).to(dev) for f in frames]
    host_frames = [torch.from_numpy(f).pin_memory() for f in frames]
    res = {"model": "CenterPoint-pillars 0.2 m (synth.CP_PILLARS): 300k x 5 points, 512 x 512 pillars, max 40000, P 20",
           "gpu": gpu_info(), "torch_device_name": torch.cuda.get_device_name(dev), "bn_gain": PILLARS_BN_GAIN,
           "frames_in_pool": bench.POOL, "l2": "input pool 192 MB > 126 MB L2; no explicit flush", "steps": args.steps,
           "warmup": args.warmup, "sweep": {}}
    first = None
    for L in [int(x) for x in args.lanes.split(",")]:
        sweep = CenterPointSweep(L, pipeline_cls=CenterPointPillarsHotPath, cfg=cfg, device=dev, seed=0)
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
    res["encoder_race"] = encoder_race(pipe, dev_frames[0], 7, 20)
    H, W = pipe.ny, pipe.nx
    fl = dense_flops(pipe.dense, H, W)
    ms_dense = bench.graph_time_ms(lambda: pipe.dense.forward_h16(*pipe.out["bev_h16"]), pipe.stream, 5)
    res["dense"] = {"algorithmic_gflop": fl / 1e9, "ms_graph": ms_dense, "achieved_tflops": fl / (ms_dense * 1e-3) / 1e12,
                    "note": "2 x MACs of the convolutions from the layer geometry; the fp16-pair kernels execute 3 fp16 MMAs "
                            "per product"}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
