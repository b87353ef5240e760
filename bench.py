#!/usr/bin/env python
"""bench.py — CenterPoint frames/s on B200 (driver contract, see the task's Measurement rules).

  python bench.py [--gpus N] [--steps K] [--warmup W]            this repo's CUDA path
                 [--dump-outputs DIR]                            + what the last timed step computed, as DIR/*.npy
  python bench.py --impl reference [--steps K] [--warmup W]      the reference's CPU arm on the host cores

A step = one synthetic nuScenes-shaped frame (300k x 5 points, 1440 x 1440 x 40 grid, max 160000 voxels) through the
whole CenterPoint-voxel model:
    hard_voxelize+VoxelMean -> SparseResNet3D (21 sparse convs) -> dense BEV -> SecondBackbone + SecondFPN + CenterHead
    (dense RPN / neck / heads, 234 GFLOP) -> centerpoint_postprocess -> boxes.
Headline geometry: 0.075 m voxels / +-54 m (the heavier one); the 0.1 m / +-72 m geometry BASELINE.json names is
measured in the same run and reported under `geometry_01m` (--geometry 01 swaps them).  --no-head reproduces the
round-1 workload (resident synthetic head tensors).

`value`  : frames/s with the frame's points already resident in HBM (CUDA-graph replay per frame), --in-flight frames
           (default 4) computing concurrently per GPU: CenterPointSweep lanes with their own buffers / graph / stream and a
           shared model (measured: 605 / 709 / 740 / 754 / 735 frames/s with 1 / 2 / 3 / 4 / 6 lanes - the latency-bound
           kernels of one frame fill the SMs the other frames leave idle).
`e2e`    : frames/s through the public API CenterPointSweep.infer_many(): pinned-host points -> H2D ->
           graph -> D2H of boxes/scores/labels/counts/status, every step; the H2D of a lane's next frame overlaps its
           compute (copy stream + two staging buffers per lane). `e2e.sync_value` is the one-frame-at-a-time
           CenterPointHotPath.infer() rate (latency mode, one lane).
`roofline`: the kernel family with the largest share of the frame (dense conv or sparse conv), `rooflines_other` the
           rest; timed live with CUDA events on the launching stream.
N > 1: frame-parallel replicas, one process per GPU (torchrun), weights broadcast once over NCCL,
no per-frame collective; value = total frames / max-over-ranks time ("weak" scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "CenterPoint frames/sec @300k pts, 0.075m voxel (0.1m voxel: geometry_01m), 1440x1440x40 grid"
UNIT = "frames/s"
WORKLOAD = ("CenterPoint-voxel nuScenes-shape frame, 300k x 5 points, 1440x1440x40 grid, %s geometry: hard_voxelize+VoxelMean "
            "-> SparseResNet3D (21 sparse convs) -> dense BEV [1,256,180,180] -> %s -> centerpoint_postprocess (6 tasks)")
HEAD_ON = "SecondBackbone + SecondFPN + CenterHead (2 x 6 + 2 + 1 + 36 + 36 convs, 234 GFLOP)"
HEAD_OFF = "resident synthetic head tensors (dense RPN/head skipped: --no-head)"
BN_GAIN = 6.0 ** 0.5  # seeded weights with BatchNorm gamma = sqrt(6): activations stay O(1) through the 21 + 54 convs
POOL = 32  # distinct frames cycled through: 32 x 6 MB = 192 MB of inputs > 126 MB L2


def make_config(geometry, with_head, in_flight=4):
    """The `config` object both arms print (identical dicts: the driver compares them)."""
    geo = "0.075 m voxels / +-54 m range" if geometry == "0075" else "0.1 m voxels / +-72 m range"
    return {"workload": WORKLOAD % (geo, HEAD_ON if with_head else HEAD_OFF), "geometry": geometry, "with_head": bool(with_head),
            "frames_in_pool": POOL, "l2": "input pool 192 MB > 126 MB L2; no explicit flush",
            "frames_in_flight_per_gpu": int(in_flight)}


def frame_pool(cfg, n_frames, seed0=0, base=4):
    """`base` ray-cast lidar clouds, expanded to n_frames by a seeded yaw rotation + jitter (cheap, distinct)."""
    from paddle3d_b200 import synth
    bases = [synth.lidar_cloud(cfg, seed0 + i) for i in range(base)]
    out = []
    for f in range(n_frames):
        rng = np.random.default_rng(1000 + seed0 + f)
        p = bases[f % base].copy()
        if f >= base:
            a = rng.uniform(0, 2 * np.pi)
            c, s = np.cos(a), np.sin(a)
            xy = p[:, :2] @ np.array([[c, -s], [s, c]], np.float32)
            p[:, :2] = xy + rng.normal(0, 0.01, size=xy.shape).astype(np.float32)
            rng.shuffle(p, axis=0)
        out.append(np.ascontiguousarray(p, dtype=np.float32))
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
                for nme, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": (sorted(load)[len(load) // 2] if load else None), "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def cpu_threads_for_reference():
    """The CPU arm uses every host core.  torchrun exports OMP_NUM_THREADS=1 to its workers; only rank 0 runs this arm
    (the other ranks exit), so it takes the whole machine back before the OpenMP runtime of the oracle is loaded."""
    n = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(n)
    return n


def build_cpu_frame(cfg, with_head, weights=None, dense_weights=None, head=None):
    """CpuFrame with the same seeded weights as the CUDA arm (generated on the CPU, no GPU needed)."""
    from paddle3d_b200 import synth
    from oracle.cpu_reference import CpuFrame
    from paddle3d_b200.layers import SparseResNet3D
    from paddle3d_b200.pipeline import CenterPointHotPath
    if weights is None:
        class _W:
            pass
        w = _W()
        w.net = SparseResNet3D(cfg["point_dim"], cfg["voxel_size"], cfg["point_cloud_range"]).init_weight(seed=0, device="cpu",
                                                                                                         bn_gain=BN_GAIN)
        weights = CenterPointHotPath.export_weights_numpy(w)
    if with_head and dense_weights is None:
        from paddle3d_b200.dense_head import DenseRPNHead
        dense_weights = DenseRPNHead(in_channels=256).init_weight(seed=1, device=None, bn_gain=BN_GAIN).export_numpy()
    if head is None:
        head = synth.centerpoint_head_outputs(0)
    return CpuFrame(cfg, weights, head, synth.CENTERPOINT_TEST_CFG, synth.label_offsets(),
                    dense_weights=dense_weights if with_head else None)


def run_reference(args):
    """CPU arm: the reference's own CPU voxelizer (oracle/_ref, when built) + the oracle port for the stages
    the reference only implements on the GPU / inside PaddlePaddle.  One step = one full frame."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores_set = cpu_threads_for_reference()
    import torch  # noqa: F401  (weights are generated with the same seeded code path as the CUDA arm)
    from paddle3d_b200 import synth
    import oracle
    cfg = synth.C3 if args.geometry == "0075" else synth.C3_01
    with_head = not args.no_head
    cf = build_cpu_frame(cfg, with_head)
    frames = frame_pool(cfg, 2, base=2)
    t_w = time.perf_counter()
    n_warm = min(args.warmup, 1)  # a frame costs ~10 s on the host: one untimed frame warms caches / page tables
    for i in range(n_warm):
        cf.run(frames[i % len(frames)])
    per_frame = (time.perf_counter() - t_w) / max(n_warm, 1)
    # bound the run: the number of timed frames is capped at what fits in about two minutes (the per-frame throughput
    # is what is reported, not a total)
    steps = max(1, min(args.steps, int(120.0 / max(per_frame, 1e-3))))
    t0 = time.perf_counter()
    stages = {}
    for i in range(steps):
        r = cf.run(frames[i % len(frames)])
        for k, v in r["times"].items():
            stages[k] = stages.get(k, 0.0) + v
    dt = time.perf_counter() - t0
    requested, args.steps = args.steps, steps
    fps = args.steps / dt
    cores = oracle.num_threads()
    sample = ("%d full frames; voxelize = %s, voxel_mean / sparse conv / to_dense / dense RPN+head / postprocess = oracle "
              "port (OpenMP, %d threads of %d host cores; the reference has no CPU implementation of them)" %
              (args.steps, "reference hard_voxelize_cpu compiled unmodified (oracle/_ref)" if cf.use_ref else "oracle port",
               cores, cores_set))
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (f64 accumulation)", "data": "synthetic",
            "config": make_config(args.geometry, with_head, max(1, args.in_flight)),
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "stage_ms": {k: 1e3 * v / args.steps for k, v in stages.items()}, "gpu_launches": 0,
            "steps_requested": requested}
    print(json.dumps(line))


def graph_time_ms(fn, stream, iters=5):
    """Device time of fn(): captured `iters` times into one CUDA graph, replayed, CUDA events on `stream`."""
    import torch
    with torch.cuda.stream(stream):
        fn()
        stream.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            for _ in range(iters):
                fn()
        g.replay()
        stream.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(stream)
        g.replay()
        e.record(stream)
    e.synchronize()
    return s.elapsed_time(e) / iters


def ncu_dram_bytes(path_name):
    """dram__bytes_read.sum + dram__bytes_write.sum summed over the launches of a committed ncu capture
    (profiles/<path_name>: rows = launches of one frame); None when the capture is not in the tree."""
    import csv
    path = os.path.join(ROOT, "profiles", path_name)
    if not os.path.exists(path):
        return None
    try:
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        total = 0.0
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = hdr.index(name)
            total += sum(float(r[i]) for r in rows[2:]) * scale[units[i]]
        return total
    except (ValueError, KeyError, IndexError, OSError):
        return None  # a malformed capture must not take the benchmark down


def ncu_tensor_active(path_name):
    """Time-weighted sm__pipe_tensor_cycles_active (% of peak sustained active) over the launches of a committed ncu capture
    (tcgen05 and legacy HMMA launches alike); None when the capture is not in the tree."""
    import csv
    path = os.path.join(ROOT, "profiles", path_name)
    if not os.path.exists(path):
        return None
    try:
        rows = list(csv.reader(open(path)))
        hdr = rows[0]
        it, ia = hdr.index("gpu__time_duration.sum"), hdr.index("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active")
        t = [float(r[it]) for r in rows[2:]]
        a = [float(r[ia]) for r in rows[2:]]
        return sum(x * y for x, y in zip(t, a)) / sum(t) if sum(t) > 0 else None
    except (ValueError, KeyError, IndexError, OSError):
        return None


def dense_flops(net, H, W):
    """Algorithmic flops (2 x MACs) of the dense RPN / neck / CenterHead at a BEV of H x W."""
    total, h, w = 0.0, H, W
    for blk in net.blocks:
        for c in blk:
            h, w = (h + 2 * c.padding - c.k) // c.stride + 1, (w + 2 * c.padding - c.k) // c.stride + 1
            total += 2.0 * h * w * c.cin * c.cout * c.k * c.k
    hh, ww = H, W
    sizes = []
    h, w = H, W
    for blk in net.blocks:
        for c in blk:
            h, w = (h + 2 * c.padding - c.k) // c.stride + 1, (w + 2 * c.padding - c.k) // c.stride + 1
        sizes.append((h, w))
    for (h, w), de in zip(sizes, net.deblocks):
        total += 2.0 * (h * de.up) * (w * de.up) * de.cin * de.cout * (1 if de.up > 1 else de.k * de.k)
        hh, ww = h * de.up, w * de.up
    total += 2.0 * hh * ww * net.shared.cin * net.shared.cout * 9
    for hs in net.heads:
        for _, a, f in hs:
            total += 2.0 * hh * ww * (a.cin * a.cout + f.cin * f.cout) * 9
    return total


def measure(sweep, dev_frames, host_frames, args, world, dist, sample_clocks, local, keep_outputs=False):
    """Device-timed resident-input rate, e2e (pipelined and one-frame-at-a-time) for one sweep engine (len(sweep) frames in
    flight, CenterPointSweep).  Returns a dict; keep_outputs adds "outputs", the results of the last timed step."""
    import torch
    pipe = sweep.lanes[0]
    st = pipe.stream

    def step_resident(i):
        sweep.launch(i, dev_frames[i % len(dev_frames)])  # D2D copy (the frame is already in HBM) + graph replay on lane i % L

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step_resident(i)
    barrier()
    sampler = None
    if sample_clocks:
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.3)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    s.record(st)
    for p in sweep.lanes[1:]:
        p.stream.wait_event(s)   # every lane starts after the start event ...
    for i in range(args.steps):
        step_resident(i)
    for p in sweep.lanes[1:]:
        st.wait_stream(p.stream)  # ... and the end event fires after the last frame of every lane
    e.record(st)
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = s.elapsed_time(e)
    outputs = last_step_outputs(sweep.lanes[(args.steps - 1) % len(sweep)]) if keep_outputs else None
    # ---- e2e through the public API (host in, host out), same K
    sweep.prepare_sweep()
    for i in range(3):
        pipe.infer(host_frames[i % len(host_frames)])
    for _res in sweep.infer_many(host_frames[i % len(host_frames)] for i in range(4 * len(sweep))):  # untimed: first use of the sweep path
        pass
    barrier()
    t1 = time.perf_counter()
    n_res = 0
    for _res in sweep.infer_many(host_frames[i % len(host_frames)] for i in range(args.steps)):  # per-frame H2D + D2H, pipelined
        n_res += 1
    assert n_res == args.steps
    barrier()
    e2e_s = time.perf_counter() - t1
    t2 = time.perf_counter()
    for i in range(args.steps):
        pipe.infer(host_frames[i % len(host_frames)])   # one frame at a time (latency mode), reported beside the headline
    barrier()
    e2e_sync_s = time.perf_counter() - t2
    clocks = sampler.finish() if sampler is not None else None
    tt = torch.tensor([dev_ms, e2e_s * 1e3, wall * 1e3, e2e_sync_s * 1e3], dtype=torch.float64, device=pipe.device)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, wall_ms, sync_ms = [float(x) for x in tt.cpu()]
    total = args.steps * world
    return {"value": total / (dev_ms * 1e-3), "ms_per_step": dev_ms / args.steps, "e2e_value": total / (e2e_ms * 1e-3),
            "e2e_sync_value": total / (sync_ms * 1e-3), "wall_ms_per_step": wall_ms / args.steps, "clocks": clocks,
            "outputs": outputs}


def last_step_outputs(lane):
    """What CenterPointHotPath.infer hands its caller for the frame `lane` computed last (boxes [K, 9], scores [K],
    labels [K]) plus the per-task box counts, as float32 / float64 numpy arrays (labels and counts are small integers)."""
    o = {k: lane.out[k].cpu() for k in ("boxes", "scores", "labels", "counts", "status")}
    lane.check_status(o["status"])
    k = int(o["counts"][-1])
    return {"boxes": o["boxes"][:k].numpy().astype(np.float32), "scores": o["scores"][:k].numpy().astype(np.float32),
            "labels": o["labels"][:k].numpy().astype(np.float64), "counts": o["counts"].numpy().astype(np.float64)}


def reference_gpu_race(dev, stream):
    """The reference's own Paddle-free CUDA kernels (compiled unmodified into oracle/_ref, the "kernels to beat" of
    SURVEY §8d-ii) timed beside this repo's ops, same process, same inputs, CUDA events.  Baseline leg only."""
    import ctypes as C
    import torch
    import oracle
    from paddle3d_b200 import synth
    from paddle3d_b200.ops import bev_pool_v2, iou3d_nms
    out = {}

    def ev_time(fn, iters=20):
        torch.cuda.synchronize()
        fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(int(1e7))  # park the GPU ~5 ms: the host queues all launches first, the events then bracket
        s.record()                   # back-to-back GPU work, not Python / ctypes call overhead
        for _ in range(iters):
            fn()
        e.record()
        e.synchronize()
        return s.elapsed_time(e) / iters * 1e3  # us

    ref = oracle.ref_lib("iou3d_gpu")
    if ref is not None:
        a = torch.from_numpy(synth.random_boxes(1000, 3)).to(dev)
        b = torch.from_numpy(synth.random_boxes(1000, 4)).to(dev)
        want = torch.empty((1000, 1000), dtype=torch.float32, device=dev)
        mask = torch.zeros((1000, 16), dtype=torch.int64, device=dev)
        out["boxes_iou_bev 1000x1000"] = {
            "reference_us": ev_time(lambda: ref.ref_boxes_iou_bev_gpu(C.c_void_p(0), 1000, C.c_void_p(a.data_ptr()), 1000,
                                                                       C.c_void_p(b.data_ptr()), C.c_void_p(want.data_ptr()))),
            "ours_us": ev_time(lambda: iou3d_nms.boxes_iou_bev_gpu(a, b))}
        out["nms 1000 boxes"] = {
            "reference_us": ev_time(lambda: ref.ref_nms_mask_gpu(C.c_void_p(0), C.c_void_p(a.data_ptr()), C.c_void_p(mask.data_ptr()),
                                                                  1000, C.c_float(0.2))),
            "ours_us": ev_time(lambda: iou3d_nms.nms_gpu(a, 0.2, device_outputs=True)),
            "note": "reference = bit-matrix kernel only (its greedy pass runs on the host after a D2H copy, iou3d_nms.cpp:115-135); "
                    "ours = bit-matrix + greedy on the device"}
    ref = oracle.ref_lib("bevpool_gpu")
    if ref is not None:
        for grid, bd in (((128, 128, 1), (-51.2, 51.2)), ((200, 200, 1), (-50.0, 50.0))):
            d = synth.bev_pool_inputs(5, grid=grid, bounds=(bd, bd, (-5.0, 3.0)))
            keys = ["depth", "feat", "ranks_depth", "ranks_feat", "ranks_bev", "interval_lengths", "interval_starts"]
            t = [torch.from_numpy(d[k]).to(dev) for k in keys]
            o = torch.zeros(d["bev_feat_shape"], dtype=torch.float32, device=dev)
            p = [C.c_void_p(x.data_ptr()) for x in t]
            out["bev_pool_v2 %dx%d" % grid[:2]] = {
                "reference_us": ev_time(lambda: ref.ref_bev_pool_v2_gpu(d["feat"].shape[-1], len(d["interval_starts"]), p[0], p[1], p[2],
                                                                         p[3], p[4], p[6], p[5], C.c_void_p(o.data_ptr()))),
                "ours_us": ev_time(lambda: bev_pool_v2.bev_pool_v2(*t, d["bev_feat_shape"])),
                "note": "ours includes the zero fill of the output (the reference op does it in a separate paddle.full)"}
    for v in out.values():
        v["speedup"] = v["reference_us"] / v["ours_us"]
    return out


def rel_errors(got, want, floor=1e-2):
    """Same definition as tests/parity.py: true relative error above floor x max, absolute (over max) below."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = float(np.abs(want).max())
    err = np.abs(got - want)
    big = np.abs(want) > floor * scale
    return {"max_rel_above_1e-2_of_max": float((err[big] / np.abs(want[big])).max()) if big.any() else 0.0,
            "max_abs_below_over_max": float(err[~big].max() / scale) if (~big).any() and scale > 0 else 0.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="f16x3", choices=["fp32", "tf32x3", "tf32x3_split", "tf32x3_tma", "f16x3"])
    ap.add_argument("--geometry", default="0075", choices=["0075", "01"], help="headline geometry (the other one is "
                    "measured as well and reported in `geometry_01m` / `geometry_0075`)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-head", action="store_true", help="skip the dense RPN / neck / CenterHead (round-1 workload)")
    ap.add_argument("--no-second-geometry", action="store_true")
    ap.add_argument("--in-flight", type=int, default=4, help="frames computing concurrently per GPU (CenterPointSweep lanes)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (boxes, scores, labels, "
                    "per-task counts of rank 0) to DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        args.steps = max(1, args.steps)
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from paddle3d_b200 import synth
    from paddle3d_b200.ops import sparse_nn as sp
    from paddle3d_b200.ops import voxelize as vox
    from paddle3d_b200.pipeline import CenterPointHotPath, CenterPointSweep

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    with_head = not args.no_head
    cfg = synth.C3 if args.geometry == "0075" else synth.C3_01
    precision = {"tf32x3": sp.TF32X3, "tf32x3_split": sp.TF32X3_SPLIT, "tf32x3_tma": sp.TF32X3_TMA, "fp32": sp.FP32,
                 "f16x3": sp.F16X3}[args.precision]
    caps = [int(x) for x in os.environ["P3D_LEVEL_CAPS"].split(",")] if os.environ.get("P3D_LEVEL_CAPS") else None
    lanes = max(1, args.in_flight)
    sweep = CenterPointSweep(lanes, cfg=cfg, device=dev, precision=precision, seed=0, level_caps=caps, with_head=with_head,
                             keep_bev=False, bn_gain=BN_GAIN)
    pipe = sweep.lanes[0]  # the lanes share one model; lane 0 is the one the rooflines / checks below look at
    if world > 1:  # weights only: one broadcast over NVLink at start, no per-frame collective (SURVEY §8e)
        from paddle3d_b200.sharding import broadcast_weights
        broadcast_weights(pipe.net, 0)
    # frames: rank r owns frames r, r + world, ... of the sweep (frame-parallel sharding)
    frames = frame_pool(cfg, POOL, seed0=rank * 100)
    dev_frames = [torch.from_numpy(f).to(dev) for f in frames]
    host_frames = [torch.from_numpy(f).pin_memory() for f in frames]
    pipe.calibrate_head(dev_frames[0])   # random-init heat maps -> ~1.4 % of cells above the score threshold (SURVEY §8d)
    pipe.points.copy_(dev_frames[0])
    pipe.capture(count_nodes=rank == 0)
    for p in sweep.lanes[1:]:
        p.points.copy_(dev_frames[0])
        p.capture()
    graph_nodes = pipe.graph_nodes["kernel"] if (rank == 0 and pipe.graph_nodes) else None
    st = pipe.stream
    m = measure(sweep, dev_frames, host_frames, args, world, dist, True, local, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in m["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    # ---- the other geometry, same model, shorter run (reported, not the headline)
    other = None
    if not args.no_second_geometry:
        ogeo = "01" if args.geometry == "0075" else "0075"
        ocfg = synth.C3_01 if ogeo == "01" else synth.C3
        osweep = CenterPointSweep(lanes, cfg=ocfg, device=dev, precision=precision, seed=0, level_caps=caps, with_head=with_head,
                                  keep_bev=False, bn_gain=BN_GAIN)
        opipe = osweep.lanes[0]
        oframes = frame_pool(ocfg, 8, seed0=rank * 100, base=2)
        odev = [torch.from_numpy(f).to(dev) for f in oframes]
        ohost = [torch.from_numpy(f).pin_memory() for f in oframes]
        if opipe.dense is not None:  # same (calibrated) head weights as the headline pipeline
            for ca, cb in zip(opipe.dense.all_convs(), pipe.dense.all_convs()):
                ca.np["bias"] = cb.np["bias"]
            opipe.dense._batched = None
        osweep.capture(odev[0])
        oargs = argparse.Namespace(steps=max(20, args.steps // 4), warmup=max(3, args.warmup // 4))
        om = measure(osweep, odev, ohost, oargs, world, dist, False, local)
        other = (ogeo, om, oargs, int(opipe.out["num_voxels"][0].item()))
        del osweep, opipe, odev, ohost

    # ---- rooflines of the dominant kernels, timed live (events on the launching stream), rank 0 only
    extra = {}
    if rank == 0:
        hbm_peak, peak_src = peaks()
        N, F, P, V = pipe.n, pipe.F, cfg["max_points"], cfg["max_voxels"]
        pts = dev_frames[0]
        # hard_voxelize op (reference API, zero-padded outputs): 4NF + 4VPF + 12V + 4V + 4 bytes (SURVEY §8d)
        vox_bytes = 4 * N * F + 4 * V * P * F + 12 * V + 4 * V + 4
        ms_vox = graph_time_ms(lambda: vox.hard_voxelize(pts, cfg["voxel_size"], cfg["point_cloud_range"], P, V), st, 10)
        # per-stage device times (eager re-run with events; first pass warms the allocator, second is timed)
        from paddle3d_b200.ops import centerpoint_postprocess as cpp
        stage, layers = {}, []
        for rep in range(2):
            with torch.cuda.stream(st):
                pipe.points.copy_(dev_frames[0])
                sp.PROFILE = [] if rep == 1 else None
                if rep == 1:
                    # park the GPU for ~10 ms so the host enqueues the whole frame first: the events below then
                    # bracket back-to-back kernels, not Python/ctypes launch gaps
                    torch.cuda._sleep(int(2e7))
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
                ev[0].record(st)
                mean, coors, npv, nv = vox.voxelize_mean(pipe.points, cfg["voxel_size"], cfg["point_cloud_range"], P, V, 0)
                ev[1].record(st)
                x, _ = pipe.net.forward_sparse(mean, coors, 1, num=nv)
                x.values()
                ev[2].record(st)
                if pipe.keep_bev:
                    bev = x.to_dense_bev()
                    pipe.net.join()
                    ev[3].record(st)
                    h = pipe.dense(bev) if pipe.dense is not None else pipe.head
                else:
                    bev16 = x.to_pixel_h16()
                    pipe.net.join()
                    ev[3].record(st)
                    h = pipe.dense.forward_h16(*bev16)
                ev[4].record(st)
                tc = pipe.test_cfg
                cpp.centerpoint_postprocess_device(h["hm"], h["reg"], h["height"], h["dim"], h["vel"], h["rot"],
                                                   cfg["voxel_size"][:2], cfg["point_cloud_range"],
                                                   tc["post_center_limit_range"], pipe.label_off, tc["down_ratio"],
                                                   tc["score_threshold"], tc["nms_iou_threshold"],
                                                   tc["nms_pre_max_size"], tc["nms_post_max_size"], True)
                ev[5].record(st)
            ev[5].synchronize()
        prof, sp.PROFILE = sp.PROFILE, None
        names = ["voxelize_mean", "sparse_backbone(eager: rulebooks + 21 convs)", "to_dense_bev", "dense_rpn_neck_head",
                 "postprocess"]
        for k in range(5):
            stage[names[k]] = ev[k].elapsed_time(ev[k + 1])
        nvox = int(nv.item())
        tc_ms, tc_flops = 0.0, 0.0
        tcp = (sp.TF32X3, sp.TF32X3_SPLIT, sp.TF32X3_TMA, sp.F16X3)
        wm_ms = 0.0
        for (cin, cout, K, prec, nbr, num, s_ev, e_ev, kern) in prof:
            rows = int(num[0].item()) if num is not None else nbr.shape[0]
            pairs = int((nbr[:rows] >= 0).sum().item())
            ms = s_ev.elapsed_time(e_ev)
            fl = 2.0 * pairs * cin * cout
            layers.append({"cin": cin, "cout": cout, "rows": rows, "pairs": pairs, "ms": round(ms, 4),
                           "precision": {sp.F16X3: "f16x3", sp.FP32: "fp32"}.get(prec, "tf32x3"), "gflop": round(fl / 1e9, 3),
                           "kernel": ("wm::conv_wm_kernel (register gather + mma.sync)" if kern == "wm" else
                                      "tcgen05" if prec in tcp else "small_cin (fp32 FMA)")})
            if prec in tcp:
                tc_ms += ms
                tc_flops += fl
                if kern == "wm":
                    wm_ms += ms
        extra["stage_ms_eager"] = stage
        extra["num_voxels_frame0"] = nvox
        extra["sparse_conv_layers"] = layers
        pkp = os.path.join(ROOT, "MEASURED_PEAKS.json")
        pk = json.load(open(pkp)) if os.path.exists(pkp) else {}
        bf16_peak = pk.get("bf16_tflops", 1590.0)
        tpeak_src = "MEASURED_PEAKS.json bf16_tflops (burst)" if pk else "fallback 1.59 PFLOP/s"
        rooflines = []
        rooflines.append({"bound": "hbm", "kernel": "hard_voxelize op (reference API: zero-padded [V, P, F] output)",
                          "achieved": vox_bytes / (ms_vox * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                          "frac": vox_bytes / (ms_vox * 1e-3) / 1e9 / hbm_peak, "traffic": ncu_dram_bytes("r02_voxelize_ncu_metrics.csv"),
                          "algorithmic_bytes": vox_bytes, "ms": ms_vox, "peak_source": peak_src})
        sparse_roof = None
        if tc_ms > 0:
            ach = tc_flops / (tc_ms * 1e-3) / 1e12
            kname = {sp.F16X3: "f16::conv_f16_kernel", sp.TF32X3_SPLIT: "tc2::gather_gemm_split_kernel"}.get(precision, "tc::gather_gemm_tf32x3_kernel")
            if wm_ms > 0:
                kname += " (wide layers) + wm::conv_wm_kernel (16/32-channel layers, %.3f ms)" % wm_ms
            sparse_roof = {"bound": "tensor", "kernel": kname + " (the 20 tensor-core sparse convs of one frame)",
                           "achieved": ach, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach / bf16_peak,
                           "traffic": ncu_dram_bytes("r02_sparse_ncu_metrics.csv"),
                           "tensor_pipe_active_pct_ncu": ncu_tensor_active("r02_sparse_ncu_metrics.csv"),
                           "algorithmic_flops": tc_flops, "ms": tc_ms,
                           "peak_source": tpeak_src,
                           "note": "achieved counts ALGORITHMIC flops 2*pairs*Cin*Cout; the kernels execute 3 fp16 MMAs per "
                                   "product on zero-padded row tiles; bound by the row gather (tcgen05 kernel: L1TEX wavefronts "
                                   "per gathered row, profiles/r02_f16_sweep.md; warp-MMA kernel: L2 latency of the register "
                                   "gather + issue slots, profiles/r02_wm_ncu_metrics.csv), not by the tensor pipe"}
        dense_roof = None
        if pipe.dense is not None:
            if pipe.out["bev_h16"] is not None:
                rows_t, shp = pipe.out["bev_h16"]
                ms_dense = graph_time_ms(lambda: pipe.dense.forward_h16(rows_t, shp), st, 3)
                fl = dense_flops(pipe.dense, shp[1], shp[2])
            else:
                bev_t = pipe.out["bev"]
                ms_dense = graph_time_ms(lambda: pipe.dense(bev_t), st, 3)
                fl = dense_flops(pipe.dense, bev_t.shape[2], bev_t.shape[3])
            ach = fl / (ms_dense * 1e-3) / 1e12
            dense_roof = {"bound": "tensor", "kernel": "dcf::dense_conv_f16_kernel (RPN + neck + CenterHead: 16 + 1 + 1 launches)",
                          "achieved": ach, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach / bf16_peak,
                          "traffic": ncu_dram_bytes("r02_dense_ncu_metrics.csv"),
                          "tensor_pipe_active_pct_ncu": ncu_tensor_active("r02_dense_ncu_metrics.csv"),
                          "algorithmic_flops": fl, "ms": ms_dense,
                          "peak_source": tpeak_src,
                          "note": "achieved counts ALGORITHMIC flops (2 x MACs of the convolutions); the kernel executes 3 fp16 "
                                  "MMAs per product (fp16-pair operands, 1e-4 parity), i.e. the tensor pipe runs at 3 x "
                                  "this fraction of the measured fp16/bf16 peak"}
        cands = [r for r in (dense_roof, sparse_roof) if r is not None]
        cands.sort(key=lambda r: -r["ms"])
        if cands:
            extra["roofline"] = cands[0]
            rooflines = cands[1:] + rooflines
        extra["rooflines_other"] = rooflines
        # CPU baseline on a bounded sample: one full frame through the oracle port (N = 1 only: under torchrun the ranks
        # share the host cores and OMP_NUM_THREADS is 1; `--impl reference` is the CPU arm of the scaling runs)
        if not args.no_cpu_baseline and world == 1:
            import oracle
            dense_w = pipe.dense.export_numpy() if pipe.dense is not None else None
            cf = build_cpu_frame(cfg, with_head, pipe.export_weights_numpy(), dense_w, pipe.head_host)
            t2 = time.perf_counter()
            r = cf.run(frames[0])
            cpu_s = time.perf_counter() - t2
            extra["cpu_baseline"] = {"value": 1.0 / cpu_s, "unit": UNIT, "cores": oracle.num_threads(), "kind": "port",
                                     "sample": "1 full frame (frame 0 of the pool); voxelize = %s; other stages = "
                                               "oracle port with OpenMP" % ("reference hard_voxelize_cpu (oracle/_ref)"
                                                                            if cf.use_ref else "oracle port"),
                                     "stage_s": r["times"]}
            # cross-check while we are here: GPU frame vs CPU frame on the same full-size input
            got = pipe.infer(host_frames[0])
            chk = {"num_voxels_equal": nvox == r["num_voxels"], "boxes_gpu": int(len(got[2])), "boxes_cpu": int(len(r["labels"]))}
            bev_gpu = pipe.bev_nchw()
            chk["bev"] = rel_errors(bev_gpu.cpu().numpy(), r["bev"])
            if r["head"] is not None:
                gh = pipe.dense(bev_gpu)
                torch.cuda.synchronize()
                worst, worst_spread = 0.0, 0.0
                for name in r["head"]:
                    for g, wv in zip(gh[name], r["head"][name]):
                        err = float(np.abs(g.cpu().numpy() - wv).max())
                        worst = max(worst, err / max(1.0, float(np.abs(wv).max())))
                        worst_spread = max(worst_spread, err / max(1e-30, float(wv.max() - wv.min())))
                chk["head_max_abs_err_over_range"] = worst
                chk["head_max_abs_err_over_spread"] = worst_spread  # error relative to how much the map actually varies
                chk["bev_abs_max"] = float(np.abs(r["bev"]).max())
            if len(got[2]) == len(r["labels"]):
                chk["labels_equal"] = bool(np.array_equal(got[2].numpy(), r["labels"]))
            extra["frame0_check"] = chk
            try:
                extra["reference_gpu"] = reference_gpu_race(dev, st)
            except Exception as e:  # noqa: BLE001  (a side measurement must not take the headline down)
                extra["reference_gpu"] = {"error": repr(e)}

    if rank == 0:
        h2d, d2h = pipe.bytes_per_frame()
        per_frame_launches = graph_nodes if graph_nodes else pipe_launch_estimate(pipe)
        line = {"metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": {"fp32": "f32", "f16x3": "f16x3 (fp16 hi/lo' pairs, f32 accumulation)"}.get(args.precision, "tf32x3 (f32 accumulation)"),
                "data": "synthetic", "config": make_config(args.geometry, with_head, lanes),
                "parallelism": "frame-parallel x%d (replicas, NCCL weight broadcast only), %d frames in flight per GPU "
                               "(CenterPointSweep lanes: own buffers / graph / stream, shared model)" % (world, lanes),
                "precision": args.precision,
                "e2e": {"value": m["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "api": "CenterPointSweep.infer_many (%d lanes; H2D of the next frame of a lane overlaps its compute)" % lanes,
                        "sync_note": "sync_value = CenterPointHotPath.infer, one frame at a time (latency mode, one lane)",
                        "sync_value": m["e2e_sync_value"] if world == 1 else None},
                "gpu_launches": per_frame_launches * args.steps,
                "gpu_launches_per_step": per_frame_launches,
                "gpu_launches_source": ("kernel nodes of the captured CUDA graph (cudaGraphGetNodes); all node types: %s" % pipe.graph_nodes)
                if graph_nodes else "estimate",
                "clocks": m["clocks"], "wall_ms_per_step": m["wall_ms_per_step"]}
        if other is not None:
            ogeo, om, oargs, onv = other
            line["geometry_01m" if ogeo == "01" else "geometry_0075"] = {
                "config": make_config(ogeo, with_head, lanes), "value": om["value"], "unit": UNIT, "ms_per_step": om["ms_per_step"],
                "steps": oargs.steps, "warmup": oargs.warmup, "num_voxels_frame0": onv,
                "e2e": {"value": om["e2e_value"], "unit": UNIT, "sync_value": om["e2e_sync_value"] if world == 1 else None}}
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def pipe_launch_estimate(pipe):
    """Fallback when the graph dump is unavailable: kernels of ours per frame, counted from the code."""
    vox_k = 5                      # init, insert, rank, slots, mean
    rb = 2 + 3 * 2 + 4 * 4         # res0 subm (insert+nbr); res1-3 subm (insert+nbr); 4 strided (insert, outputs, finish, nbr)
    conv = 21 + 1                  # 21 convs + the fp32 -> fp16-pair conversion after the 5-channel layer
    dense = 2                      # scat_map + scat_write
    head = (1 + 16 + 1 + 1) if pipe.dense is not None else 0   # layout + 12 backbone + 2 neck + shared + big head conv + finals
    post = 5
    return vox_k + rb + conv + dense + head + post


if __name__ == "__main__":
    main()
