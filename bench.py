#!/usr/bin/env python
"""bench.py — headline benchmark of the FaceAna hot path on B200 (BASELINE.json).

Workload (N=1): BASELINE configs[1] — Student@256 landmark-only, batch 256 pre-cropped
256x256 uint8 faces per step, one step = one pass of the landmark network + heat-map decode.

  value  faces/s, crops already resident in HBM, CUDA-event timed on the launching stream
  e2e    faces/s through the public operator call (ONNXEngine.stream_u8) with HOST buffers:
         pinned H2D of the crops and D2H of landmarks+scores inside the timed region
  roofline   the dominant kernel (largest conv by MACs), algorithmic FLOPs / event time / measured peak
  cpu_baseline  the oracle port of the reference CPU path (torch-CPU graph executor, batch-1 loop as
         face_landmark.py:40-48) on a bounded sample, all host threads

Multi-GPU (torchrun): every rank runs the same per-GPU batch (weak scaling, no collective on the data
path); time = max over ranks.  `--impl reference` times the reference's CPU path (oracle port).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

BATCH = 256
STUDENT_FLOP_PER_FACE = 2 * 1482829696          # 2*MAC, SURVEY.md 8(d)
STUDENT_README_GFLOP = 1.39e9                   # README "Flops(G)" convention (thop MACs / 2^30)
WORKLOAD = "student256_landmark_only_batch256"


def log(msg):
    sys.stderr.write("[bench %.1fs] %s\n" % (time.perf_counter() - _T0, msg))
    sys.stderr.flush()


_T0 = time.perf_counter()


def host_cores():
    """CPU threads this process may actually use: affinity mask capped by the cgroup quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def shard_frames(items, rank, world):
    """Frame-level round-robin sharding across ranks (SURVEY 8e): no collective on the data path."""
    return list(items[rank::world])


def whole_job_rate(world, per_rank_units_per_step, steps, seconds):
    """Weak scaling: every rank processes the same per-GPU batch; time is the max over ranks."""
    return world * per_rank_units_per_step * steps / seconds


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ reference arm
REF_LABEL = ("oracle port of the reference CPU path: batch-1 loop of face_landmark.py:40-48 on a node-by-node torch-CPU "
             "executor of kps_student.onnx (onnxruntime, the reference's engine, is absent from this image)")


class CpuReference:
    """The reference's CPU path for this workload.  Built ONCE (ONNX parse + weight conversion stay outside every
    timed region); `rate(n)` times only forward_crops on n faces."""

    def __init__(self):
        import torch
        import frames
        from oracle.faceana_ref import LandmarkRef
        torch.set_num_threads(host_cores())
        self.frames = frames
        self.ref = LandmarkRef()
        self.ref.forward_crops(frames.noise_crops(2, seed=7))          # first-call allocations, thread pool start-up

    def rate(self, n_faces, seed=0):
        crops = self.frames.noise_crops(n_faces, seed=seed)
        t0 = time.perf_counter()
        self.ref.forward_crops(crops)
        dt = time.perf_counter() - t0
        return n_faces / dt, dt


def dump_outputs(out_dir, named):
    """Write each output tensor as out_dir/<name>.npy in float32, so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in named.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def workload_config(B):
    return {"workload": WORKLOAD, "batch_per_gpu": B, "input": "uint8 256x256x3 crops",
            "l2": "inputs rotate over 4 x 50 MB sets (> 126 MB L2); activations per batch exceed L2"}


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path on this box's host cores.  One step = the
    batch-1 loop over one batch of crops; the batch is the full 256 faces when K+W steps of it fit ~150 s at the measured
    rate, else the largest power-of-two fraction that does (stated in cpu_baseline.sample)."""
    if rank != 0:
        return
    cpu = CpuReference()
    v0, _ = cpu.rate(8)
    budget_s = 150.0
    sample = args.batch
    while sample > 8 and (args.steps + args.warmup) * sample / v0 > budget_s:
        sample //= 2
    for k in range(args.warmup):
        cpu.rate(sample, seed=1000 + k)
    dt = 0.0
    for k in range(args.steps):
        dt += cpu.rate(sample, seed=k)[1]                   # only forward_crops is inside the clock
    fps = args.steps * sample / dt
    line = {
        "impl": "reference", "metric": "faces/sec Student@256 batch=256", "value": fps, "unit": "faces/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.batch),
        "cpu_baseline": {"value": fps, "unit": "faces/s", "cores": host_cores(), "kind": "port",
                         "sample": "%d of %d faces per step, %d steps; %s" % (sample, args.batch, args.steps, REF_LABEL)},
        "e2e": {"value": fps, "unit": "faces/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="skip the full-pipeline (configs 3/5) and detector legs")
    ap.add_argument("--pipeline-streams", type=int, default=16)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the landmarks and scores of the last timed step (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import frames
    from peppa_pig_face_landmark_b200 import ONNXEngine, runtime as rt

    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL writes its version/INFO banner to fd 1 when the communicator is created; stdout must carry exactly one JSON
        # line, so fd 1 points at stderr while the communicator comes up (the caller's NCCL_DEBUG is left untouched)
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    B = args.batch
    onnx = os.path.join(ROOT, "peppa_pig_face_landmark_b200", "pretrained", "kps_student.onnx")
    eng = ONNXEngine(onnx, device="cuda:%d" % local_rank, max_batch=B)
    lib = rt.load_library()
    stream = eng.stream

    # 4 distinct input sets of 50 MB each (200 MB > 126 MB L2), rotated per step; the intermediate
    # activations (GBs per batch) exceed L2 by themselves
    n_sets = 4
    host_sets = [torch.from_numpy(frames.noise_crops(B, seed=100 + rank * 16 + i)).pin_memory() for i in range(n_sets)]
    host_sets[0][:min(B, 64)].copy_(torch.from_numpy(frames.crop_variants(min(B, 64))))
    dev_sets = [h.cuda(non_blocking=True) for h in host_sets]
    outs = [torch.empty((B, e), dtype=torch.float32, device="cuda") for e in eng.out_elems]
    torch.cuda.synchronize()
    log("engine + inputs ready")

    def step_device(i):
        eng.forward_device(dev_sets[i % n_sets], outs, stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks/throttle reasons are sampled from before the warm-up to the end of the timed region (nvidia-smi needs
    # a few hundred ms to start, the timed region itself can be shorter than that)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        t_wait = time.perf_counter()
        while not sampler.samples and time.perf_counter() - t_wait < 3.0:
            time.sleep(0.05)
    with torch.cuda.stream(stream):
        for i in range(args.warmup):
            step_device(i)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record()
        for i in range(args.steps):
            step_device(i)
        ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    faces_per_s = whole_job_rate(world, B, args.steps, ms * 1e-3)
    log("device-resident: %.1f faces/s (%.3f ms/step)" % (faces_per_s, ms / args.steps))
    if args.dump_outputs and rank == 0:
        # `outs` is written by the timed steps only: it holds the last step's results (input set (steps - 1) % n_sets)
        dump_outputs(args.dump_outputs, {"landmarks": outs[0], "scores": outs[1]})
        log("outputs of the last timed step written to %s" % args.dump_outputs)

    # ---- end to end through the operator call with host buffers (pinned), H2D + D2H inside the timed region
    e2e_steps = max(5, min(args.steps, 20))
    host_np = [h.numpy() for h in host_sets]
    for out in eng.stream_u8(host_np[i % n_sets] for i in range(3)):
        pass
    barrier()
    t0 = time.perf_counter()
    n_done = 0
    for lm, sc in eng.stream_u8(host_np[i % n_sets] for i in range(e2e_steps)):
        n_done += 1                       # landmarks + scores of that step are in host memory here
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_fps = world * B * e2e_steps / e2e_s
    log("e2e: %.1f faces/s" % e2e_fps)
    h2d = B * 256 * 256 * 3
    d2h = B * (196 + 98) * 4

    # ---- BASELINE configs 3 and 5: the whole FaceAna path (frame upload -> detector -> NMS -> crops -> landmarks ->
    # temporal layer -> results on the host) for S concurrent video streams per GPU; streams shard across ranks with no
    # data-path collective, under torchrun the result rows are collected with one NCCL all_gather per call
    pipeline = None
    if not args.no_pipeline:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_streams
        pipeline = {}
        for name in ("1080p_4faces", "4k_16faces"):
            r = bench_streams.run_config(name, n_streams=args.pipeline_streams, batches=10, warmup=3, gather=world > 1,
                                         dist=dist if world > 1 else None, rank=rank, world=world, length=4)
            if r is not None:
                pipeline[name] = r
                log("pipeline %s: %.0f frames/s, %.0f faces/s" % (name, r["frames_per_s"], r["faces_per_s"]))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-op times (each op launched alone, CUDA events on the launching stream): roofline of the dominant
    # tensor-bound kernel (largest conv by MACs) and of the slowest HBM-bound kernel, plus the time split by op class
    from peppa_pig_face_landmark_b200 import plan as P
    peak_tf, peak_hbm, peak_src = measured_peaks()

    def conv_macs(op):
        if op.type == P.OP_CONV:
            return op.outs[0].C * op.outs[0].H * op.outs[0].W * op.ins[0].C * op.k[0] * op.k[1]
        if op.type == P.OP_DWPW:
            return op.outs[0].C * op.outs[0].H * op.outs[0].W * op.w.shape[1]
        return 0

    def time_op(idx, reps):
        with torch.cuda.stream(stream):
            for _ in range(3):
                rt.check(lib.skps_engine_run_op(eng.handle, idx, B, stream.cuda_stream))
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            for _ in range(reps):
                rt.check(lib.skps_engine_run_op(eng.handle, idx, B, stream.cuda_stream))
            k1.record()
        torch.cuda.synchronize()
        return k0.elapsed_time(k1) / reps

    op_ms = [time_op(i, 5) for i in range(len(eng.plan.ops))]
    split = {}
    if os.environ.get("SKPS_BENCH_OPS"):
        for i, (op, t) in enumerate(zip(eng.plan.ops, op_ms)):
            log("op %2d %-18s %7.1f us  %s" % (i, P.OP_NAMES[op.type], 1e3 * t, op.name[-60:]))
    for op, t in zip(eng.plan.ops, op_ms):
        kind = P.OP_NAMES[op.type] + ("/xf_scale" if op.flags & P.FLAG_XF else "/tc" if op.flags & P.FLAG_TC else "")
        split[kind] = split.get(kind, 0.0) + t
    best = max(range(len(eng.plan.ops)), key=lambda i: conv_macs(eng.plan.ops[i]) if eng.plan.ops[i].type == P.OP_CONV else 0)
    bop, best_macs = eng.plan.ops[best], conv_macs(eng.plan.ops[best])
    k_ms = time_op(best, 10)
    achieved_tf = 2.0 * best_macs * B / (k_ms * 1e-3) / 1e12
    log("dominant kernel %.3f ms -> %.2f TFLOP/s" % (k_ms, achieved_tf))
    # DRAM traffic of the dominant launch: read from the committed `ncu --set full` summary of THIS kernel (same op, same
    # batch); null when no matching capture is on file
    traffic, traffic_src = None, None
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_conv2_final.json")))
        if cap["op"] == bop.name and cap["batch"] == B:
            traffic = cap["dram__bytes_read"] + cap["dram__bytes_write"]
            traffic_src = "profiles/r2_ncu_conv2_final.json (%s)" % cap["capture"]
    except Exception:
        pass
    # slowest kernel that is bound by HBM (no dense contraction): algorithmic bytes = its input + output tensors
    hb = max((i for i, op in enumerate(eng.plan.ops) if conv_macs(op) == 0 and op.type != P.OP_HM_DECODE),
             key=lambda i: op_ms[i])
    hop = eng.plan.ops[hb]
    h_bytes = eng.plan.bytes_per_sample(hop) * B
    h_gbs = h_bytes / (op_ms[hb] * 1e-3) / 1e9
    roofline = {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved_tf / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                "traffic_algorithmic": B * eng.plan.bytes_per_sample(bop),
                "precision": "fp16 hi/lo split, 3 tcgen05 MMAs per K-step -> ceiling = peak/3",
                "frac_of_split_ceiling": achieved_tf / (peak_tf / 3.0),
                "kernel": "%s (%dx%d conv %d->%d @%dx%d, batch %d)" % (bop.name, bop.k[0], bop.k[1], bop.ins[0].C,
                                                                     bop.outs[0].C, bop.outs[0].H, bop.outs[0].W, B),
                "kernel_ms": k_ms, "kernel_share_of_step": k_ms / (ms / args.steps),
                "peak_source": "%s bf16 dense burst (MEASURED_PEAKS.json)" % peak_src,
                "hbm_kernel": {"bound": "hbm", "kernel": "%s %s (%d ch @%dx%d, batch %d)" % (
                                   P.OP_NAMES[hop.type], hop.name, hop.outs[0].C, hop.outs[0].H, hop.outs[0].W, B),
                               "achieved": h_gbs, "peak": peak_hbm, "unit": "GB/s", "frac": h_gbs / peak_hbm,
                               "bytes_algorithmic": h_bytes, "kernel_ms": op_ms[hb],
                               "kernel_share_of_step": op_ms[hb] / (ms / args.steps)},
                "op_class_ms": {k: round(v, 4) for k, v in sorted(split.items(), key=lambda kv: -kv[1])},
                "op_sum_ms": sum(op_ms),
                "whole_net_tflops": faces_per_s / world * STUDENT_FLOP_PER_FACE / 1e12,
                "whole_net_frac_2mac": faces_per_s / world * STUDENT_FLOP_PER_FACE / 1e12 / peak_tf,
                "whole_net_frac_of_split_ceiling": faces_per_s / world * STUDENT_FLOP_PER_FACE / 1e12 / (peak_tf / 3.0),
                "whole_net_frac_readme_1.39G": faces_per_s / world * STUDENT_README_GFLOP / 1e12 / peak_tf}

    detector = None
    if not args.no_pipeline:
        import bench_detector
        detector = [bench_detector.run(b, n=30, peaks=(peak_tf, peak_hbm)) for b in (1, 16)]
        log("detector: " + ", ".join("batch %d %.2f ms" % (d["batch"], d["ms"]) for d in detector))

    cpu = None
    if not args.no_cpu_baseline:
        log("cpu baseline on %d host threads" % host_cores())
        ref = CpuReference()
        v1, _ = ref.rate(8)
        n = int(max(8, min(256, 12.0 * v1)))          # ~12 s of CPU work
        v, dt = ref.rate(n, seed=1)
        cpu = {"value": v, "unit": "faces/s", "cores": host_cores(), "kind": "port",
               "sample": "%d faces in %.1f s; %s" % (n, dt, REF_LABEL)}

    line = {
        "metric": "faces/sec Student@256 batch=256", "value": faces_per_s, "unit": "faces/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(B),
        "e2e": {"value": e2e_fps, "unit": "faces/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "api": "ONNXEngine.stream_u8 (pinned host crops in, host landmarks+scores out, 2 batches in flight: H2D of step i+1 overlaps compute of step i)"},
        "gpu_launches": lib.skps_engine_launches_for_batch(eng.handle, B) * args.steps,
        "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "pipeline": pipeline, "detector": detector,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
