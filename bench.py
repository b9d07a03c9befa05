#!/usr/bin/env python
"""Headline benchmark: ResNet-50 fp16 batch-8 inferences/sec (+ p50/p99 request latency) through the
per-request hot path, N replicas on N GPUs of one node (no collective: requests are independent).

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port of the reference path
  python bench.py ... --dump-outputs DIR                   # + DIR/prob.npy: what the last timed step computed

A "step" is one pass of the hot path over one batch of 8 synthetic 3x224x224 images.
  value : whole-job inferences/s with inputs already resident in HBM (4 ExecutionContexts on 4 streams,
          input ring larger than L2), timed with CUDA events.
  e2e   : the same metric through the reference-facing InferenceManager/InferRunner/InferBench pipeline
          with PINNED HOST buffers: H2D of every request's input and D2H of its output inside the timed
          region (reference trtlab/tensorrt/src/infer_bench.cc:46-110).  The K timed requests are completions
          W+1..W+K of ONE continuous closed loop (pipeline full on both sides of the window); `e2e.bracketed`
          is the same K requests run on their own from an empty pipeline (fill + drain included).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 8
CONTEXTS = 4          # BASELINE.json configs[1]: 4 concurrent ExecutionContexts / streams
BUFFERS = 8           # 2x contexts, reference examples/00_TensorRT/infer.cc:88
RING = 32             # 32 x 4.82 MB = 154 MB of distinct inputs > 126 MB L2
METRIC = "ResNet-50 fp16 b=8 inferences/sec"
UNIT = "inferences/s"
ALGO_BYTES_PER_STEP = 470.9e6   # SURVEY.md 8(d): fp16 weights + conv in/out + residual reads, batch 8


def _dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_inputs():
    from tensorrt_laboratory_b200 import weights
    return weights.synthetic_input(BATCH, seed=1234, ring=RING)   # [RING, 8, 3, 224, 224] fp32 N(0,1)


def cpu_forward_setup():
    from tensorrt_laboratory_b200 import graph, weights
    net = graph.resnet_caffe(50)
    return net, weights.random_weights(net, 0)


def usable_cores() -> int:
    """Host cores this process may really use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = int(f.read())
            if q > 0:
                n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def pick_cpu_threads(net, wts, ring) -> int:
    """Oversubscribed intra-op threads can be catastrophically slow on shared hosts: try a few counts on one
    batch each and keep the fastest (bounded: stops trying as soon as a candidate takes > 8 s)."""
    from oracle.caffe_forward import caffe_forward
    cores = usable_cores()
    best, best_t = None, None
    for t in sorted({c for c in (8, 16, 32, cores) if c <= cores} or {1}):
        caffe_forward(net, wts, ring[0][:2], threads=t)
        t0 = time.perf_counter()
        caffe_forward(net, wts, ring[0], threads=t)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = t, dt
        if dt > 8.0:
            break
    return best or 1


def time_cpu(net, wts, ring, warm: int, iters: int, threads: int):
    from oracle.caffe_forward import caffe_forward
    for i in range(warm):
        caffe_forward(net, wts, ring[i % len(ring)], threads=threads)
    t0 = time.perf_counter()
    for i in range(iters):
        caffe_forward(net, wts, ring[i % len(ring)], threads=threads)
    dt = time.perf_counter() - t0
    return BATCH * iters / dt, dt / iters


def run_reference(args):
    """CPU arm: TensorRT (the reference's engine) cannot be built or run here (closed source, absent from
    /root/reference), so the reference arm is the oracle port of the same graph: fp32, torch CPU ops, all host
    cores, same weights and inputs."""
    rank, world, _ = _dist_env()
    if rank != 0:
        return
    net, wts = cpu_forward_setup()
    ring = build_inputs()[:4]
    cores = pick_cpu_threads(net, wts, ring)
    warm = max(1, min(args.warmup, 3))
    # bounded sample: stop near 120 s of CPU work
    ips_probe, s_per_step = time_cpu(net, wts, ring, warm, 2, cores)
    steps = max(3, min(args.steps, int(120.0 / max(s_per_step, 1e-3))))
    ips, s_per_step = time_cpu(net, wts, ring, 0, steps, cores)
    sample = f"{steps} of {args.steps} requested steps x batch {BATCH} (bounded to ~120 s), fp32 torch-CPU oracle port"
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ResNet-50 (Caffe-v1 deploy graph) batch=8 3x224x224, CPU forward", "global_batch": BATCH},
        "cpu_baseline": {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir: str, arrays: dict):
    """The arrays the headline leg's last timed step returned (ResNet-50 `prob`, [8, 1000]: 32 KB), one float32
    DIR/<binding>.npy each, so that two builds can be compared output for output on identical seeded inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, np.float32))


def run_config2(capi, builder, peaks_int8_tops: float = 4500.0):
    """BASELINE.json configs[2]: ResNet-152 INT8, batch 32, dynamic batching (examples/03_Batching), 8 streams, 1 GPU.
    Device-resident throughput of 8 execution contexts + the end-to-end rate of single-image requests merged by
    BatchedInferRunner (2 ms window) -- a SECONDARY line; the headline stays on configs[1]."""
    from tensorrt_laboratory_b200 import weights
    batch, contexts, steps = 32, 8, 96
    blob = builder.build_resnet_plan(152, builder.PREC_INT8, batch, seed=0)
    ring = weights.synthetic_input(batch, seed=4242, ring=8)                     # 8 x 19.3 MB = 154 MB > L2
    ms, launches = capi.device_throughput(blob, contexts, batch, steps, 16, ring)
    value = steps * batch / (ms * 1e-3)
    ops = capi.Engine(blob, inspect_only=True).flops(batch)                      # 2 * MACs of one batch-32 forward pass
    mgr = capi.InferenceManager(contexts, 2 * contexts, pre_threads=1, cuda_threads=1, post_threads=3)
    try:
        mgr.register_model("rn152i8", blob)
        mgr.update_resources()
        x = ring.reshape(-1, *ring.shape[2:])[:256]                              # 256 distinct images, cycled
        mgr.infer_batched("rn152i8", x, window_us=2000)                          # warm-up
        n_img, warm, cool = 6144, 1024, 1024
        _, win, dt, nb = mgr.bench_batched("rn152i8", x, n_img, warm, cool, window_us=2000)
        steady = (n_img - warm - cool) / win
    finally:
        mgr.close()
    return {
        "workload": "ResNet-152 int8 batch=32, dynamic batching, 8 streams, 1xB200 (BASELINE.json configs[2])",
        "metric": "ResNet-152 int8 b=32 inferences/sec", "value": value, "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
        "contexts": contexts, "dtype": "s8 (bottleneck convolutions; fp16 stem and classifier)", "gpu_launches": launches * steps,
        "e2e": {"value": steady, "unit": UNIT, "requests": n_img - warm - cool, "warm_requests": warm, "cool_requests": cool,
                "timed_region": "completions of requests warm..n-cool of ONE flood of single-image requests (batcher, lanes and Buffers busy on both sides)",
                "bracketed": n_img / dt, "merged_batches": nb,
                "api": "single-image requests -> BatchedInferRunner (Dispatcher<StandardBatcher>, 2000 us window) -> InferRunner; pinned H2D/D2H per merged batch",
                "h2d_bytes_per_request": 3 * 224 * 224 * 4, "d2h_bytes_per_request": 4000},
        "roofline": {"bound": "tensor", "kernel": "conv_i8_tcgen05 (the 154 INT8 convolutions of one forward pass)",
                     "achieved": ops * steps / (ms * 1e-3) / 1e12, "peak": peaks_int8_tops, "unit": "TOP/s",
                     "frac": ops * steps / (ms * 1e-3) / 1e12 / peaks_int8_tops,
                     # DRAM bytes (read + write) of the 155 conv launches of one batch-32 forward pass, committed ncu pass
                     "traffic": 1171.1e6, "traffic_source": "profiles/ncu_metrics_r2_int8.csv",
                     "peak_source": "NOMINAL dense int8 4.5 POP/s (B200_PROFILING.md table; MEASURED_PEAKS.json has no int8 entry)"},
    }


def run_b200(args):
    rank, world, local = _dist_env()
    from tensorrt_laboratory_b200 import builder, capi

    lib = capi.load()
    if capi.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device visible and there is no CPU fallback for the product path")
    capi.check(lib.b2_device_set(local))
    # this replica's threads next to its GPU (NVML cpu affinity, reference DeviceInfo::Affinity); pool threads bind themselves
    affinity_cpus = capi.bind_thread_to_device(local) if os.environ.get("TRTLAB_AFFINITY", "1") != "0" else 0
    # Each replica keeps ~6 host threads (bench loop, pre/cuda pools, 3 post threads).  When the replicas of this box
    # outnumber its usable cores, spin-waiting on CUDA events starves the threads that feed the GPUs: block instead.
    sync_mode = os.environ.get("B2_BENCH_SYNC", "auto")
    blocking = sync_mode == "block" or (sync_mode == "auto" and usable_cores() < 6 * world)
    capi.check(lib.b2_device_set_blocking_sync(1 if blocking else 0))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_
        torch.cuda.set_device(local)
        dist_.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
        dist = dist_

    blob = builder.build_resnet_plan(50, builder.PREC_FP16, BATCH, seed=0)
    ring = build_inputs()
    eng_meta = capi.Engine(blob, inspect_only=True)
    flops_step = eng_meta.flops(BATCH)
    in_bytes = BATCH * 3 * 224 * 224 * 4
    out_bytes = BATCH * 1000 * 4

    def barrier():
        capi.check(lib.b2_device_sync())
        if dist is not None:
            dist.barrier()

    from tensorrt_laboratory_b200 import replicas  # the N > 1 host logic (MAX / gather over ranks; gloo-tested on CPU)

    def gather_over_ranks(x: float):
        return replicas.gather_over_ranks(x, dist)

    def max_over_ranks(x: float) -> float:
        return replicas.max_over_ranks(x, dist)

    # ---- value: device-resident inputs, CONTEXTS streams, CUDA events ---------------------------------------
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    elapsed_ms, launches_per_step, *last = capi.device_throughput(blob, CONTEXTS, BATCH, args.steps, max(args.warmup, 3), ring,
                                                                  return_outputs=args.dump_outputs is not None)
    barrier()
    clocks = sampler.stop()
    if last and rank == 0:
        dump_outputs(args.dump_outputs, last[0])
    elapsed_ms = max_over_ranks(elapsed_ms)
    ms_per_step = elapsed_ms / args.steps
    value = world * args.steps * BATCH / (elapsed_ms * 1e-3)

    # ---- e2e: InferenceManager / InferRunner / InferBench with pinned host buffers -------------------------
    # Tactics are timed at RegisterModel and every (lane-pinned context, batch) plan + graph is built in
    # AllocateResources, so nothing is tuned, captured or instantiated inside the timed region; the warm-up still
    # cycles through every pooled Buffers / execution token at least twice.
    e2e_warm = max(max(args.warmup, 3) * CONTEXTS, 2 * BUFFERS * 2)
    per_rank = []  # per leg: every rank's own end-to-end rate
    steady = []    # per leg: the mid-stream window measurement

    def e2e_run(plan_blob):
        # thread counts of examples/00_TensorRT/infer.cc:100-102 (1 / 1 / 3); B2_BENCH_THREADS="pre,cuda,post" for experiments
        pre_t, cuda_t, post_t = (int(v) for v in os.environ.get("B2_BENCH_THREADS", "1,1,3").split(","))
        mgr = capi.InferenceManager(CONTEXTS, BUFFERS, pre_threads=pre_t, cuda_threads=cuda_t, post_threads=post_t)
        mgr.register_model("rn50", plan_blob)
        mgr.update_resources()
        mgr.prefill_inputs("rn50", ring[:BUFFERS])
        mgr.bench("rn50", BATCH, seconds=600.0, max_batches=e2e_warm, want_latencies=False)
        barrier()
        res, lats = mgr.bench("rn50", BATCH, seconds=600.0, max_batches=args.steps, want_latencies=True)
        barrier()
        per_rank.append(gather_over_ranks(args.steps * BATCH / res["kWalltime"]))
        wall = max_over_ranks(res["kWalltime"])
        # the same K requests rated INSIDE one continuous loop (pipeline full on both sides of the window): a bracketed run
        # of K = 20 requests is mostly the fill and drain of an 8-deep pipeline (1.4 ms each way against 3.4 ms of work)
        # ... and FIVE such windows back to back in the same loop, rated by their median: at K = 20 a window is 3.4 ms, and one
        # scheduling hiccup of the host (seen once: a 3.2 ms request in an otherwise 1.4 ms stream) would halve a single one
        n_win = 5
        win_s, win_lat = mgr.bench_windows("rn50", BATCH, warm=e2e_warm, steps=args.steps, windows=n_win, cool=2 * BUFFERS)
        barrier()
        rates = [world * args.steps * BATCH / max_over_ranks(float(w)) for w in win_s]
        steady.append({"value": float(np.median(rates)), "unit": UNIT, "windows": rates,
                       "p50_ms": float(np.percentile(win_lat, 50) * 1e3), "p99_ms": float(np.percentile(win_lat, 99) * 1e3),
                       "requests": args.steps,
                       "how": f"median of {n_win} consecutive windows of {args.steps} completions each (completions {e2e_warm + 1}.."
                              f"{e2e_warm + n_win * args.steps}) of ONE continuous closed loop of {e2e_warm + n_win * args.steps + 2 * BUFFERS} "
                              "requests (InferBench::Run); every request still does its pinned H2D, forward and D2H inside the loop"})
        mgr.close()
        return (world * args.steps * BATCH / wall,
                float(np.percentile(lats, 50) * 1e3) if len(lats) else None,
                float(np.percentile(lats, 99) * 1e3) if len(lats) else None,
                res["kGpuComputeTimePerBatch"] * 1e3)

    br_value, br_p50, br_p99, e2e_gpu_ms = e2e_run(blob)
    # headline e2e = the steady-state window (see e2e_run); the bracketed run of the same K requests is reported beside it
    e2e_value, p50, p99 = steady[0]["value"], steady[0]["p50_ms"], steady[0]["p99_ms"]
    # secondary mode (SURVEY.md 8d): the same engine with an fp16 input binding -- half the H2D bytes per request
    blob_h = builder.build_resnet_plan(50, builder.PREC_FP16, BATCH, seed=0, input_dtype="f16")
    e2e_run(blob_h)
    e2e_h_value, p50_h, p99_h = steady[1]["value"], steady[1]["p50_ms"], steady[1]["p99_ms"]

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- rank 0 only: per-layer share (live CUDA events), roofline, CPU baseline ---------------------------
    eng = capi.Engine(blob)
    sess = capi.Session(eng)
    sess.infer(ring[0])
    prof = sess.profile(BATCH)
    prof = sess.profile(BATCH)
    total_ms = sum(p["ms"] for p in prof)
    conv = [p for p in prof if p["name"].startswith("conv_tcgen05")]
    conv_ms = sum(p["ms"] for p in conv)
    conv_flops = sum(p["flops"] for p in conv)
    conv_share = conv_ms / total_ms if total_ms > 0 else 1.0
    n_conv = len(conv)
    sess.close()
    eng.destroy()
    # the same kernels WITHOUT other contexts to overlap with: one context, one stream (latency-bound at batch 8)
    iso_steps = max(20, min(args.steps, 400))
    iso_ms, _ = capi.device_throughput(blob, 1, BATCH, iso_steps, 10, ring)
    iso_ms_per_step = iso_ms / iso_steps

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
        peak_tf, peak_src = float(peaks["bf16_tflops_sustained"]), "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
        peak_hbm = float(peaks["hbm_gbs"])
    except Exception:
        peak_tf, peak_src, peak_hbm = 1400.0, "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)", 6650.0
    # the conv kernel's time inside one step of the timed region = step time x its share of the forward pass
    conv_ms_per_step = ms_per_step * conv_share
    achieved_tf = conv_flops / (conv_ms_per_step * 1e-3) / 1e12
    roofline = {
        "bound": "tensor", "kernel": "conv_f16_tcgen05 (all %d conv launches of one forward pass)" % n_conv,
        "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
        # DRAM bytes (read+write) of the 53 conv launches of ONE forward pass = one step, from the committed ncu pass
        # profiles/ncu_metrics_r2l.csv (cold L2; outputs stay L2-resident inside each kernel)
        "traffic": 267.3e6, "traffic_source": "profiles/ncu_metrics_r2l.csv",
        "peak_source": peak_src,
        "flops_per_step": conv_flops, "conv_share_of_step": conv_share,
        # aggregate over 4 overlapping contexts (above) vs the kernels in isolation on ONE stream: conv FLOPs / (single-
        # stream step time x conv share) -- at batch 8 a lone forward pass is a chain of ~56 dependent, latency-bound launches
        "per_kernel_isolated": {"achieved": conv_flops / (iso_ms_per_step * conv_share * 1e-3) / 1e12,
                                "frac": conv_flops / (iso_ms_per_step * conv_share * 1e-3) / 1e12 / peak_tf,
                                "ms_per_step_single_stream": iso_ms_per_step, "steps": iso_steps},
        "hbm_view": {"algorithmic_bytes_per_step": ALGO_BYTES_PER_STEP,
                     "achieved_gbs": ALGO_BYTES_PER_STEP / (ms_per_step * 1e-3) / 1e9, "peak_gbs": peak_hbm},
    }
    try:
        # every convolution against the roof that binds IT: the tensor peak, or -- for the wide short-K layers whose
        # activations live in L2 -- the read / write bandwidth of L2 for unique streaming data (tensorrt_laboratory_b200/roofs.py)
        from tensorrt_laboratory_b200 import graph, roofs, weights
        net = graph.resnet_caffe(50)
        floors = roofs.conv_floors(graph.lower(net, weights.random_weights(net, 0)), BATCH, peak_tf)
        floor_us = sum(f["floor_us"] for f in floors)
        roofline["per_layer_roofs"] = {
            "floor_us_per_step": floor_us, "frac": floor_us / (conv_ms_per_step * 1e3),
            "tensor_bound_layers": sum(f["roof"] == "tensor" for f in floors), "memory_bound_layers": sum(f["roof"] == "memory" for f in floors),
            "tensor_floor_us": sum(f["tensor_floor_us"] for f in floors), "memory_floor_us": sum(f["memory_floor_us"] for f in floors),
            "l2_read_tbs": roofs.L2_READ_BPS / 1e12, "l2_write_tbs": roofs.L2_WRITE_BPS / 1e12,
            "source": "per layer max(2MNK / tensor peak, reads / L2 read bw + writes / L2 write bw); L2 figures: tools/micro/l2_stream.cu, "
                      "profiles/l2_stream_r2.log; per-layer table: profiles/roofline_r2_saturated.md"}
    except Exception as ex:  # an explanatory view must never take the line down
        roofline["per_layer_roofs"] = {"error": f"{type(ex).__name__}: {ex}"}

    config2 = None
    if world == 1 and not args.no_config2:
        try:
            config2 = run_config2(capi, builder)
        except Exception as ex:  # the secondary line must never take the headline down
            config2 = {"error": f"{type(ex).__name__}: {ex}"}

    cpu = None
    try:
        import onnxruntime  # noqa: F401  (the north star names ONNX Runtime for the CPU leg)
        ort = "importable but unused: the torch oracle port is what the tests pin"
    except Exception:
        ort = "onnxruntime is not installed on this box: torch-CPU oracle port instead"
    if not args.no_cpu:
        net, wts = cpu_forward_setup()
        cores = pick_cpu_threads(net, wts, ring)
        ips, spb = time_cpu(net, wts, ring, 3, args.cpu_batches, cores)
        cpu = {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "onnxruntime": ort,
               "sample": f"3 warm-up + {args.cpu_batches} timed batches of {BATCH} (same graph/weights/inputs), fp32 torch-CPU oracle port, {cores} threads of {usable_cores()} usable cores, {spb*1e3:.1f} ms/batch"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": "ResNet-50 fp16 batch=8, 1xB200 per replica, 4 concurrent ExecutionContexts/streams, synthetic 3x224x224 (BASELINE.json configs[1])",
                   "global_batch": BATCH * world, "contexts": CONTEXTS, "buffers": BUFFERS,
                   "l2_policy": f"inputs larger than L2: ring of {RING} distinct batches = {RING * in_bytes / 1e6:.0f} MB",
                   "parallelism": f"replicas x{world} (no collective)",
                   "host_sync": "blocking" if blocking else "spin", "host_cores": usable_cores(),
                   "gpu_affinity_cpus": affinity_cpus,
                   "enqueue_depth": int(os.environ.get("TRTLAB_ENQUEUE_DEPTH", "2"))},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
                "p50_ms": p50, "p99_ms": p99, "gpu_ms_per_request": e2e_gpu_ms,
                "requests": args.steps, "warm_requests": e2e_warm,
                "per_rank_bracketed": per_rank[0], "h2d_gbs_per_rank_bracketed": [v / BATCH * in_bytes / 1e9 for v in per_rank[0]],
                "timed_region": steady[0]["how"], "windows": steady[0]["windows"],
                "bracketed": {"value": br_value, "unit": UNIT, "p50_ms": br_p50, "p99_ms": br_p99,
                              "how": "the same K requests as a run of their own (clock starts with an EMPTY pipeline and stops when it has "
                                     "drained): at K = 20 this is mostly the fill and drain of the 8-Buffers pipeline"},
                "api": "InferenceManager+InferRunner+InferBench (pinned host Buffers, H2D/D2H per request)"},
        "e2e_fp16_input": {"value": e2e_h_value, "unit": UNIT, "h2d_bytes_per_step": in_bytes // 2, "d2h_bytes_per_step": out_bytes,
                           "p50_ms": p50_h, "p99_ms": p99_h,
                           "note": "SECONDARY mode: same engine, input binding declared fp16 (not the reference's fp32 binding contract)"},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "tflops_whole_forward": flops_step / (ms_per_step * 1e-3) / 1e12,
        "config2": config2,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-batches", type=int, default=20)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-config2", action="store_true", help="skip the secondary ResNet-152 INT8 line (BASELINE configs[2])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the headline leg's last timed step (its input: "
                    f"batch (steps - 1) mod {RING} of the seeded input ring) as DIR/<binding>.npy, float32")
    args = ap.parse_args()
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 implementation")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: re-launch ourselves one rank per GPU (the driver does this itself via torchrun)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
