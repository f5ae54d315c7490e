#!/usr/bin/env python
"""bench.py - end-to-end FPS of the SMAP inference hot path (backbone + association + 3D lift) on B200.

Usage: `python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]`, under torchrun for
N > 1; one JSON line on stdout from rank 0.

A "step" = one pass of the whole hot path over one batch of B synthetic 832x512 frames per GPU
(BASELINE.json configs[1]: batch=8, 1xB200, full backbone + GPU association; for N > 1 each rank owns its own
B frames and the per-image skeleton records are exchanged with ONE NCCL all-gather per step - weak scaling).

  value : frames/s with the input batch already resident in HBM (smapb_infer_device + all-gather)
  e2e   : frames/s through the C-ABI call with HOST buffers (smapb_infer_host: H2D of the frames from pinned
          memory, the whole path, D2H of the skeleton records) + all-gather
  roofline : the tensor-core convolution kernel (conv_tc_kernel, the dominant kernel): algorithmic conv FLOPs of
          one step / (its share of the step, from per-launch CUDA events, x the timed ms_per_step), against
          MEASURED_PEAKS.json bf16_tflops_sustained.
          In bf16x3 mode every algorithmic FLOP is issued as 3 tensor-core FLOPs, so the tensor pipe runs at
          3 x frac of the bf16 peak.
  --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed device-resident step returned (the
          skeleton records of its B frames, all ranks' with N > 1) as DIR/pred2d.npy (float32 [F,127,15,4]), pred3d.npy
          (float64 [F,127,15,4]), root_depth.npy (float64 [F,127]) and count.npy (float64 [F]).  Inputs and weights are
          seeded, so the same arguments give the same inputs on every run and two builds can be compared array by array.
  cpu_baseline : the CPU oracle of the same path (oracle/: PyTorch fp32 backbone on all cores + C++ association
          + numpy lift) on a bounded sample of the same workload.
`--impl reference` times that CPU oracle alone (the reference has no GPU-free path of its own for the association
and /root/reference does not exist on the GPU box; see DESIGN.md).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IN_H, IN_W = 512, 832
WORKLOAD = "configs[1]: batch=8 832x512 synthetic frames per GPU, random-init SMAP weights, full backbone + association + lift"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="smap_b200", choices=["smap_b200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="frames per GPU per step")
    ap.add_argument("--flip", type=int, default=0, help="flip-TTA (doubles the backbone work); BASELINE configs use 0")
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--engines", type=int, default=int(os.environ.get("SMAPB_BENCH_ENGINES", "2")),
                    help="handles per GPU: >1 keeps that many batches in flight on independent streams")
    ap.add_argument("--profile-csv", default="")
    ap.add_argument("--ncu-one-step", action="store_true",
                    help="bracket exactly one device-resident step with cudaProfilerStart/Stop and exit (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the records of the last timed step as DIR/<field>.npy (float32/float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "smap_b200":
        ap.error("--dump-outputs needs --impl smap_b200")
    return args


def dump_outputs(out_dir, rec):
    """Records (uint8 [F, RECORD_BYTES], any device) -> out_dir/{pred2d,pred3d,root_depth,count}.npy."""
    from smap_b200.engine import records_to_numpy

    os.makedirs(out_dir, exist_ok=True)
    r = records_to_numpy(rec)
    for name in ("pred2d", "pred3d", "root_depth"):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(r[name]))
    np.save(os.path.join(out_dir, "count.npy"), r["count"].astype(np.float64))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe).  NVML in-process (a sample every
    few ms, so that even a 0.2 s timed region gets tens of samples); `nvidia-smi` polling (~0.15 s per sample) only when
    the NVML binding is missing."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self.stop_flag = False
        self.source = "nvml"
        self.nvml = self.handle = None
        try:
            import pynvml

            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber the devices: address the GPU by the UUID torch reports
            import torch

            try:
                uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nvml = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = self.handle = None
            self.source = "nvidia-smi"

    def _nvml_sample(self):
        n = self.nvml
        self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for bit, name in self.REASONS.items():
            if mask & bit:
                self.reasons.add(name)

    def run(self):
        if self.nvml is not None:
            while not self.stop_flag:
                try:
                    self._nvml_sample()
                except Exception:
                    pass
                time.sleep(0.005)
            return
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.15)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "source": self.source}


# ------------------------------------------------------------------------------------------------
# CPU oracle legs (the only place bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU legs may use: the affinity mask, clipped by the cgroup CPU quota, at most 64."""
    n = len(os.sched_getaffinity(0))
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 64))


_PICKED_THREADS = None


def pick_threads():
    """The GPU boxes are shared: with more runnable threads than free cores oneDNN's barriers collapse (measured: 128
    threads -> 100 s per frame instead of 1.4 s).  Probe one backbone-sized convolution at a few thread counts and keep
    the fastest; costs well under a second when the box is healthy."""
    global _PICKED_THREADS
    if _PICKED_THREADS is not None:
        return _PICKED_THREADS
    import torch

    top = host_threads()
    x = torch.randn(1, 256, 64, 104)
    w = torch.randn(256, 256, 3, 3)
    best_t, best = top, 1e30
    for t in sorted({top, max(1, top // 2), max(1, top // 4), min(top, 16)}, reverse=True):
        torch.set_num_threads(t)
        dt = 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            torch.nn.functional.conv2d(x, w, padding=1)
            dt = min(dt, time.perf_counter() - t0)
        if dt < best * 0.9:  # prefer more threads unless fewer are clearly faster
            best, best_t = dt, t
    _PICKED_THREADS = best_t
    return best_t


class CpuOracle:
    """Whole path on the host: oracle backbone (torch fp32, all host threads) + C++ association (single thread, as the
    reference's is: its OpenMP pragmas are commented out, extensions/association.cpp:79,100) + numpy lift.  Weights, the
    association library and the scale record are set up ONCE (outside every timed region)."""

    def __init__(self, threads=None):
        import torch

        from oracle import assoc, lift_numpy, smap_torch

        self.torch, self.assoc, self.lift_numpy, self.smap_torch = torch, assoc, lift_numpy, smap_torch
        # host cores (torchrun exports OMP_NUM_THREADS=1, which would starve the CPU baseline)
        torch.set_num_threads(threads or pick_threads())
        self.threads = torch.get_num_threads()
        self.sd = smap_torch.make_state_dict(0, "identity")
        self.scale = lift_numpy.default_scale(1920, 1080)
        assoc.lib()

    def make_frames(self, n, seed=1):
        return self.smap_torch.make_input(n, IN_H, IN_W, seed=seed)

    def run(self, x, budget_s=None):
        """-> (seconds, frames_done, persons): the frames of x one by one, stopping early (after at least one) when
        budget_s seconds are used up."""
        t0 = time.perf_counter()
        persons = done = 0
        for i in range(x.shape[0]):
            hm, dd, rd = self.smap_torch.smap_forward(self.sd, x[i:i + 1])
            self.smap_torch.rescale_reference_cuda(hm)
            bodies = self.assoc.connect(hm[0].numpy(), rd[0, 0].numpy())
            p2, p3, rdep = self.lift_numpy.lift(bodies, dd[0].numpy(), rd[0, 0].numpy(), self.scale)
            persons += len(p2)
            done += 1
            if budget_s is not None and time.perf_counter() - t0 >= budget_s:
                break
        return time.perf_counter() - t0, done, persons


def ref_gpu_path_note():
    """The reference's own single-GPU path (eager PyTorch/cuDNN backbone + unmodified dapalib per image + numpy lift) is
    measured builder-side by tests/ref_gpu_compare.py on the same kind of box; bench.py only quotes the committed numbers."""
    p = os.path.join(ROOT, "profiles", "r02_reference_gpu_path.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    bb, e2e = d.get("backbone_only", {}), d.get("whole_gpu_path", {})
    return {"value": d.get("value"), "unit": "frames/s", "what": d.get("what"),
            "config4_15_persons_frames_per_s": e2e.get("reference_config4_15_persons", {}).get("frames_per_s"),
            "backbone_only_ms_per_batch8": {"cudnn_tf32": bb.get("eager_cudnn_tf32_True_benchmark_False", {}).get("ms_per_batch"),
                                            "cudnn_fp32": bb.get("eager_cudnn_tf32_False_benchmark_False", {}).get("ms_per_batch"),
                                            "smap_b200_bf16x3": bb.get("smap_b200_bf16x3", {}).get("ms_per_batch")},
            "source": "profiles/r02_reference_gpu_path.json (tests/ref_gpu_compare.py, builder-side run on a B200)"}


def run_reference(args):
    """Reference arm: the CPU port of the whole path (oracle/) on the box's host cores; each step = a bounded sample of
    the workload (1 frame of the 8-frame batch).  Only the per-frame work is inside the timed region."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frames_per_step = 1
    oracle = CpuOracle()
    xs = [oracle.make_frames(frames_per_step, seed=1 + s) for s in range(args.warmup + args.steps)]
    for s in range(args.warmup):
        oracle.run(xs[s])
    t0 = time.perf_counter()
    for s in range(args.steps):
        oracle.run(xs[args.warmup + s])
    total = time.perf_counter() - t0
    value = args.steps * frames_per_step / total
    line = {
        "impl": "reference", "metric": "end-to-end FPS @832x512 (backbone+association+lift)", "value": value,
        "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": frames_per_step,
                   "arm": "cpu port of the reference path (oracle/); the reference has no GPU-free association of its own "
                          "and /root/reference does not travel to the GPU box"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": oracle.threads, "kind": "port",
                         "sample": "%d frame(s) per step x %d steps, whole path on host cores; weights/input/library set up "
                                   "outside the timed region" % (frames_per_step, args.steps)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    g = ref_gpu_path_note()
    if g:
        line["reference_gpu_path"] = g
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from smap_b200 import dist as sdist
    from smap_b200 import schema
    from smap_b200.engine import RECORD_BYTES, Engine, scale_row

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    sd0 = schema.make_state_dict(0, "identity")
    NE = max(1, args.engines)
    # one handle per batch in flight; every handle issues on its OWN non-blocking stream (nothing in the timed loops
    # touches the legacy default stream) and owns its NCCL communicator, so the per-step all-gather is ordered only
    # against the batch it belongs to
    engines = []
    for _ in range(NE):
        e = Engine(local, max_batch=B, in_h=IN_H, in_w=IN_W, stream=torch.cuda.Stream(dev))
        e.load_state_dict(sd0, precision=args.precision)
        engines.append(e)
    gather = world > 1 and not os.environ.get("SMAPB_BENCH_NO_GATHER")  # (diagnostic switch: N independent replicas)
    if gather:
        for e in engines:
            e.init_comm()
    eng = engines[0]
    cur = torch.cuda.current_stream()

    # inputs: NROT distinct batches so that consecutive steps never re-read the same frames from L2
    NROT = 4
    host_batches = [schema.make_input(B, IN_H, IN_W, seed=1 + rank * 100 + r).pin_memory() for r in range(NROT)]
    dev_batches = [hb.to(dev) for hb in host_batches]
    sc = dict(scale=IN_W / 1920, img_width=1920, img_height=1080, net_width=IN_W, net_height=IN_H, f_x=1920.0,
              f_y=1920.0, cx=960.0, cy=540.0)
    scales_host = torch.from_numpy(np.stack([scale_row(sc)] * B)).pin_memory()
    scales_dev = scales_host.to(dev)
    NOUT = B * (world if gather else 1)
    dev_outs = [torch.empty(NOUT, RECORD_BYTES, dtype=torch.uint8, device=dev) for _ in range(NE)]
    torch.cuda.synchronize()
    if gather:
        # tile shapes: the committed table covers this workload; anything it does not cover is tuned by rank 0 only
        if rank == 0:
            eng.infer_device(dev_batches[0], scales_dev, out=torch.empty(B, RECORD_BYTES, dtype=torch.uint8, device=dev))
            torch.cuda.synchronize()
        dist.barrier()
        sdist.sync_tile_table()

    def step_device(i):
        # whole path + ONE ncclAllGather of the skeleton records per step (world > 1): the path on the handle's stream (CUDA
        # graph), the exchange behind an event on the handle's gather stream, so that no rank's compute waits for a peer
        engines[i % NE].infer_device(dev_batches[i % NROT], scales_dev, do_flip=bool(args.flip), out=dev_outs[i % NE],
                                     gather=gather, defer=gather and not os.environ.get("SMAPB_BENCH_SYNC_GATHER"))

    DEPTH = 2 * NE  # batches in flight on the host path: two slots per handle
    host_outs = [torch.empty(NOUT, RECORD_BYTES, dtype=torch.uint8).pin_memory() for _ in range(DEPTH)]

    def finish_host(j):
        engines[j % NE].wait((j // NE) % 2)  # step j's (gathered) records are in host memory

    def step_host(i, last=False):
        # pipeline through the C ABI (two slots per handle): the H2D of step i overlaps the compute of earlier steps;
        # every step still performs its own H2D (pinned frames) and D2H (records) inside the timed region.  With
        # world > 1 the records are all-gathered on the device before the single D2H.
        if i >= DEPTH:
            finish_host(i - DEPTH)
        engines[i % NE].submit_host((i // NE) % 2, host_batches[i % NROT], scales_host, host_outs[i % DEPTH],
                                    do_flip=bool(args.flip), gather=gather)
        if last:
            for j in range(max(0, i - DEPTH + 1), i + 1):
                finish_host(j)

    def run_device(steps):
        for i in range(steps):
            step_device(i)

    def run_host(steps):
        for i in range(steps):
            step_host(i, last=(i == steps - 1))

    def timed(fn, steps):
        """CUDA events bracketing every stream the step uses: e0 on the current stream, every handle stream waits for it;
        every handle stream is joined back before e1.  Barrier + synchronize on both sides, max over ranks."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(cur)
        for e in engines:
            e.stream.wait_event(e0)
        fn(steps)
        for e in engines:
            if gather:
                e.gather_sync()  # every exchange of the timed steps has completed before e1
            cur.wait_stream(e.stream)
        e1.record(cur)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        per_rank = [ms / steps]
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
            allt = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            per_rank = [float(a[0]) / steps for a in allt]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = t[0].item(), t[1].item() * 1e-3
            dist.barrier()
        timed.per_rank = per_rank
        return ms, wall

    # SETUP (not warm-up, not timed): every (handle, input batch) pair the loops will use goes through its two eager
    # runs (lazy allocations, NCCL connections) and its CUDA-graph capture.  Then exactly --warmup untimed steps.
    n_setup = 3 * NE * NROT // math.gcd(NE, NROT)
    run_device(n_setup)
    torch.cuda.synchronize()
    if args.ncu_one_step:
        torch.cuda.profiler.start()
        step_device(0)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        for e in engines:
            e.close()
        return
    run_device(args.warmup)
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    l0 = sum(e.launch_count() for e in engines)
    ms_dev, wall_dev = timed(run_device, args.steps)
    per_rank_ms = timed.per_rank
    launches = sum(e.launch_count() for e in engines) - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dev_outs[(args.steps - 1) % NE])  # step i wrote dev_outs[i % NE]

    run_host(max(DEPTH, args.warmup))  # slot buffers + graphs for the slot pointers, then the host warm-up
    torch.cuda.synchronize()
    ms_host, wall_host = timed(run_host, args.steps)
    sampler.stop_flag = True  # the clock sampler covers both timed regions (device-resident and host-buffer steps)
    sampler.join(timeout=2)

    # roofline leg: per-kernel CUDA events on the launching stream (one handle, eager, every launch bracketed) give each
    # kernel's SHARE of the serialised step; the headline mode (graph replay, NE handles overlapping) cannot be
    # event-bracketed per kernel, so the kernel time in that mode is share x the timed ms_per_step.
    n_conv, conv_flops = eng.plan_info(B)
    prof_steps = min(args.steps, 5)
    prof_out = torch.empty(B, RECORD_BYTES, dtype=torch.uint8, device=dev)
    eng.profile_begin()
    for i in range(prof_steps):
        eng.infer_device(dev_batches[i % NROT], scales_dev, do_flip=bool(args.flip), out=prof_out)
    prof = eng.profile_end(args.profile_csv or None)
    torch.cuda.synchronize()

    if rank == 0:
        peak_tf, peak_bw, peak_src = measured_peaks()
        frames = world * B * args.steps
        value = frames / (ms_dev * 1e-3)
        e2e = frames / (wall_host)
        ms_per_step = ms_dev / args.steps
        conv_ms, conv_n = prof["conv"]
        fwd = 2 if args.flip else 1
        total_prof_ms = sum(v[0] for v in prof.values()) / prof_steps
        conv_ms_serial = conv_ms / prof_steps
        share = conv_ms_serial / total_prof_ms
        conv_ms_per_step = share * ms_per_step  # in the timed (graph, NE handles) mode
        achieved = conv_flops * fwd / (conv_ms_per_step * 1e-3) * 1e-12 if conv_ms_per_step > 0 else 0.0
        traffic, traffic_src = None, None
        for name in ("r02_conv_traffic.json", "r01_conv_traffic.json"):
            tp = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tp):  # committed ncu capture of the same command (tools/gpu_profile.sh)
                tj = json.load(open(tp))
                traffic, traffic_src = tj["mean_dram_bytes_per_launch"], "profiles/" + name
                break
        # association (nms + paf + group) against the HBM roofline: algorithmic bytes per frame (SURVEY 8(d)) = heat-maps
        # read once 43*128*208*4 + root-depth map 128*208*4 + skeleton records written
        assoc_ms = prof["assoc"][0] / prof_steps
        assoc_bytes = B * (43 * 128 * 208 * 4 + 128 * 208 * 4 + 127 * 15 * 4 * 4)
        assoc_gbs = assoc_bytes / (assoc_ms * 1e-3) * 1e-9 if assoc_ms > 0 else 0.0
        line = {
            "metric": "end-to-end FPS @832x512 (backbone+association+lift)", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate; fp32-faithful)" if args.precision == "bf16x3" else "bf16",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_gpu_per_step": B, "flip_tta": int(args.flip),
                       "l2": "inputs rotate over %d distinct batches (%.0f MB) and every step streams >2 GB of activations (> 126 MB L2)"
                             % (NROT, NROT * B * 3 * IN_H * IN_W * 4 / 1e6),
                       "parallelism": "dp%d, one ncclAllGather of skeleton records per step (handle-owned communicator, gather stream behind an event)" % world,
                       "batches_in_flight_per_gpu": NE,
                       "setup_steps_before_warmup": n_setup,
                       "setup": "graph capture per (handle, input batch) pair; not warm-up, not timed"},
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": B * 3 * IN_H * IN_W * 4 + B * 9 * 8,
                    "d2h_bytes_per_step": NOUT * RECORD_BYTES, "ms_per_step": 1e3 * wall_host / args.steps,
                    "batches_in_flight_per_gpu": DEPTH},
            "gpu_launches": int(launches),
            "ms_per_step_per_rank": [round(v, 4) for v in per_rank_ms],
            "clocks": sampler.result(),
            "roofline": {"bound": "tensor", "kernel": "conv_tc_kernel (%d launches/step)" % (conv_n // prof_steps),
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "peak_source": peak_src + " bf16_tflops_sustained",
                         "algorithmic_gflop_per_step": conv_flops * fwd * 1e-9,
                         "tensor_pipe_flop_multiplier": 3 if args.precision == "bf16x3" else 1,
                         "kernel_ms_per_step": conv_ms_per_step, "share_of_step": share,
                         "how": "share (per-launch CUDA events, one handle, eager) x timed ms_per_step (graph replay, %d handles)" % NE,
                         "kernel_ms_per_step_serialised_eager": conv_ms_serial,
                         "traffic": traffic, "traffic_unit": "bytes per launch (dram read+write, ncu)",
                         "traffic_source": traffic_src},
            "roofline_assoc": {"bound": "hbm", "kernel": "nms_kernel + paf_kernel + group_kernel",
                               "achieved": assoc_gbs, "peak": peak_bw, "unit": "GB/s", "frac": assoc_gbs / peak_bw,
                               "algorithmic_bytes_per_step": assoc_bytes, "kernel_ms_per_step": assoc_ms,
                               "note": "batch 8: 3 launches of 120 / 112 / 8 CTAs - latency bound, not bandwidth bound; the "
                                       "B=64 ncu capture in profiles/ is the bandwidth number"},
            "breakdown_ms_per_step": {k: v[0] / prof_steps for k, v in prof.items() if v[1]},
        }
        g = ref_gpu_path_note()
        if g:
            line["reference_gpu_path"] = dict(g, ratio_value=value / g["value"] if g.get("value") else None)
        if not args.no_cpu_baseline:
            oracle = CpuOracle()
            x = oracle.make_frames(8)
            dt, nfr, persons = oracle.run(x, budget_s=20.0)
            line["cpu_baseline"] = {"value": nfr / dt, "unit": "frames/s", "cores": oracle.threads, "kind": "port",
                                    "sample": "%d frames of the same workload (bounded to ~20 s), whole path (oracle/: torch fp32 "
                                              "backbone on %d threads + single-thread C++ association + numpy lift), %.1f s"
                                              % (nfr, oracle.threads, dt)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
    for e in engines:
        e.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
