#!/usr/bin/env python
"""Benchmark of the SiamMask per-frame inference hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU cores
    python bench.py --config {2,3,5} ...                     # BASELINE.json configs[1..4] presets (default: 2 -> configs[1])

One "step" = one pass of the hot path over one batch of synthetic search regions — the whole frame of
`siamese_track` (tools/test.py:201-261): `track_mask` (backbone -> depthwise xcorr -> cls/loc/mask heads) ->
score/box post-processing + argmax ON THE DEVICE -> `track_refine` at the selected position, for B paired tracker
streams per GPU (BASELINE.json configs[1]: "batch=64 synthetic search regions, 1xB200, full track() path with mask
refine"); templates are cached per slot (configs[3]).  N>1: one process per GPU (torchrun), streams are sharded, the
packed weights are broadcast ONCE over NCCL at init, no per-frame collective ("weak" scaling).

Prints ONE JSON line (rank 0).  `value` = whole-job frames/s with inputs resident in HBM (C ABI `sm_step`); `e2e` =
the same frame through the host-buffer call `sm_step_host_async` (H2D of every frame + target sizes, D2H of the
records and refine logits inside the timed region, SAME flags as `value`); `roofline` = the tensor-core conv family
(dominant kernel) timed per launch with CUDA events; `cpu_baseline` = the oracle port of the reference timed on all of
this box's host cores; `parity_check` = max relative error of this run's outputs against the CPU oracle.
`value` times exactly --steps steps; the `e2e` region is at least --min-seconds long (default 2 s).
--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, see `dump_step_outputs`.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "search-region frames/sec (127/255 SiamMask-sharp)"
GFLOP_SHARP = {255: 33.915, 383: 77.938}              # BASELINE.md §2 (algorithmic, conv_kernel cached)
GFLOP_RPN = {255: 30.811, 383: 71.139}
XCORR_BYTES = {255: 1526784, 383: 3820544}            # per branch per frame, fp32 algorithmic (BASELINE.md §2)
PENALTY_K, WINDOW_INFLUENCE = 0.04, 0.4               # config_davis.json hp


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "tflops_burst": d["bf16_tflops"], "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  The process is
    started (and its first sample awaited) before the warm-up, so its start-up cost never lands inside the timed
    region; a reader thread time-stamps every sample and `stop()` keeps those inside [t0, t1]."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, uuid):
        import threading
        self.proc, self.lines = None, []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", uuid, f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.first = threading.Event()

        def reader():
            for line in self.proc.stdout:
                self.lines.append((time.perf_counter(), line))
                self.first.set()
        self.thread = threading.Thread(target=reader, daemon=True)
        self.thread.start()
        self.first.wait(5.0)

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        self.thread.join(5.0)
        sm, mx, pw, reasons = [], [], [], set()
        for ts, line in self.lines:
            if not (t0 <= ts <= t1 + 0.03):
                continue
            f = [t.strip() for t in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(self.NAMES, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples inside the timed region"]}
        bad = reasons & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        stuck = statistics.median(sm) < 0.6 * max(mx) and not reasons
        return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons), "rejected": bool(bad or stuck)}


# ---------------------------------------------------------------------------------------------------
# the reference's CPU implementation of the path (oracle port), on ALL host cores
def _cpu_worker(args):
    """One CPU worker process: B=`ref_batch` paired frames per step, `threads` torch threads.  Waits for the common
    start time, then runs for `seconds` (or `steps` steps) and prints {"frames": n, "seconds": dt}."""
    import torch
    from oracle.siammask_oracle import Oracle
    from siammask_b200.checkpoint import synthetic_state_dict
    torch.set_num_threads(args.threads)
    sd = synthetic_state_dict(0, mask=not args.rpn_only, refine=not args.rpn_only)
    bs = args.ref_batch
    g = torch.Generator().manual_seed(1 + args.worker_id)
    z = torch.rand(bs, 3, 127, 127, generator=g) * 255
    xs = [torch.rand(bs, 3, args.search, args.search, generator=g) * 255 for _ in range(2)]
    o = Oracle(sd)
    o.template(z)

    def step(i):
        if args.rpn_only:
            o.track(xs[i % 2])
        else:
            o.track_mask(xs[i % 2])
            o.track_refine((12, 12))
    for i in range(max(1, args.warmup)):
        step(i)
    print("READY", flush=True)
    sys.stdin.readline()                      # the parent releases all workers together
    n, t0 = 0, time.perf_counter()
    if args.worker_seconds > 0:
        while time.perf_counter() - t0 < args.worker_seconds:
            step(n); n += 1
    else:
        for i in range(args.steps):
            step(i); n += 1
    dt = time.perf_counter() - t0
    print(json.dumps({"frames": n * bs, "seconds": dt, "steps": n}), flush=True)


def cpu_quota():
    """CPUs this container may actually use: min(os.cpu_count(), cgroup quota)."""
    n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(math.ceil(int(q) / int(per)))))
    except (OSError, ValueError):
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    return n


def _run_fleet(args, nproc, threads, seconds, steps):
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), MKL_NUM_THREADS=str(threads))
    procs = []
    for w in range(nproc):
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "_cpu_worker", "--threads", str(threads),
               "--worker-id", str(w), "--worker-seconds", str(seconds), "--steps", str(steps), "--warmup",
               str(args.warmup), "--search", str(args.search), "--ref-batch", str(args.ref_batch)]
        if args.rpn_only:
            cmd.append("--rpn-only")
        procs.append(subprocess.Popen(cmd, stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True, env=env))
    for p in procs:
        line = p.stdout.readline()
        if "READY" not in line:
            raise RuntimeError("cpu worker failed to start: " + line)
    for p in procs:
        p.stdin.write("go\n"); p.stdin.flush()
    frames, longest = 0, 0.0
    for p in procs:
        rec = json.loads(p.stdout.readline())
        frames += rec["frames"]; longest = max(longest, rec["seconds"])
        p.wait(30)
    return frames, max(longest, 1e-9)


def run_cpu_fleet(args, seconds=0.0, steps=0):
    """The reference algorithm on ALL usable host cores.  The path shards over independent streams on the CPU exactly
    as it does over GPUs, so the host's best configuration is some number of worker processes x torch threads; which
    one wins depends on the box (torch's CPU convs stop scaling at ~16 threads per process; memory bandwidth and the
    container's CPU quota cap the fleet).  A short probe tries the candidate layouts, the best one is then timed for
    `seconds` (or `steps` steps per worker).  Returns (frames/s, cores used, description, seconds)."""
    ncpu = cpu_quota()
    if args.cpu_threads > 0:
        layouts = [(max(1, ncpu // args.cpu_threads), args.cpu_threads)]
    else:
        layouts = sorted({(max(1, ncpu // t), t) for t in (4, 8, 16, 32) if t <= ncpu} |
                         {(1, t) for t in (16, 32) if t <= ncpu} | ({(1, ncpu)} if ncpu <= 8 else set()))
    best, best_rate, probes = layouts[0], 0.0, []
    if len(layouts) > 1:
        for nproc, threads in layouts:
            fr, dt = _run_fleet(args, nproc, threads, 2.0, 0)
            probes.append(f"{nproc}x{threads}:{fr / dt:.1f}")
            if fr / dt > best_rate:
                best, best_rate = (nproc, threads), fr / dt
    nproc, threads = best
    frames, dt = _run_fleet(args, nproc, threads, seconds, steps)
    what = "track" if args.rpn_only else "track_mask+track_refine"
    sample = (f"{nproc} worker process(es) x {threads} torch threads = {nproc * threads} of {ncpu} usable host CPUs "
              f"(os.cpu_count {os.cpu_count()}), each B={args.ref_batch} paired frames per step, {what}, oracle port "
              f"(torch CPU fp32), {frames} frames in {dt:.1f} s; layout = best of a 2 s probe each "
              f"[processes x threads : frames/s] {' '.join(probes)}")
    return frames / dt, nproc * threads, sample, dt


def run_reference(args, rank):
    if rank != 0:
        return
    fps, cores, sample, dt = run_cpu_fleet(args, steps=args.steps)
    print(json.dumps({
        "impl": "reference", "metric": metric_name(args), "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.batch, max(1, args.gpus)),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "host_cpus": os.cpu_count(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def metric_name(args):
    return METRIC.replace("SiamMask-sharp", "SiamRPN-only") if args.rpn_only else METRIC.replace("255", str(args.search))


def workload_config(args, batch_per_gpu, world):
    R = (args.search - 127) // 8 + 9
    if args.rpn_only:
        what = "SiamRPN-only (experiments/siamrpn_resnet): track -> cls/loc + on-device score/box selection"
    else:
        what = ("SiamMask-sharp config_davis: track_mask (incl. 256->3969 mask head) + on-device score/box selection + "
                "track_refine at the selected position")
    return {"workload": f"{what}; template 127 / search {args.search}, response {R}x{R}, {batch_per_gpu} paired streams "
                        f"per GPU, templates cached per slot (BASELINE.json configs[{args.config - 1}])",
            "global_batch": batch_per_gpu * world, "batch_per_gpu": batch_per_gpu, "search": args.search,
            "parallelism": f"streams sharded over {world} GPU(s), one NCCL weight broadcast at init, "
                           "no per-frame collective; inside a GPU the batch runs as two concurrent lanes of "
                           "batch_per_gpu/2 streams (batches >= 16)",
            "l2": "inputs rotate over 4 device buffers (4 x 50 MB at B=64) and every step streams > 5 GB of "
                  "activations (>> 126 MB L2)"}


# ---------------------------------------------------------------------------------------------------
def cudnn_context(args, dev, seconds=1.5):
    """The de-facto 'existing Blackwell implementation' (SURVEY §2.3, §8d): the same network in PyTorch on this GPU
    (cuDNN/cuBLAS), fp32 strict and TF32 allowed, B=1 and the bench batch.  Context only — not the product path."""
    import torch
    from oracle.siammask_oracle import Oracle
    from siammask_b200.checkpoint import synthetic_state_dict
    sd = {k: v.to(dev) for k, v in synthetic_state_dict(0, mask=not args.rpn_only, refine=not args.rpn_only).items()}
    out = {}
    for tf32 in (False, True):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        for bs in (1, args.batch):
            try:
                g = torch.Generator(device=dev).manual_seed(5)
                o = Oracle(sd)
                o.template(torch.rand(bs, 3, 127, 127, device=dev, generator=g) * 255)
                x = torch.rand(bs, 3, args.search, args.search, device=dev, generator=g) * 255

                def one():
                    if args.rpn_only:
                        o.track(x)
                    else:
                        o.track_mask(x); o.track_refine((12, 12))
                for _ in range(3):
                    one()
                torch.cuda.synchronize(dev)
                n, t0 = 0, time.perf_counter()
                while time.perf_counter() - t0 < seconds:
                    one(); n += 1
                    torch.cuda.synchronize(dev)
                dt = time.perf_counter() - t0
                out[f"{'tf32' if tf32 else 'fp32'}_b{bs}"] = round(n * bs / dt, 1)
                del o, x
            except Exception as exc:                       # context only: never fail the bench on it
                out[f"{'tf32' if tf32 else 'fp32'}_b{bs}"] = f"failed: {type(exc).__name__}"
            torch.cuda.empty_cache()
    torch.backends.cudnn.allow_tf32 = True
    out["what"] = ("oracle port (torch functional restatement of the reference model) on this GPU via cuDNN/cuBLAS, "
                   "frames/s, shared refine position, eager mode")
    return out


def run_gpu(args, rank, local_rank, world):
    import ctypes as C
    import torch
    import torch.distributed as dist
    import siammask_b200 as smb
    from siammask_b200 import _lib, anchors as anc
    from siammask_b200.parallel import broadcast_weights, max_over_ranks, shard_streams

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    class _StdoutToStderr:
        """NCCL writes its version banner to stdout when the first communicator comes up; the contract of this script
        is ONE JSON line on stdout, so fd 1 points at stderr while the process group initialises."""
        def __enter__(self):
            sys.stdout.flush()
            self.saved = os.dup(1)
            os.dup2(2, 1)

        def __exit__(self, *exc):
            sys.stdout.flush()
            os.dup2(self.saved, 1)
            os.close(self.saved)

    if world > 1:
        with _StdoutToStderr():
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
    S = args.search
    sharp = not args.rpn_only
    # weak scaling: args.batch streams per GPU; this rank owns a contiguous block of the global stream ids
    B = len(shard_streams(args.batch * world, world, rank))
    R = (S - 127) // 8 + 9
    A = 5
    # two independent groups of B streams (slots [0,B) and [B,2B)) so the host-buffer pipeline can keep one step in
    # flight without pretending that frame k+1 of a tracker is available before frame k is finished
    m = smb.Custom(anchors=smb.DEFAULT_ANCHORS, search_size=S, max_batch=B, num_slots=2 * B, precision=args.precision,
                   mask=sharp)
    sd = smb.synthetic_state_dict(0, mask=sharp, refine=sharp)
    if rank == 0:
        m.load_state_dict(sd)
    m.eval().to(dev)
    if world > 1:                       # the one collective of the whole job: weights, once, at init
        with _StdoutToStderr():
            broadcast_weights(m.weight_blob(), src=0)
            torch.cuda.synchronize()
        if rank != 0:
            m.adopt_weights()
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    z = torch.rand(B, 3, 127, 127, device=dev, generator=gen) * 255
    xs = [torch.rand(B, 3, S, S, device=dev, generator=gen) * 255 for _ in range(4)]
    # what siamese_init prepares per stream (tools/test.py:142-161): anchors, cosine window, target size in the crop
    anchors_dev = torch.from_numpy(anc.generate_anchor(smb.DEFAULT_ANCHORS, R)).to(dev)
    window_dev = torch.from_numpy(anc.cosine_window(R, A).astype(np.float32)).to(dev)
    tsz_dev = (torch.rand(B, 2, device=dev, generator=gen) * 60 + 30).double()
    m.template(z, slot0=0)
    m.template(z, slot0=B)

    last = {}

    def step(i, mask_head=True):
        # the whole frame of siamese_track (tools/test.py:201-261) in one engine call, nothing leaves the device
        last["out"] = m.step(xs[i % 4], anchors_dev, window_dev, tsz_dev, PENALTY_K, WINDOW_INFLUENCE, refine=sharp,
                             mask_head=sharp and mask_head)
        return last["out"]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1), device=dev)

    sampler = ClockSampler("GPU-" + str(torch.cuda.get_device_properties(dev).uuid)) if rank == 0 else None
    warm = max(args.warmup, 3)
    for i in range(warm):
        step(i)
    est_ms = timed(step, 3) / 3           # sizes the e2e region below
    l0 = m.launch_count
    t_start = time.perf_counter()
    ms = timed(step, args.steps)
    t_end = time.perf_counter()
    launches = m.launch_count - l0
    clocks = sampler.stop(t_start, t_end) if sampler else None
    if args.dump_outputs and rank == 0:   # before any later call overwrites the engine's output buffers
        dump_step_outputs(args.dump_outputs, last["out"])
    fps = world * B * args.steps / (ms * 1e-3)
    fps_skip = None
    if sharp:
        n_skip = max(3, args.steps // 4)
        ms_skip = timed(lambda i: step(i, mask_head=False), n_skip)
        fps_skip = world * B * n_skip / (ms_skip * 1e-3)

    # ---- parity of THIS run's outputs against the CPU oracle (first and last stream of this rank)
    parity = None
    if args.verify:
        parity = verify_against_oracle(args, m, sd, z, xs[1], anchors_dev, window_dev, tsz_dev, B, dev, sharp)
        if world > 1:
            t = torch.tensor([parity["max_rel"]], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            worst = float(t.item())
            t2 = torch.tensor([1.0 if parity["argmax_equal"] else 0.0], device=dev)
            dist.all_reduce(t2, op=dist.ReduceOp.MIN)
            parity = dict(parity, max_rel_all_ranks=worst, argmax_equal_all_ranks=bool(t2.item() > 0.5), ranks=world)

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D of x + target sizes, the same frame, D2H
    lib = _lib.load()
    xh = [torch.empty(B, 3, S, S).pin_memory() for _ in range(2)]
    for t_ in xh:
        t_.copy_(xs[0].cpu())
    tszh = tsz_dev.cpu().contiguous().pin_memory()
    rech = [torch.empty(B, 8).pin_memory() for _ in range(2)]
    refh = [torch.empty(B, 127 * 127).pin_memory() for _ in range(2)] if sharp else [None, None]
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    ios = {}

    def make_io(g, mask_head):
        io = _lib.SmStepIO()
        io.x_host = xh[g].data_ptr(); io.tsz_host = tszh.data_ptr()
        io.anchors_dev = anchors_dev.data_ptr(); io.window_dev = window_dev.data_ptr()
        io.penalty_k = PENALTY_K; io.window_influence = WINDOW_INFLUENCE
        io.flags = ((_lib.SM_TRACK_MASK_FEATURES if sharp else 0) |
                    (_lib.SM_TRACK_MASK_HEAD if (sharp and mask_head) else 0))
        io.records_host = rech[g].data_ptr()
        io.refine_host = refh[g].data_ptr() if sharp else None
        return io

    def submit(g, mask_head):
        io = ios.setdefault((g, mask_head), make_io(g, mask_head))
        tk = C.c_int32()
        _lib.check(lib.sm_step_host_async(m.handle, g * B, B, C.byref(io), stream, C.byref(tk)))
        return tk.value

    def host_loop(n, mask_head, groups=2):
        # two independent groups of B tracker streams alternate: while group 0's frame is on the GPU the host
        # collects group 1's results and submits its next frame (a group's frame k+1 is only submitted after its
        # frame k has been waited for — the dependency a real tracker has).  groups=1: strictly serial.
        pending = [None, None]
        for i in range(n):
            g = i % groups
            if pending[g] is not None:
                _lib.check(lib.sm_track_host_wait(m.handle, pending[g]))
            pending[g] = submit(g, mask_head)
        for g in range(groups):
            if pending[g] is not None:
                _lib.check(lib.sm_track_host_wait(m.handle, pending[g]))

    def e2e_rate(mask_head, groups, n):
        host_loop(3, mask_head, groups)
        barrier()
        t0 = time.perf_counter()
        host_loop(n, mask_head, groups)      # every step's results are in host memory when this returns
        dt = max_over_ranks(time.perf_counter() - t0, device=dev)
        return world * B * n / dt, dt
    n_e2e = max(args.steps, math.ceil(args.min_seconds * 1e3 / est_ms))
    e2e_fps, e2e_dt = e2e_rate(True, 2, n_e2e)
    e2e_skip = e2e_rate(False, 2, max(3, n_e2e // 4))[0] if sharp else None
    e2e_serial = e2e_rate(True, 1, max(3, n_e2e // 4))[0]
    h2d = xh[0].numel() * 4 + tszh.numel() * 8
    d2h = rech[0].numel() * 4 + (refh[0].numel() * 4 if sharp else 0)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-launch CUDA-event timing of every kernel (same workload, separate pass)
    peaks = load_peaks()
    m.profile(True)
    nprof = 3
    for i in range(nprof):
        step(i)
    rows = m.profile_dump()
    m.profile(False)
    cats = {}
    for name, cat, t, fl, by in rows:
        c = cats.setdefault(cat, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
        c["ms"] += t / nprof; c["flops"] += fl / nprof; c["bytes"] += by / nprof; c["launches"] += 1 / nprof
    gemm = cats.get("conv_gemm", {"ms": 1e-9, "flops": 0.0, "bytes": 0.0, "launches": 0})
    tot_ms = sum(c["ms"] for c in cats.values())
    achieved = gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12
    layers = {}
    for name, cat, t, fl, by in rows:
        if cat == "conv_gemm":
            L = layers.setdefault(name, [0.0, 0.0])
            L[0] += t / nprof; L[1] += fl / nprof
    top = sorted(layers.items(), key=lambda kv: -kv[1][0])[:6]
    if args.dump_layers:
        with open(args.dump_layers, "w") as f:
            f.write("name\tcat\tms\tgflop\tMB\tTFLOPs\tGBps\n")
            for name, cat, t, fl, by in rows[:len(rows) // nprof]:
                f.write(f"{name}\t{cat}\t{t:.4f}\t{fl / 1e9:.2f}\t{by / 1e6:.1f}\t{fl / (t * 1e-3) / 1e12:.1f}\t"
                        f"{by / (t * 1e-3) / 1e9:.0f}\n")
    traffic = None
    tpath = os.path.join(ROOT, "profiles", args.traffic_file)
    if os.path.exists(tpath) and args.precision == "exact" and B == 64 and S == 255 and sharp:
        tj = json.load(open(tpath))           # ncu dram__bytes_read+write of the family's launches in one step
        traffic = {"bytes_per_step": tj["conv_gemm_traffic_bytes_per_step"],
                   "launches_per_step": tj["conv_gemm_launches_per_step"], "measured_in_run": False,
                   "source": f"profiles/{args.traffic_file} (committed ncu capture of this command, not measured in this run)"}
    roofline = {
        "bound": "tensor", "kernel": "conv_gemm_kernel (tcgen05 implicit-GEMM conv family, all layers of one step)",
        "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
        "peak_source": peaks["src"] + ", sustained cuBLAS bf16", "traffic": traffic,
        "algorithmic_bytes_per_step": gemm["bytes"],
        # the parity mode issues 3 fp16 MMAs per algorithmic MAC: tensor-pipe work actually executed vs the same peak
        "mma_issued_frac": (3.0 if args.precision == "exact" else 1.0) * achieved / peaks["tflops"],
        "launches_per_step": gemm["launches"], "ms_per_step": gemm["ms"], "share_of_step": gemm["ms"] / tot_ms,
        "algorithmic_gflop_per_step": gemm["flops"] / 1e9,
        "note": "algorithmic FLOPs (2*M*N*K per conv, no padding, no x3 for the split-fp16 passes) / summed "
                "CUDA-event durations of the launches (one launch per layer over the whole batch, lanes off)",
        "top_layers": [{"layer": k, "ms": v[0], "tflops": v[1] / (v[0] * 1e-3) / 1e12} for k, v in top],
    }
    by_cat = {k: {"ms": round(v["ms"], 4), "launches": round(v["launches"], 1),
                  "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2) if v["ms"] > 0 else 0.0,
                  "gbps": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["ms"] > 0 else 0.0}
              for k, v in sorted(cats.items(), key=lambda kv: -kv[1]["ms"])}

    # ---- standalone depthwise xcorr operator (the "xcorr GB/s" half of the metric): branches x streams planes
    nbr = 3 if sharp else 2
    planes_b = nbr * B
    xc = torch.randn(planes_b, 256, R + 4, R + 4, device=dev)
    kc = torch.randn(planes_b, 256, 5, 5, device=dev)
    for _ in range(3):
        smb.conv2d_dw_group(xc, kc)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    reps = 20
    e0.record()
    for _ in range(reps):
        out = smb.conv2d_dw_group(xc, kc)
    e1.record()
    torch.cuda.synchronize()
    xms = e0.elapsed_time(e1) / reps
    xbytes = planes_b * XCORR_BYTES.get(S, (256 * ((R + 4) ** 2 + 25 + R * R)) * 4)
    xgbs = xbytes / (xms * 1e-3) / 1e9
    del xc, kc, out

    gfl = (GFLOP_SHARP if sharp else GFLOP_RPN).get(S, 0.0)
    result = {
        "metric": metric_name(args), "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f16x3 (hi+lo split fp16 operands on tcgen05, f32 accumulate; f32 CUDA-core stem/xcorr/refine)"
                 if args.precision == "exact" else "f16 (single-pass tcgen05, f32 accumulate)",
        "data": "synthetic", "config": workload_config(args, B, world),
        "precision_mode": args.precision,
        "timed_region_s": ms * 1e-3,
        "algorithmic_tflops": fps * gfl / 1e3,
        "value_skip_dead_mask_head": fps_skip,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "timed_region_s": e2e_dt, "value_skip_dead_mask_head": e2e_skip, "value_serial_one_group": e2e_serial,
                "api": "sm_step_host_async / sm_track_host_wait (C ABI, pinned host buffers): H2D frames + target "
                       "sizes -> track_mask incl. mask head -> on-device selection -> refine at the selected position "
                       "-> D2H records + refine logits; same flags as `value`; two independent groups of "
                       "batch_per_gpu streams alternate (one step in flight), value_serial_one_group = no overlap"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": roofline,
        "kernels_ms_per_step": by_cat,
        "xcorr": {"op": "sm_xcorr_depthwise fp32 NCHW", "planes": planes_b * 256, "ms": xms, "GBps": xgbs,
                  "peak": peaks["hbm_gbs"], "frac": xgbs / peaks["hbm_gbs"], "peak_source": peaks["src"]},
        "parity_check": parity,
        "device_bytes": m.device_bytes,
    }
    if world == 1 and sharp and S == 255 and not args.no_loop:
        result["loop"] = tracker_loop_rate(args, m, B, dev)
    if world == 1 and not args.no_cpu:
        cfps, cores, sample, _ = run_cpu_fleet(args, seconds=args.cpu_seconds)
        result["cpu_baseline"] = {"value": cfps, "unit": "frames/s", "cores": cores, "host_cpus": os.cpu_count(),
                                  "kind": "port", "sample": sample}
    if world == 1 and not args.no_context:
        del m
        torch.cuda.empty_cache()
        result["context"] = {"cudnn": cudnn_context(args, dev)}
    print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


DUMP_ARRAY_BYTES = 8 << 20      # per array: Custom.step returns at most 7, so a dump stays under 64 MB


def dump_step_outputs(path, out):
    """Writes one step's outputs (the dict `Custom.step` returns) as path/<name>.npy: integer outputs as float64 (exact),
    the rest as float32.  An array larger than DUMP_ARRAY_BYTES (the raw mask head: 635 MB at B=64) is written as
    <name>_sample.npy, its elements at flat indices drawn from a generator seeded with 0: the same in every run."""
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in out.items():
        if t is None:
            continue
        t = t.float() if t.is_floating_point() else t.double()
        cap = DUMP_ARRAY_BYTES // t.element_size()
        if t.numel() > cap:
            idx = torch.randint(t.numel(), (cap,), generator=torch.Generator().manual_seed(0)).to(t.device)
            name, t = name + "_sample", t.flatten()[idx]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def tracker_loop_rate(args, m, B, dev, seconds=1.5):
    """The whole tracker loop of tools/test.py:172-315 for B concurrent streams with device-resident state
    (siammask_b200.tracker.BatchTracker): uint8 frames in HBM -> search-window arithmetic -> cv2-exact crop + resize ->
    track_mask + selection + refine -> state update -> mask paste-back + threshold.  Frames: synthetic 480x640 BGR,
    one per stream, already on the device (a video decoder's output)."""
    import torch
    from siammask_b200.tracker import BatchTracker, TrackerParams
    H, W = 480, 640
    g = torch.Generator(device=dev).manual_seed(7)
    frames = [(torch.rand(B, H, W, 3, device=dev, generator=g) * 255).to(torch.uint8) for _ in range(2)]
    boxes = np.tile(np.array([[280.0, 200.0, 80.0, 60.0]]), (B, 1)) + np.random.RandomState(0).rand(B, 4) * 20
    bt = BatchTracker(m, TrackerParams(instance_size=args.search), slot0=0)
    bt.init(frames[0], boxes)
    for i in range(3):
        bt.track(frames[i % 2])
    torch.cuda.synchronize(dev)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        r = bt.track(frames[n % 2])
        n += 1
        if n % 4 == 0:
            r.state[0, 0].item()                 # the host looks at results now and then (bounded queue depth)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    return {"value": B * n / dt, "unit": "frames/s", "frames": n * B, "seconds": dt, "frame_hw": [H, W],
            "what": "BatchTracker.track(mask=True, refine=True): sm_tracker_prepare + sm_crop_resize + sm_step + "
                    "sm_tracker_update + sm_warp_affine + threshold, uint8 frames resident in HBM, masks left on the device"}


def verify_against_oracle(args, m, sd, z, x, anchors_dev, window_dev, tsz_dev, B, dev, sharp):
    """Outputs of one engine step at THIS run's batch / tile / lane configuration vs the CPU oracle, for the first
    and the last stream of this rank (max|a-b| / max|b| per tensor, the parity metric of tests/conftest.py)."""
    import torch
    from oracle.siammask_oracle import Oracle
    out = m.step(x, anchors_dev, window_dev, tsz_dev, PENALTY_K, WINDOW_INFLUENCE, refine=sharp, mask_head=sharp,
                 mask_col=sharp)
    torch.cuda.synchronize(dev)
    streams = sorted({0, B - 1})
    o = Oracle(sd)
    torch.set_num_threads(min(16, os.cpu_count() or 1))
    errs, same = {}, True

    def rel(a, b):
        a, b = a.detach().double().cpu(), b.detach().double().cpu()
        return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    for b in streams:
        o.template(z[b:b + 1].cpu())
        if sharp:
            ocls, oloc, omask = o.track_mask(x[b:b + 1].cpu())
        else:
            ocls, oloc = o.track(x[b:b + 1].cpu())
        errs["cls"] = max(errs.get("cls", 0.0), rel(out["cls"][b:b + 1], ocls))
        errs["loc"] = max(errs.get("loc", 0.0), rel(out["loc"][b:b + 1], oloc))
        # the selection of the engine vs the reference arithmetic (numpy, float64) on the ORACLE's cls/loc
        from oracle.ref_loop import select_numpy
        from siammask_b200 import anchors as anc
        R = (args.search - 127) // 8 + 9
        with np.errstate(all="ignore"):      # random-init weights: exp() of a large loc output may overflow, as in numpy
            bid, box, score, pen, ps = select_numpy(    ocls, oloc, anc.generate_anchor({"stride": 8, "ratios": [0.33, 0.5, 1, 2, 3], "scales": [8], "round_dight": 0}, R),
                anc.cosine_window(R, 5), tsz_dev[b].cpu().numpy(), PENALTY_K, WINDOW_INFLUENCE)
        same = same and int(out["best"][b]) == bid
        if sharp:
            pos = tuple(int(v) for v in out["pos"][b].cpu())
            errs["refine"] = max(errs.get("refine", 0.0), rel(out["refine"][b:b + 1], o.track_refine(pos)))
            errs["mask_col"] = max(errs.get("mask_col", 0.0), rel(out["mask_col"][b], omask[0, :, pos[0], pos[1]]))
    return {"max_rel": max(errs.values()), "per_tensor": errs, "argmax_equal": same, "streams": streams,
            "tolerance": 1e-3, "ok": max(errs.values()) <= 1e-3, "oracle": "oracle/siammask_oracle.py (torch CPU fp32)"}


PRESETS = {2: dict(batch=64, search=255, rpn_only=False),     # BASELINE.json configs[1] (and configs[3] at N=8)
           3: dict(batch=256, search=255, rpn_only=True),     # configs[2]
           4: dict(batch=64, search=255, rpn_only=False),     # configs[3]: 512 streams over 8 GPUs = 64 per GPU
           5: dict(batch=128, search=383, rpn_only=False)}    # configs[4]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "_cpu_worker"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(PRESETS),
                    help="BASELINE.json config number (1-based): 2 = B=64 sharp (default), 3 = SiamRPN-only B=256, "
                         "4 = 512 streams on 8 GPUs, 5 = search 383 B=128")
    ap.add_argument("--batch", type=int, default=None, help="paired tracker streams per GPU (overrides the preset)")
    ap.add_argument("--search", type=int, default=None)
    ap.add_argument("--precision", default="exact", choices=["exact", "fast"])
    ap.add_argument("--rpn-only", action="store_true", default=None,
                    help="SiamRPN-only engine (experiments/siamrpn_resnet): step = track -> cls/loc")
    ap.add_argument("--min-seconds", type=float, default=2.0, help="minimum length of the e2e timed region")
    ap.add_argument("--ref-batch", type=int, default=2, help="frames per step of each CPU reference worker")
    ap.add_argument("--cpu-threads", type=int, default=0, help="torch threads per CPU worker (0 = pick)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="length of the cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-context", action="store_true", help="skip the PyTorch/cuDNN context leg")
    ap.add_argument("--no-loop", action="store_true", help="skip the whole-tracker-loop leg")
    ap.add_argument("--no-verify", dest="verify", action="store_false", help="skip the oracle parity check")
    ap.add_argument("--traffic-file", default="r02_traffic.json")
    ap.add_argument("--dump-layers", default=None, help="write the per-launch CUDA-event table of one step here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (same arguments, same inputs)")
    # internal (cpu worker processes)
    ap.add_argument("--threads", type=int, default=8)
    ap.add_argument("--worker-id", type=int, default=0)
    ap.add_argument("--worker-seconds", type=float, default=0.0)
    args = ap.parse_args()
    if args.steps < 1 and args.impl != "_cpu_worker":     # a CPU worker gets --steps 0 when it runs for --worker-seconds
        ap.error("--steps must be at least 1")
    preset = PRESETS[args.config]
    if args.batch is None:
        args.batch = preset["batch"]
    if args.search is None:
        args.search = preset["search"]
    if args.rpn_only is None:
        args.rpn_only = preset["rpn_only"]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "_cpu_worker":
        _cpu_worker(args)
    elif args.impl == "reference":
        run_reference(args, rank)
    else:
        run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
