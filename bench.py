#!/usr/bin/env python
"""bench.py -- profiled trajectories/s of the batched spline -> motion-profile engine on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config cfg2|cfg3] [--dump-outputs DIR]

A "step" is one pass of the whole hot path (build_path -> tables -> distance sampling -> forward/backward ->
time-domain resampling) over one batch of synthetic random-node paths.

--config cfg2 (default; BASELINE.json configs[1], the configuration the metric is quoted on): 4096 random 8-node paths,
  factory constraints.  At N > 1 every rank profiles its own 4096-path batch (weak scaling, no data-path collective; the
  only exchange is the NCCL all_gather of the 40-byte per-path summary rows, preallocated and on a side stream).
  Consecutive steps are INDEPENDENT batches, so they are software-pipelined two deep on the device (two CUDA graphs on two
  streams: the latency-bound tail of step n overlaps the bandwidth-bound front of step n+1); every step still launches
  every kernel.  `ms_per_step_serial` in `config` is the unpipelined latency of one step.
--config cfg3 (BASELINE.json configs[2]): ONE job of 2**20 random 16-node paths (seed 1), sharded over the ranks in
  contiguous work-balanced shards (strong scaling), processed in tiles that fit HBM; value = paths of the whole job / time.

`--impl reference` times the CPU restatement of the reference (oracle/, a C port with OpenMP) on all host cores over a
bounded sample of the same workload; the unmodified Python reference itself (baseline/_ref, staged by
baseline/make_ref.py) is timed next to it as cpu_baseline.reference_python when it travelled with the snapshot.
Rank 0 prints ONE JSON line.

--dump-outputs DIR: after the timed steps rank 0 writes what the last timed step returned as DIR/<name>.npy (float64, at
  most 64 MB in all), so that two builds can be compared output for output on the same seeded inputs.  cfg2 (and
  --profile-step): `summary` [B, 5] (n_out, total length, t_end, max|v|, status) and `n_samples` [B] of every path, and for
  a fixed, seeded sample of paths (`paths`, ascending) their `nodes_map` / `actions_map` rows (-1 padded) and each output
  stream (times, positions, linear_vels, accelerations, headings, angular_vels, x, y, and the pass velocities `vel`) with
  the sampled paths' rows cut at n_out (vel: n_samples) and concatenated in `paths` order.  cfg3 and --impl reference:
  the `summary` rows the job returns.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

UNIT = "trajectories/s"
FACTORY_CONS = dict(max_vel=4.0, max_acc=8.0, max_dec=8.0, friction_coef=0.8, max_jerk=16.0, track_width=12.5 / 12)
DUMP_BYTES = 64 << 20


def metric_name(nodes: int) -> str:
    return f"profiled trajectories/sec ({nodes}-node paths)"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ --dump-outputs
def write_dump(dirname, arrays):
    """Every array as DIR/<name>.npy in float64; more than DUMP_BYTES in all is an error."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed {DUMP_BYTES}")
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, f"{k}.npy"), a)


def summary_dump(rows, seed=0):
    """The summary rows of a job; a job too large for DUMP_BYTES keeps a fixed, seeded sample of its rows (`paths`)."""
    rows = np.asarray(rows)
    cap = DUMP_BYTES // (8 * (rows.shape[1] + 1))
    if len(rows) <= cap:
        return {"summary": rows}
    paths = np.sort(np.random.default_rng(seed).choice(len(rows), cap, replace=False))
    return {"summary": rows[paths], "paths": paths}


def profile_dump(res, max_paths=256, seed=0):
    """A ProfileResult as the arrays of --dump-outputs (module docstring).  The seeded sample is the first `max_paths` of
    a fixed permutation of the batch, halved (the same permutation's shorter prefix) until the arrays fit DUMP_BYTES."""
    import torch
    from vexautonomousplanner_b200.engine import OUT_NAMES
    summary = res.summary.cpu().numpy()
    n_out = res.n_out.cpu().numpy().astype(np.int64)
    n_samples = res.n_samples.cpu().numpy().astype(np.int64)
    n_maps = res.n_maps.cpu().numpy()
    order = np.random.default_rng(seed).permutation(res.B)
    width = res.nodes_map.shape[1] + res.actions_map.shape[1]

    def nbytes(p):
        return 8 * (summary.size + res.B + len(p) * (1 + width) + len(OUT_NAMES) * n_out[p].sum() + n_samples[p].sum())

    k = min(res.B, max_paths)
    while k > 1 and nbytes(order[:k]) > DUMP_BYTES:
        k //= 2
    paths = np.sort(order[:k])
    idx = torch.as_tensor(paths, device=res.out.device)
    out = res.out[:, idx, :int(n_out[paths].max())].cpu().numpy()
    vel = res.vel[idx, :int(n_samples[paths].max())].cpu().numpy()
    dump = {"summary": summary, "n_samples": n_samples, "paths": paths}
    for name, maps, lens in (("nodes_map", res.nodes_map, n_maps[paths, 0]), ("actions_map", res.actions_map, n_maps[paths, 1])):
        m = maps[idx].cpu().numpy().astype(np.int64)
        m[np.arange(m.shape[1])[None, :] >= lens[:, None]] = -1
        dump[name] = m
    for i, name in enumerate(OUT_NAMES):
        dump[name] = np.concatenate([out[i, j, :n_out[p]] for j, p in enumerate(paths)])
    dump["vel"] = np.concatenate([vel[j, :n_samples[p]] for j, p in enumerate(paths)])
    return dump


# ------------------------------------------------------------------------------------------------ CPU baselines
def cpu_port_rate(packed, seconds: float, threads: int):
    """Time the C oracle (OpenMP over paths) on a bounded sample; returns (paths/s, sample description, elapsed)."""
    import oracle
    oracle.build()
    oracle.set_sq_mode(0)
    n0 = min(packed.B, max(2 * threads, 16))
    t = time.perf_counter()
    oracle.full_batch(packed.node_attr[:n0], packed.node_flags[:n0], packed.cons[:n0], threads=threads)
    r0 = n0 / (time.perf_counter() - t)
    n = int(min(packed.B, max(n0, r0 * seconds)))
    reps = max(1, int(round(r0 * seconds / n)))          # bounded sample: about `seconds` of CPU work
    t = time.perf_counter()
    for _ in range(reps):
        s = oracle.full_batch(packed.node_attr[:n], packed.node_flags[:n], packed.cons[:n], threads=threads)
    el = time.perf_counter() - t
    assert (s[:, 4] == 0).all()
    return n * reps / el, f"{reps} x the first {n}", el


PYREF_DIR = os.path.join(ROOT, "baseline", "_ref", "src")


def _pyref_init(ref_src):
    """Worker initialiser: import the UNMODIFIED reference (baseline/_ref/src) headless.  splines.spline_manager needs
    gui.node.Node / gui.action_point.ActionPoint as annotations only (spline_manager.py:8-9): attribute-only stand-ins."""
    import logging
    import types
    import warnings
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    gui = types.ModuleType("gui"); gui.__path__ = []
    node_mod, ap_mod = types.ModuleType("gui.node"), types.ModuleType("gui.action_point")

    class Node:
        def __init__(self):
            self.is_reverse_node = False; self.turn = 0; self.wait_time = 0; self.stop = False; self.tangent = None
            self.incoming_magnitude = None; self.outgoing_magnitude = None; self.max_velocity = 0; self.max_acceleration = 0

    class ActionPoint:
        def __init__(self, t):
            self.t = t; self.stop = False; self.wait_time = 0; self.max_velocity = 0; self.max_acceleration = 0

    node_mod.Node, ap_mod.ActionPoint = Node, ActionPoint
    sys.modules.update({"gui": gui, "gui.node": node_mod, "gui.action_point": ap_mod})
    sys.path.insert(0, ref_src)
    logging.disable(logging.CRITICAL)
    warnings.filterwarnings("ignore")
    global _REF
    from splines.spline_manager import QuinticHermiteSplineManager
    import motion_profiling_v2.motion_profile_generator as mpg
    _REF = (QuinticHermiteSplineManager, mpg, Node)


def _pyref_one(pts_ft):
    """build_path + generate_motion_profile (which calls rebuild_tables, motion_profile_generator.py:402) for one path."""
    Manager, mpg, Node = _REF
    sm = Manager()
    nodes = [Node() for _ in range(len(pts_ft))]
    assert sm.build_path(np.asarray(pts_ft, dtype=float), nodes, [])
    out = mpg.generate_motion_profile(sm, mpg.Constraints(**FACTORY_CONS))
    return len(out[0])


def python_reference_rate(packed, n_paths: int, procs: int):
    """The unmodified Python reference on the host cores (multiprocessing, one worker per core); None if it did not travel."""
    if not os.path.isdir(os.path.join(PYREF_DIR, "splines")):
        return None
    import multiprocessing as mp
    n = min(packed.B, max(n_paths, procs))
    pts = [packed.node_attr[b, : int(packed.n_nodes[b]), 0:2].copy() for b in range(n)]
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs, initializer=_pyref_init, initargs=(PYREF_DIR,)) as pool:
        pool.map(_pyref_one, pts[:procs])                       # imports + first-call costs outside the timed region
        t = time.perf_counter()
        T = pool.map(_pyref_one, pts, chunksize=1)
        el = time.perf_counter() - t
    return {"value": n / el, "unit": UNIT, "cores": procs, "kind": "reference",
            "sample": f"{n} paths, {el:.1f} s wall, unmodified src/splines + src/motion_profiling_v2 (baseline/_ref), "
                      "build_path + generate_motion_profile incl. rebuild_tables, multiprocessing one worker per core",
            "per_core": n / el / procs, "mean_T": float(np.mean(T))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from vexautonomousplanner_b200 import synth
    threads = os.cpu_count() or 1
    B, N, seed, label = workload(args)
    packed = synth.random_paths(min(B, 4096), N, seed=seed)
    import oracle
    oracle.build()
    sample = min(packed.B, args.ref_sample if N <= 8 else args.ref_sample // 4)
    sub = packed.slice(0, sample)
    for _ in range(args.warmup):
        oracle.full_batch(sub.node_attr, sub.node_flags, sub.cons, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s = oracle.full_batch(sub.node_attr, sub.node_flags, sub.cons, threads=threads)
    el = time.perf_counter() - t0
    if args.dump_outputs:
        write_dump(args.dump_outputs, summary_dump(s))
    value = sample * args.steps / el
    pyref = None if args.no_pyref else python_reference_rate(packed, 2 * threads, threads)
    line = {
        "impl": "reference", "metric": metric_name(N), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.config == "cfg3" else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": label, "paths_per_gpu": B, "nodes": N, "sample": f"first {sample} paths per step"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} paths x {args.steps} steps, C restatement of the reference (oracle/), OpenMP",
                         "reference_python": pyref},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload(args):
    if args.config == "cfg3":
        B = args.paths or (1 << 20)
        N = args.nodes or 16
        return B, N, 1, (f"{B} random {N}-node paths (seed 1) as ONE job sharded over the ranks, factory constraints, "
                         "dt=0.01 dd=0.005 (BASELINE.json configs[2])")
    B = args.paths or 4096
    N = args.nodes or 8
    return B, N, 0, (f"{B} random {N}-node paths per GPU, factory constraints, dt=0.01 dd=0.005 (BASELINE.json configs[1])")


# ------------------------------------------------------------------------------------------------ helpers (GPU arm)
def set_local_affinity(local_rank: int):
    """Pin this rank (and therefore its pinned-buffer allocations) to the CPUs NVML reports as local to its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        cpus = [c for c in cpus if c < (os.cpu_count() or 1)]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"cpus": len(cpus), "first": cpus[0] if cpus else None, "last": cpus[-1] if cpus else None}
    except Exception as e:                                   # noqa: BLE001
        return {"error": str(e)[:80]}


def d2h_microbench(torch, dev, dist, world, mb: int = 512, reps: int = 6):
    """What the host can sink: every rank copies `mb` MB device -> pinned host `reps` times at the same moment."""
    src = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
    dst = torch.empty(mb << 20, dtype=torch.uint8, pin_memory=True)
    dst.copy_(src); torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    e.record(); torch.cuda.synchronize()
    gbs = reps * (mb << 20) / 1e9 / (s.elapsed_time(e) * 1e-3)
    t = torch.tensor([gbs, gbs], dtype=torch.float64, device=dev)
    if world > 1:
        tmin = t.clone()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        return {"per_rank_min_GBps": float(tmin[0].item()), "aggregate_GBps": float(t[0].item())}
    return {"per_rank_min_GBps": gbs, "aggregate_GBps": gbs}


def dfma_peak(torch, eng):
    import ctypes as C
    out = torch.zeros(1, dtype=torch.float64, device=eng.device)
    ctas, iters = 148 * 8, 1 << 14
    best = 0.0
    for _ in range(4):
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record()
        eng.lib.vap_bench_dfma(C.c_int64(ctas), C.c_int64(iters), C.c_void_p(out.data_ptr()), eng._stream())
        e.record(); torch.cuda.synchronize()
        best = max(best, ctas * 256 * iters * 16 / (s.elapsed_time(e) * 1e-3) / 1e12)
    return best


def load_kernel_table(B, N):
    """ncu per-kernel table of the same workload, regenerated by profiles/tools/ktable_json.py from a capture of the
    committed code (the JSON names the commit)."""
    for name in ("profiles/r02_kernel_table.json", "profiles/r01b_kernel_table.json"):
        try:
            with open(os.path.join(ROOT, name)) as f:
                prof = json.load(f)
            if (B, N) == (4096, 8):
                return prof, name
        except Exception:
            continue
    return None, None


def stage_table(torch, eng, db, flush, steps, N):
    """Per-stage device times of an eager (unpipelined, ungraphed) step: CUDA events on the launch stream, median."""
    eng.profile(db, reuse_plan=True)
    torch.cuda.synchronize()
    per_step = []
    for _ in range(max(steps, 3)):
        flush.zero_()
        eng.stage_events = []
        res = eng.profile(db, reuse_plan=True)
        torch.cuda.synchronize()
        acc = {}
        for name, s, e in eng.stage_events:
            acc[name] = acc.get(name, 0.0) + s.elapsed_time(e)
        per_step.append(acc)
    eng.stage_events = None
    stage_ms = {k: float(np.median([a[k] for a in per_step])) for k in per_step[0]}
    B = db.B
    Dsum = float(res.n_samples.double().sum().item())
    Tsum = float(res.n_out.double().sum().item())
    Q, P = 1000.0 * B, 1000.0 * N * B            # random paths have one spline each
    # algorithmic bytes per stage (SURVEY.md 8d): 8 B per fp64 element, each array once per stage that must touch it
    stage_bytes = {"S0_build_path": 8 * (2 * N + 9 * N) * B, "S1_lut": 8 * 2 * Q, "S2_props": 8 * 2 * P,
                   "S3_dist_sample": 8 * 5 * Dsum, "S45_fwd_bwd": 8 * 4 * Dsum, "S345_velocity": 8 * 9 * Dsum, "S6_resample": 8 * (Dsum + 9 * Tsum)}
    return stage_ms, stage_bytes, Dsum, Tsum, res


# ------------------------------------------------------------------------------------------------ cfg2 (default)
def run_cfg2(args):
    import torch
    import torch.distributed as dist

    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import Engine, PipelinedProfiler
    from vexautonomousplanner_b200.sharding import SummaryGatherer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    affinity = set_local_affinity(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, N, _, label = workload(args)
    packed = synth.random_paths(B, N, seed=rank)      # weak scaling: every rank its own cfg2 batch
    eng = Engine(dev, chunks=args.chunks)
    db = eng.upload(packed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    # what a caller pays ONCE per batch shape and every timed step below does not: the first call sizes D_cap / T_cap from
    # the data (two read-backs), builds the path-independent tables and grows the allocator's pools
    torch.cuda.synchronize()
    t_first = time.perf_counter()
    eng.profile(db, reuse_plan=True)
    torch.cuda.synchronize()
    first_call_ms = (time.perf_counter() - t_first) * 1e3
    t_second = time.perf_counter()
    eng.profile(db, reuse_plan=True)
    torch.cuda.synchronize()
    second_call_ms = (time.perf_counter() - t_second) * 1e3
    if args.profile_step:
        # what profiles/tools/capture.sh runs under ncu: the same step, eager and unpipelined (every kernel one launch)
        for _ in range(max(args.warmup, 1)):
            eng.profile(db, reuse_plan=True)
        torch.cuda.synchronize()
        l0 = eng.launches
        for _ in range(args.steps):
            flush.zero_()
            res = eng.profile(db, reuse_plan=True)
        torch.cuda.synchronize()
        if args.dump_outputs and rank == 0:
            write_dump(args.dump_outputs, profile_dump(res))
        print(json.dumps({"profile_step": True, "steps": args.steps, "launches_per_step": (eng.launches - l0) // args.steps}))
        return
    depth = max(1, args.pipeline)
    pipe = PipelinedProfiler(eng, db, depth=depth)
    gatherer = SummaryGatherer([B] * world, dev)
    main = torch.cuda.current_stream(dev)

    def consume(res):
        gatherer.submit(res.summary)                  # snapshot + all_gather on a side stream: nobody waits for it

    def run_steps(K):
        """K steps enqueued back to back; returns the events around the whole region (on the caller's stream) and the
        result of the last step."""
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(main)
        for k in range(K):
            with torch.cuda.stream(pipe.streams[pipe.n % depth]):
                pipe.streams[pipe.n % depth].wait_stream(main)
                flush.zero_()                         # L2 flushed before every step (on the step's own stream)
            last = pipe.submit(None, consume)
        pipe.drain()
        gatherer.wait()
        e.record(main)
        return s, e, last

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    run_steps(max(args.warmup, 3))
    barrier()
    # ---------------- timed region: K steps, device time, max over ranks
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = eng.launches
    barrier()
    wall0 = time.perf_counter()
    s, e, last = run_steps(args.steps)
    barrier()
    wall = time.perf_counter() - wall0
    launches = (eng.launches - l0) // args.steps
    dev_ms = s.elapsed_time(e)
    clocks = sampler.stop() if sampler else None
    tt = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_per_step = float(tt.item()) / args.steps
    value = world * B / (ms_per_step * 1e-3)
    res = pipe.graphs[0].res
    assert bool((res.status == 0).all().item())
    allrows = gatherer.rows()
    assert allrows.shape == (world * B, 5) and bool((allrows[:, 4] == 0).all().item())
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, profile_dump(last))      # before the replays below overwrite the graphs' outputs

    # ---------------- unpipelined latency of one step (one graph replay at a time, per-step events)
    lat = []
    for _ in range(max(3, min(args.steps, 10))):
        flush.zero_()
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); pipe.graphs[0].graph.replay(); b.record()
        torch.cuda.synchronize()
        lat.append(a.elapsed_time(b))
    serial_ms = float(np.median(lat))

    # ---------------- per-stage device times + roofline
    stage_ms, stage_bytes, Dsum, Tsum, _ = stage_table(torch, eng, db, flush, args.steps, N)
    peak, peak_src = measured_peak()
    stages = {k: {"ms": round(v, 4), "alg_GB": round(stage_bytes[k] / 1e9, 4),
                  "GBps": round(stage_bytes[k] / 1e9 / (v * 1e-3), 1)} for k, v in stage_ms.items()}
    dom = max(stage_ms, key=stage_ms.get)
    achieved = stage_bytes[dom] / 1e9 / (stage_ms[dom] * 1e-3)
    total_bytes = sum(stage_bytes[k] for k in stage_ms)          # only the stages that ran (fused or staged velocity stage)
    prof, prof_name = load_kernel_table(B, N)
    traffic, ncu_kernels, prof_commit = None, None, None
    if prof is not None:
        try:
            traffic = prof["stages"][dom]["dram_bytes_per_step"]
            prof_commit = prof.get("commit")
            ncu_kernels = {k: {"ms": v["ms"], "dram_GBps": v["dram_GBps"], "dram_frac_of_peak": round(v["dram_GBps"] / peak, 3),
                               "fp64_pipe_pct": v["fp64_pipe_pct"]} for k, v in prof["kernels"].items() if v["ms"] >= 0.05}
        except Exception:
            traffic = None
    fp64_tflops = dfma_peak(torch, eng)
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "traffic_source": (f"{prof_name} (ncu dram__bytes_read+write summed over the stage's kernels; capture of commit "
                                   f"{prof_commit})" if prof_name else None),
                "whole_step": {"alg_GB": total_bytes / 1e9, "GBps": total_bytes / 1e9 / (ms_per_step * 1e-3),
                               "frac": total_bytes / 1e9 / (ms_per_step * 1e-3) / peak,
                               "frac_unpipelined": total_bytes / 1e9 / (serial_ms * 1e-3) / peak},
                "stages": stages, "stages_note": "eager, unpipelined step; CUDA events on the launch stream, median",
                "ncu_kernels": ncu_kernels, "fp64_peak_tflops_measured": round(fp64_tflops, 2)}

    # ---------------- end to end through the public API with HOST buffers (h2d + d2h inside the timed region):
    # numpy node tables on the host -> Engine -> every output stream of every path back in (pinned) host memory
    for hres in eng.stream_to_host([packed] * 3, tiles=args.e2e_tiles):
        pass
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for hres in eng.stream_to_host([packed] * args.steps, tiles=args.e2e_tiles):
        pass
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    assert int(hres.n_out.sum()) == int(res.n_out.sum().item())
    b0 = hres.path(B - 1)
    assert np.array_equal(b0["x"], res.path(B - 1)["x"])
    tt = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_step_ms = float(tt.item())
    d2h_bytes = hres.bytes_per_step()
    h2d = sum(a.nbytes for a in (packed.node_attr, packed.node_flags, packed.n_nodes, packed.ap_attr, packed.ap_flags,
                                 packed.n_ap, packed.cons))
    host_sink = d2h_microbench(torch, dev, dist, world)
    e2e_gbps = world * d2h_bytes / 1e9 / (e2e_step_ms * 1e-3)
    e2e = {"value": world * B / (e2e_step_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_step_ms,
           "d2h_GBps_achieved_all_ranks": round(e2e_gbps, 1), "host_sink_microbench": host_sink,
           "frac_of_host_sink": round(e2e_gbps / host_sink["aggregate_GBps"], 3),
           "how": (f"host numpy node tables -> pinned -> device, {args.e2e_tiles} tile(s), dense result rows packed on the "
                   f"device and moved by the copy engine; {args.steps} batches streamed through a 3-deep pipeline (batch n+1 "
                   "computes and batch n+2 is enqueued while batch n crosses PCIe), wall clock of the whole stream incl. fill "
                   "and drain / batches.  host_sink_microbench = every rank copying 512 MB device -> pinned host at once "
                   "(what this box's PCIe / host memory can absorb)")}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        rate, n, el = cpu_port_rate(packed, args.cpu_seconds, threads)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{n} of the {B} paths, {el:.1f} s, C restatement of the reference (oracle/) with OpenMP",
               "reference_python": None if args.no_pyref else python_reference_rate(packed, 2 * threads, threads)}
    if rank == 0:
        line = {
            "metric": metric_name(N), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": label, "paths_per_gpu": B, "nodes": N,
                       "l2": "flushed before every timed step (256 MB write on the step's stream); a step also streams "
                             "about 5 GB of intermediates through the 126 MB L2",
                       "pipeline_depth": depth, "cuda_graph": True, "ms_per_step_serial": serial_ms,
                       "first_call_ms": round(first_call_ms, 2), "second_call_eager_ms": round(second_call_ms, 2),
                       "pipelining": "consecutive steps are independent batches: two CUDA graphs replayed on two streams; "
                                     "timed region = K steps enqueued back to back, CUDA events on the launching stream "
                                     "around the whole region, max over ranks",
                       "mean_D": Dsum / B, "mean_T": Tsum / B, "wall_s": wall, "cpu_affinity": affinity},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ cfg3 (sharded job)
def run_cfg3(args):
    import torch
    import torch.distributed as dist

    from vexautonomousplanner_b200 import synth
    from vexautonomousplanner_b200.engine import ST_CAPACITY, Engine, PipelinedProfiler
    from vexautonomousplanner_b200.packing import pack_arrays
    from vexautonomousplanner_b200.sharding import SummaryGatherer, shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    affinity = set_local_affinity(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, N, seed, label = workload(args)
    tile = args.tile
    # every rank draws the same pixels (seed 1), balances the contiguous shards on the chord-length sums and packs its own
    rng = np.random.default_rng(seed)
    px = synth.random_pixels(rng, B, N)
    chord = np.linalg.norm(np.diff(px, axis=1), axis=2).sum(axis=1)
    bounds = shard_bounds(B, world, chord)
    lo, hi = bounds[rank]
    packed = pack_arrays(None, synth.FACTORY, points_px=px[lo:hi])
    del px
    Bl = packed.B
    n_tiles = (Bl + tile - 1) // tile
    eng = Engine(dev, chunks=args.chunks)

    def tile_packed(k):
        a, b = k * tile, min(Bl, (k + 1) * tile)
        sub = packed.slice(a, b)
        if sub.B < tile:                               # ragged last tile: pad with copies of its first path (results dropped)
            pad = tile - sub.B
            rep = lambda x: np.concatenate([x, np.repeat(x[:1], pad, axis=0)])    # noqa: E731
            sub = type(sub)(rep(sub.node_attr), rep(sub.node_flags), rep(sub.n_nodes), rep(sub.ap_attr), rep(sub.ap_flags),
                            rep(sub.n_ap), rep(sub.cons))
        return sub, b - a

    tiles_host = [tile_packed(k) for k in range(n_tiles)]
    tiles_dev = [eng.upload(t) for t, _ in tiles_host]                    # inputs resident in HBM (value); 25 MB per tile
    pin = [[torch.from_numpy(a).pin_memory() for a in (t.node_attr, t.node_flags, t.n_nodes, t.ap_attr, t.ap_flags, t.n_ap, t.cons)]
           for t, _ in tiles_host]
    depth = max(1, args.pipeline)
    pipe = PipelinedProfiler(eng, tiles_dev[0], depth=depth, margin=args.margin)
    summaries = torch.zeros((n_tiles * tile, 5), dtype=torch.float64, device=dev)
    counters = torch.zeros((n_tiles * tile, 2), dtype=torch.float64, device=dev)      # D, T per path (roofline bytes)
    gatherer = SummaryGatherer([b - a for a, b in bounds], dev, slots=2)
    main = torch.cuda.current_stream(dev)
    from vexautonomousplanner_b200.engine import DeviceBatch

    def job(from_host: bool):
        """The whole shard: every tile through the pipelined graphs; summaries (and D, T) kept, trajectories reduced away."""
        for k in range(n_tiles):
            def consume(res, k=k):
                summaries[k * tile:(k + 1) * tile].copy_(res.summary, non_blocking=True)
                counters[k * tile:(k + 1) * tile, 0].copy_(res.n_samples, non_blocking=True)
                counters[k * tile:(k + 1) * tile, 1].copy_(res.n_out, non_blocking=True)
            if from_host:
                slot = pipe.graphs[pipe.n % depth]
                st = pipe.streams[pipe.n % depth]
                st.wait_stream(main)
                with torch.cuda.stream(st):            # h2d of this tile's inputs from pinned host memory, on the slot's stream
                    for dst, src in zip((slot.db.node_attr, slot.db.node_flags, slot.db.n_nodes, slot.db.ap_attr,
                                         slot.db.ap_flags, slot.db.n_ap, slot.db.cons), pin[k]):
                        dst.copy_(src, non_blocking=True)
                pipe.submit(None, consume)
            else:
                pipe.submit(tiles_dev[k], consume)
        pipe.drain()
        redone_now = redo_overflows()                 # inside the job (and its timing): one status read-back per job
        gatherer.submit(summaries[:Bl])
        gatherer.wait()
        return redone_now

    def redo_overflows():
        """Exact re-run (outside the graphs) of any tile whose paths did not fit the planned capacities."""
        st = summaries[:, 4]
        bad = torch.nonzero(st == ST_CAPACITY).flatten().tolist()
        redone = sorted({i // tile for i in bad})
        for k in redone:
            r = eng.profile(tiles_dev[k], reuse_plan=False)
            summaries[k * tile:(k + 1) * tile].copy_(r.summary)
            counters[k * tile:(k + 1) * tile, 0].copy_(r.n_samples); counters[k * tile:(k + 1) * tile, 1].copy_(r.n_out)
        return redone

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    redone = []
    for _ in range(max(1, args.warmup)):
        redone = job(False)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = eng.launches
    barrier()
    s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    s.record(main)
    for _ in range(args.steps):
        redone = job(False)
    e.record(main)
    barrier()
    wall = time.perf_counter() - wall0
    launches = (eng.launches - l0) // args.steps
    clocks = sampler.stop() if sampler else None
    tt = torch.tensor([s.elapsed_time(e)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_per_step = float(tt.item()) / args.steps
    value = B / (ms_per_step * 1e-3)
    ok = summaries[:Bl, 4] == 0
    assert bool(ok.all().item()), "paths with a non-zero status"
    allrows = gatherer.rows()
    assert allrows.shape == (B, 5)
    if args.dump_outputs and rank == 0:
        write_dump(args.dump_outputs, summary_dump(allrows.cpu().numpy()))

    # roofline with every path's actual Q, P, D, T (SURVEY.md 8d): B_path = 8 (2Q + 2P + 10D + 9T) + 88 N
    Dsum = float(counters[:Bl, 0].sum().item()); Tsum = float(counters[:Bl, 1].sum().item())
    stats = torch.tensor([Dsum, Tsum, float(Bl)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    Dall, Tall, Ball = (float(x) for x in stats.tolist())
    alg_bytes = 8 * (2 * 1000.0 * Ball + 2 * 1000.0 * N * Ball + 10 * Dall + 9 * Tall) + 88 * N * Ball
    peak, peak_src = measured_peak()
    roofline = {"bound": "hbm", "kernel": "whole job (all stages, all tiles)", "achieved": alg_bytes / 1e9 / (ms_per_step * 1e-3) / world,
                "peak": peak, "unit": "GB/s", "frac": alg_bytes / 1e9 / (ms_per_step * 1e-3) / world / peak, "traffic": None,
                "peak_source": peak_src, "per_gpu": True, "alg_GB_job": alg_bytes / 1e9,
                "note": "achieved = algorithmic bytes of the whole job (each path's own Q, P, D, T) / job time / GPUs"}

    # end to end: the inputs of every tile come from pinned host memory inside the timed region; the per-path summary rows
    # of the shard go back to the host.  (The trajectories of the full job are 190 GB: they stay on the producing GPU /
    # are reduced per tile; nothing the reference's caller of this config could hold either.)
    job(True); barrier()
    t0 = time.perf_counter()
    for _ in range(max(1, args.steps // 2)):
        job(True)
        host_rows = summaries[:Bl].cpu()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / max(1, args.steps // 2)
    tt = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_ms = float(tt.item())
    h2d = sum(t.numel() * t.element_size() for tl in pin for t in tl)
    e2e = {"value": B / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": host_rows.numel() * 8,
           "ms_per_step": e2e_ms, "how": "per rank: every tile's node tables pinned host -> device on the tile's stream inside "
           "the timed region, summary rows of the shard device -> host; wall clock, max over ranks"}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        rate, n, el = cpu_port_rate(packed.slice(0, min(Bl, 2048)), args.cpu_seconds, threads)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{n} of the job's paths, {el:.1f} s, C restatement of the reference (oracle/) with OpenMP",
               "reference_python": None if args.no_pyref else python_reference_rate(packed, threads, threads)}
    if rank == 0:
        line = {
            "metric": metric_name(N), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(1, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": label, "paths_total": B, "nodes": N, "tile_paths": tile, "tiles_per_rank": n_tiles,
                       "shards": [b - a for a, b in bounds], "shard_balance": "contiguous, chord-length sums",
                       "pipeline_depth": depth, "capacity_margin": args.margin, "tiles_redone_exactly": redone,
                       "l2": "no flush: every tile streams tens of GB through the 126 MB L2", "step": "one whole job",
                       "mean_D": Dall / Ball, "mean_T": Tall / Ball, "wall_s": wall, "cpu_affinity": affinity},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3"])
    ap.add_argument("--paths", type=int, default=None)
    ap.add_argument("--nodes", type=int, default=None)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-sample", type=int, default=1024)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pyref", action="store_true", help="skip timing the unmodified Python reference (baseline/_ref)")
    ap.add_argument("--chunks", type=int, default=32, help="speculative chunks per path in the velocity passes")
    ap.add_argument("--pipeline", type=int, default=2, help="independent batches in flight on the device (1: none)")
    ap.add_argument("--tile", type=int, default=8192, help="cfg3: paths per tile")
    ap.add_argument("--margin", type=float, default=1.3, help="cfg3: capacity margin over the first tile's plan")
    ap.add_argument("--e2e-tiles", type=int, default=1, help="tiles of the end-to-end (host in / host out) run")
    ap.add_argument("--profile-step", action="store_true",
                    help="cfg2: run only warm-up + K eager, unpipelined steps (the command profiles/tools/capture.sh puts under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 3 if args.config == "cfg3" else 10
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "cfg3":
        run_cfg3(args)
    else:
        run_cfg2(args)


if __name__ == "__main__":
    main()
