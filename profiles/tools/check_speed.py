"""Bulk check speed: reading saved trajectory text back on the device and comparing it with fresh bodies, 4096 paths.

    python profiles/tools/check_speed.py OUTDIR

Workloads as profiles/tools/save_speed.py: cfg2 (4096 random 8-node paths, factory constraints) and cfg5
(synth.mixed_paths(4096, 8, seed=3) with random int action tuples).  The fresh bodies of save_text_batch are written to
a temporary directory as the saved files.  Per workload, medians of --reps warmed runs:
- device parse: CUDA events around parse_text_batch's stages (upload, lines, parse), text GB/s over lines + parse, and
  the host wall time of the whole call (synchronised);
- per-kernel device times of one parse_text_batch under torch.profiler (a run of its own);
- the whole --check of the batch (save_routes.check_batch: profile, fresh bodies, file reads, device compare), host
  clock, synchronised; every file must come back up to date;
- the Python float() loop over the trajectory-row tokens of the first 256 bodies, scaled to the batch by row count.
Writes OUTDIR/check_speed.json.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

N_SAMPLE = 256
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--paths", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import torch
    from save_speed import workload
    from vexautonomousplanner_b200 import export as ex, synth
    from vexautonomousplanner_b200.engine import Engine
    from vexautonomousplanner_b200.save_routes import check_batch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), paths=a.paths, workloads={})
    eng = Engine("cuda:0")
    for name in ("cfg2", "cfg5"):
        packed, na, aa = workload(synth, name, a.paths)
        db = eng.upload(packed)
        res = eng.profile(db)
        text, offs, ok = ex.save_text_batch(eng, res, db, na, aa)
        nbytes = int(offs[-1])
        ex.parse_text_batch(eng, text, offs)                                  # warm-up
        stages, walls = {}, []
        for _ in range(a.reps):
            eng.stage_events = []
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            p = ex.parse_text_batch(eng, text, offs)
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
            for st, s, e in eng.stage_events:
                stages.setdefault(st, []).append(s.elapsed_time(e))
            eng.stage_events = None
        med = {k: float(np.median(v)) for k, v in stages.items()}
        parse_ms = med["read_lines"] + med["read_parse"]
        R = int(p.rows.shape[0])
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            ex.parse_text_batch(eng, text, offs)
            torch.cuda.synchronize()
        kernels = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            if t:
                kernels[ev.key[:80]] = kernels.get(ev.key[:80], 0.0) + t / 1e3          # ms
        files = tempfile.mkdtemp()
        paths = [os.path.join(files, f"r{b}.txt") for b in range(res.B)]
        for b in range(res.B):
            if ok[b]:
                with open(paths[b], "wb") as f:
                    f.write(text[offs[b]:offs[b + 1]].tobytes())
        check_batch(eng, db, na, aa, paths)                                    # warm-up
        checks = []
        for _ in range(a.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, ok2, present, ints, floats = check_batch(eng, db, na, aa, paths)
            checks.append(time.perf_counter() - t0)
            assert (ints[ok2, 0] == -1).all(), "a saved file did not come back up to date"
        shutil.rmtree(files)
        # the Python loop: float() of every trajectory-row token of the first N_SAMPLE bodies
        sample = bytes(text[offs[0]:offs[min(N_SAMPLE, res.B)]]).decode().splitlines()
        t0 = time.perf_counter()
        r_sample = 0
        for line in sample:
            tok = line.split()
            if tok[0] == "0":
                [float(v) for v in tok]
                r_sample += 1
        t_loop = time.perf_counter() - t0
        report["workloads"][name] = dict(
            ok_paths=int(ok.sum()), text_bytes=nbytes, lines=int(p.line_kinds.shape[0]), trajectory_rows=R,
            numeric_tokens=7 * R, host_fallback_tokens=p.n_host,
            parse_stage_ms_median=med, parse_device_ms=parse_ms, parse_text_gbs=nbytes / (parse_ms * 1e-3) / 1e9,
            parse_text_batch_wall_ms_median=1e3 * float(np.median(walls)),
            parse_kernels_ms_profiler=dict(sorted(kernels.items(), key=lambda kv: -kv[1])[:12]),
            check_batch_wall_ms_median=1e3 * float(np.median(checks)),
            python_float_loop=dict(sample_paths=min(N_SAMPLE, res.B), sample_rows=r_sample, sample_s=t_loop,
                                   scaled_to_batch_s=t_loop * R / max(r_sample, 1)))
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "check_speed.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
