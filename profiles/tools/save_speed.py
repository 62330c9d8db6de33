"""Bulk save speed: profile + device text assembly + copy + files for 4096 paths, against the per-path trajectory_text loop.

    python profiles/tools/save_speed.py OUTDIR [--parent-tree DIR]

Workloads: cfg2 (4096 random 8-node paths, factory constraints, node rows [0, 0], no action points) and cfg5
(synth.mixed_paths(4096, 8, seed=3): turns, waits, reverses, stops, 0-2 action points; random int action tuples of
length 0-3).  Per workload: profile time (host clock around Engine.profile, synchronised), device time of the text
assembly per phase (CUDA events of save_text_batch's stages, after warm-up), text bytes and the text rate against the
B200's 7.7 TB/s, the device-to-host copy, and the wall time from profile to files written (to a temporary directory).
--parent-tree DIR: a checkout of the commit before save_text_batch, with libvap.so built in it; the per-path loop
(export_text_device once, then trajectory_text per path with its device_text) runs there on the first 256 paths of the
same seeded batch, in a subprocess, and is scaled to the batch.  Writes OUTDIR/save_speed.json.
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

HBM_GBS = 7700.0
N_SAMPLE = 256


def workload(synth, name, B):
    if name == "cfg2":
        packed = synth.random_paths(B, 8, seed=0)
        na = [[[0, 0]] * int(n) for n in packed.n_nodes]
        aa = [[] for _ in range(B)]
    else:
        packed = synth.mixed_paths(B, 8, seed=3)
        rng = np.random.default_rng(5)
        tup = lambda: [int(x) for x in rng.integers(0, 10, rng.integers(0, 4))]
        na = [[tup() for _ in range(int(n))] for n in packed.n_nodes]
        aa = [[tup() for _ in range(int(a))] for a in packed.n_ap]
    return packed, na, aa


def per_path_loop(tree, B):
    """The parent's per-path loop, run in `tree` (imported from there): seconds for N_SAMPLE paths and for the export."""
    sys.path.insert(0, tree)
    import torch
    from vexautonomousplanner_b200 import export as ex, synth
    from vexautonomousplanner_b200.engine import Engine
    eng = Engine("cuda:0")
    out = {}
    for name in ("cfg2", "cfg5"):
        packed, na, aa = workload(synth, name, B)
        db = eng.upload(packed)
        res = eng.profile(db)
        for rep in range(2):                        # the first pass warms up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dev = ex.export_text_device(eng, res, db)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            nbytes = 0
            for b in range(N_SAMPLE):
                nbytes += len(ex.trajectory_text(eng, res, b, na[b], aa[b], db=db, device_text=dev))
            t2 = time.perf_counter()
        out[name] = dict(export_s=t1 - t0, loop_s=t2 - t1, sample_paths=N_SAMPLE, sample_bytes=nbytes)
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--parent-tree")
    ap.add_argument("--paths", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--per-path-only", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.per_path_only:
        return per_path_loop(a.per_path_only, a.paths)
    root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, root)
    import torch
    from vexautonomousplanner_b200 import export as ex, synth
    from vexautonomousplanner_b200.engine import Engine
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), paths=a.paths, workloads={})
    eng = Engine("cuda:0")
    for name in ("cfg2", "cfg5"):
        packed, na, aa = workload(synth, name, a.paths)
        db = eng.upload(packed)
        res = eng.profile(db)                                           # warm-up of the profile
        torch.cuda.synchronize()
        prof = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            res = eng.profile(db)
            torch.cuda.synchronize()
            prof.append(time.perf_counter() - t0)
        ex.save_text_batch(eng, res, db, na, aa)                        # warm-up of the assembly
        stages, walls, files = {}, [], tempfile.mkdtemp()
        for _ in range(a.reps):
            eng.stage_events = []
            t0 = time.perf_counter()
            text, offs, ok = ex.save_text_batch(eng, res, db, na, aa)
            t_asm = time.perf_counter() - t0
            torch.cuda.synchronize()
            for st, s, e in eng.stage_events:
                stages.setdefault(st, []).append(s.elapsed_time(e))
            eng.stage_events = None
            walls.append(t_asm)
        # wall time to files: profile + assembly + one write per path
        t0 = time.perf_counter()
        res = eng.profile(db)
        text, offs, ok = ex.save_text_batch(eng, res, db, na, aa)
        for b in range(res.B):
            if ok[b]:
                with open(os.path.join(files, f"r{b}.txt"), "wb") as f:
                    f.write(text[offs[b]:offs[b + 1]].tobytes())
        t_files = time.perf_counter() - t0
        shutil.rmtree(files)
        med = {k: float(np.median(v)) for k, v in stages.items()}
        dev_ms = med["text_format"] + med["text_splice_plan"] + med["text_splice_copy"]
        nbytes = int(offs[-1])
        report["workloads"][name] = dict(
            ok_paths=int(ok.sum()), text_bytes=nbytes, lines=int((text == 10).sum()),
            profile_ms_median=1e3 * float(np.median(prof)), stage_ms_median=med, assembly_device_ms=dev_ms,
            assembly_text_gbs=nbytes / (dev_ms * 1e-3) / 1e9,
            assembly_text_share_of_hbm=nbytes / (dev_ms * 1e-3) / 1e9 / HBM_GBS,
            d2h_gbs=nbytes / (med["text_d2h"] * 1e-3) / 1e9,
            save_text_batch_wall_ms_median=1e3 * float(np.median(walls)), profile_to_files_wall_ms=1e3 * t_files)
    if a.parent_tree:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), a.outdir, "--paths", str(a.paths),
                            "--per-path-only", os.path.abspath(a.parent_tree)], capture_output=True, text=True,
                           cwd=a.parent_tree)
        if r.returncode != 0:
            report["per_path_error"] = r.stderr[-2000:]
        else:
            pp = json.loads(r.stdout.strip().splitlines()[-1])
            for name, v in pp.items():
                v["loop_scaled_to_batch_s"] = v["loop_s"] * a.paths / v["sample_paths"]
                v["export_plus_scaled_loop_s"] = v["export_s"] + v["loop_scaled_to_batch_s"]
                w = report["workloads"][name]
                w["parent_per_path"] = v
                w["speedup_vs_parent_per_path"] = v["export_plus_scaled_loop_s"] / (w["save_text_batch_wall_ms_median"] * 1e-3)
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "save_speed.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
