"""Footprint check speed: vap_footprint_check over the export rows of 4096 paths, against the numpy reference.

    python profiles/tools/footprint_speed.py OUTDIR

Workloads: cfg2 (synth.random_paths(4096, 8, seed=0)) and cfg5 (synth.mixed_paths(4096, 8, seed=3)), rows from
export_rows; an 18 x 15 in robot, the default field and three keep-out boxes (the layout of tests/test_footprint_check.py).
Per workload: the kernel's device time (CUDA events around --reps warmed launches of vap_footprint_check alone,
median), rows/s, the bytes the kernel reads (7 doubles per row, each row read twice -- for itself and as the previous
row of the next one, counted once here -- plus the offsets) over the kernel time against the B200's 7.7 TB/s, and the
whole export.footprint_check call (host clock, synchronised, including the read-back).  The rows of one batch (about
360 MB for cfg2) do not fit the 126 MB L2.  The numpy reference of tests/test_footprint_check.py runs on the first 256
paths and is scaled to the batch by row count (labelled as scaled).  The card's name, power limit and clock come from
nvidia-smi in the same run.  Writes OUTDIR/footprint_speed.json.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

HBM_GBS = 7700.0
N_SAMPLE = 256
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
LENGTH_IN, WIDTH_IN = 18.0, 15.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--paths", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    from test_footprint_check import _boxes_for, ref_batch
    from vexautonomousplanner_b200 import _lib, export as ex, synth
    from vexautonomousplanner_b200.engine import Engine, _p
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), paths=a.paths, robot_in=[LENGTH_IN, WIDTH_IN],
                  hbm_gbs_datasheet=HBM_GBS, workloads={})
    eng = Engine("cuda:0")
    field = ex.default_field()
    boxes = _boxes_for(field)
    for name in ("cfg2", "cfg5"):
        packed = synth.random_paths(a.paths, 8, seed=0) if name == "cfg2" else synth.mixed_paths(a.paths, 8, seed=3)
        res = eng.profile(eng.upload(packed))
        rows, off = ex.export_rows(eng, res)
        R, B = int(rows.shape[0]), res.B
        arr = np.ascontiguousarray(np.asarray(boxes, dtype=np.float64))
        out_i = torch.empty((B, len(ex.FP_I)), dtype=torch.int64, device=eng.device)
        out_f = torch.empty((B, len(ex.FP_F)), dtype=torch.float64, device=eng.device)
        per_k = {}
        for K in (0, len(boxes)):
            def launch():
                _lib.check(eng.lib.vap_footprint_check(
                    C.c_int64(B), _p(rows), _p(off), C.c_double(LENGTH_IN / 2), C.c_double(WIDTH_IN / 2),
                    *map(C.c_double, field), C.c_int(K), arr.ctypes.data_as(C.c_void_p), C.c_double(0.0), _p(out_i),
                    _p(out_f), eng._stream()), "vap_footprint_check")
            for _ in range(3):
                launch()
            times = []
            for _ in range(a.reps):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                launch()
                e.record()
                e.synchronize()
                times.append(s.elapsed_time(e))
            ms = float(np.median(times))
            nbytes = R * 7 * 8 + (B + 1) * 8 + B * (len(ex.FP_I) + len(ex.FP_F)) * 8
            per_k[f"K{K}"] = dict(kernel_ms_median=ms, kernel_ms_min=float(np.min(times)), kernel_ms_max=float(np.max(times)),
                                  rows_per_s=R / (ms * 1e-3), bytes_read_and_written=nbytes,
                                  gbs=nbytes / (ms * 1e-3) / 1e9, share_of_hbm_datasheet=nbytes / (ms * 1e-3) / 1e9 / HBM_GBS)
        walls = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            gi, gf = ex.footprint_check(eng, rows, off, LENGTH_IN, WIDTH_IN, keep_out=boxes)
            walls.append(time.perf_counter() - t0)
        n_s = min(N_SAMPLE, B)
        o = off.cpu().numpy()
        host_rows = rows[:int(o[n_s])].cpu().numpy()
        t0 = time.perf_counter()
        ref_batch(host_rows, o[:n_s + 1], LENGTH_IN / 2, WIDTH_IN / 2, field, boxes, 0.0)
        t_ref = time.perf_counter() - t0
        report["workloads"][name] = dict(
            rows=R, ok_paths=int((res.status == 0).sum()), paths_with_hits=int((gi[:, 1] >= 0).sum()), launch=per_k,
            footprint_check_wall_ms_median=1e3 * float(np.median(walls)),
            numpy_reference=dict(sample_paths=n_s, sample_rows=int(o[n_s]), sample_s=t_ref,
                                 scaled_to_batch_s=t_ref * R / max(int(o[n_s]), 1), scaled=True))
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "footprint_speed.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
