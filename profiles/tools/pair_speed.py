"""Pair check speed: vap_pair_check over cross products of synth.mixed_paths routes, against the numpy reference.

    python profiles/tools/pair_speed.py OUTDIR

Workloads: synth.mixed_paths(2 N, 8, seed=3) profiled once, rows from export_rows; routes 0 .. N-1 are side A, N .. 2N-1
side B, every A route against every B route (N = 64 and 256: 4096 and 65536 pairs), an 18 x 15 in robot against an
18 x 18 in one, min_gap 0.  Both sides are one row set, so vap_pose_planes runs once over all 2N routes.
Per workload: device times (CUDA events, median of --reps warmed launches) of vap_pose_planes and of vap_pair_check
alone, events/s (na + nb per pair), the whole export.pair_check call (host clock, synchronised, read-back included),
and the numpy reference of tests/test_pair_check.py on a sample of pairs, scaled to the workload by events (labelled
as scaled).  A control launch puts every A route against one-row B routes (each B route's first row): the held-row
search then takes one step, the geometry per event is unchanged, so its time per event against the cross product's
shows what the search costs.  The card's name, power limit and clock come from nvidia-smi in the same run.  Writes
OUTDIR/pair_speed.json.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
SIZE_A, SIZE_B = (18.0, 15.0), (18.0, 18.0)
N_SAMPLE = 64


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    from test_pair_check import ref_pair
    from vexautonomousplanner_b200 import _lib, export as ex, synth
    from vexautonomousplanner_b200.engine import Engine, _p
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), robot_a_in=SIZE_A, robot_b_in=SIZE_B, min_gap_in=0.0,
                  workloads={})
    eng = Engine("cuda:0")
    st = eng._stream()

    def median_ms(launch):
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
        return float(np.median(times)), float(np.min(times)), float(np.max(times))

    for N in (64, 256):
        res = eng.profile(eng.upload(synth.mixed_paths(2 * N, 8, seed=3)))
        rows, off = ex.export_rows(eng, res)
        R, B = int(rows.shape[0]), 2 * N
        pairs = np.array([(i, N + j) for i in range(N) for j in range(N)], dtype=np.int64)
        P = len(pairs)
        planes = torch.empty(5 * max(R, 1), dtype=torch.float64, device=eng.device)
        bad = torch.empty((B, 2), dtype=torch.int64, device=eng.device)
        pr = torch.from_numpy(pairs).to(eng.device)
        out_i = torch.empty((P, len(ex.PC_I)), dtype=torch.int64, device=eng.device)
        out_f = torch.empty((P, len(ex.PC_F)), dtype=torch.float64, device=eng.device)

        def planes_launch():
            _lib.check(eng.lib.vap_pose_planes(C.c_int64(B), _p(rows), _p(off), C.c_int64(R), _p(planes), _p(bad), st),
                       "vap_pose_planes")

        def pair_launch(pr_=pr, off_b=off, planes_b=planes, R_b=R, B_b=B, bad_b=bad, P_=P):
            _lib.check(eng.lib.vap_pair_check(
                C.c_int64(P_), _p(pr_), C.c_int64(B), _p(planes), C.c_int64(R), _p(off), _p(bad),
                C.c_double(SIZE_A[0] / 2), C.c_double(SIZE_A[1] / 2), C.c_int64(B_b), _p(planes_b), C.c_int64(R_b),
                _p(off_b), _p(bad_b), C.c_double(SIZE_B[0] / 2), C.c_double(SIZE_B[1] / 2), C.c_double(0.0), _p(out_i),
                _p(out_f), st), "vap_pair_check")

        t_planes = median_ms(planes_launch)
        t_pairs = median_ms(pair_launch)
        events = int(out_i[:, 1].sum().item())
        # control: the same A routes against one-row routes (each B route's first row)
        o = off.cpu().numpy()
        first_rows = rows[torch.from_numpy(o[N:B]).to(eng.device)].contiguous()
        off1 = torch.arange(N + 1, dtype=torch.int64, device=eng.device)
        planes1 = torch.empty(5 * N, dtype=torch.float64, device=eng.device)
        bad1 = torch.empty((N, 2), dtype=torch.int64, device=eng.device)
        _lib.check(eng.lib.vap_pose_planes(C.c_int64(N), _p(first_rows), _p(off1), C.c_int64(N), _p(planes1), _p(bad1), st),
                   "vap_pose_planes")
        pr1 = torch.from_numpy(pairs - np.array([0, N])).to(eng.device)
        t_ctrl = median_ms(lambda: pair_launch(pr1, off1, planes1, N, N, bad1))
        events_ctrl = int(out_i[:, 1].sum().item())
        walls = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            gi, gf, _, _ = ex.pair_check(eng, rows, off, SIZE_A, rows, off, SIZE_B, pairs)
            walls.append(time.perf_counter() - t0)
        host_rows = rows.cpu().numpy()
        rng = np.random.default_rng(0)
        sample = pairs[rng.choice(P, size=min(N_SAMPLE, P), replace=False)]
        ev_s = 0
        t0 = time.perf_counter()
        for i, j in sample:
            ra, rb = host_rows[o[i]:o[i + 1]], host_rows[o[j]:o[j + 1]]
            ref_pair(ra, rb, (SIZE_A[0] / 2, SIZE_A[1] / 2), (SIZE_B[0] / 2, SIZE_B[1] / 2), 0.0)
            ev_s += len(ra) + len(rb)
        t_ref = time.perf_counter() - t0
        report["workloads"][f"{N}x{N}"] = dict(
            routes=B, rows=R, pairs=P, events=events, pairs_checked=int((gi[:, 0] == 0).sum()),
            pairs_in_contact=int((gi[:, 2] >= 0).sum()), plane_bytes=5 * 8 * R,
            pose_planes_ms=dict(median=t_planes[0], min=t_planes[1], max=t_planes[2]),
            pair_check_ms=dict(median=t_pairs[0], min=t_pairs[1], max=t_pairs[2]),
            events_per_s=events / (t_pairs[0] * 1e-3), ns_per_event=t_pairs[0] * 1e6 / events,
            control_one_row_b=dict(events=events_ctrl, ms_median=t_ctrl[0], ns_per_event=t_ctrl[0] * 1e6 / events_ctrl),
            pair_check_call_wall_ms_median=1e3 * float(np.median(walls)),
            numpy_reference=dict(sample_pairs=len(sample), sample_events=ev_s, sample_s=t_ref,
                                 scaled_to_workload_s=t_ref * events / ev_s, scaled=True))
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "pair_speed.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
