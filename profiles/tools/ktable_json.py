"""ncu launch list (CSV of profiles/tools/ncu_table.sh) -> per-kernel / per-stage JSON table that bench.py reads for the
measured DRAM traffic of the dominant stage.  usage: ktable_json.py <launches.csv> <out.json> [peak GB/s] [commit]"""
import collections
import csv
import json
import sys

STAGE = {"k_build_path": "S0_build_path", "k_build_lut": "S1_lut", "k_build_lut_index": "S1_lut", "k_build_props": "S2_props",
         "k_flag_lengths": "S345_velocity", "k_count_samples": "S345_velocity", "k_sample_prepass": "S345_velocity",
         "k_resolve_events": "S345_velocity", "k_prepass_ovr": "S345_velocity", "k_fwd_chunked": "S345_velocity",
         "k_bwd_chunked": "S345_velocity", "k_flag_times": "S345_velocity",
         "k_time_state": "S6_resample", "k_time_sample": "S6_resample", "k_time_events": "S6_resample",
         "k_time_finalize": "S6_resample", "k_need_rows": "S6_resample"}
M = {"ms": "gpu__time_duration.sum", "rd": "dram__bytes_read.sum", "wr": "dram__bytes_write.sum", "inst": "smsp__inst_executed.sum",
     "issue": "smsp__issue_active.avg.pct_of_peak_sustained_active", "fp64": "sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active",
     "warps": "sm__warps_active.avg.pct_of_peak_sustained_active"}


def main():
    src, dst = sys.argv[1], sys.argv[2]
    peak = float(sys.argv[3]) if len(sys.argv) > 3 else 6544.7
    commit = sys.argv[4] if len(sys.argv) > 4 else None
    rows = [r for r in csv.reader(open(src)) if len(r) > 5]
    hdr = rows[0]
    ik, im, iv, iid = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("ID")
    per = collections.OrderedDict()
    for r in rows[1:]:
        name = r[ik].split("(")[0].replace("void ", "").split("<")[0]
        per.setdefault((r[iid], name), {})[r[im]] = float(r[iv].replace(",", ""))
    agg = collections.OrderedDict()
    for (_, name), m in per.items():
        if name not in STAGE:
            continue
        a = agg.setdefault(name, collections.Counter())
        a["n"] += 1
        for k, v in m.items():
            a[k] += v
    steps = max(a["n"] for a in agg.values() if a["n"]) if agg else 1
    steps = min(steps, 2) if steps >= 2 else 1
    kernels, stages = {}, {}
    for name, a in agg.items():
        n = a["n"]
        ms = a[M["ms"]] / n / 1e6
        rd, wr = a[M["rd"]] / n, a[M["wr"]] / n
        kernels[name] = {"launches_sampled": int(n), "ms": round(ms, 4), "dram_read_MB": round(rd / 1e6, 1),
                         "dram_write_MB": round(wr / 1e6, 1), "dram_GBps": round((rd + wr) / 1e9 / (ms * 1e-3), 1),
                         "dram_frac_of_measured_peak_%g" % peak: round((rd + wr) / 1e9 / (ms * 1e-3) / peak, 3),
                         "warp_inst_M": round(a[M["inst"]] / n / 1e6, 1), "issue_active_pct": round(a[M["issue"]] / n, 1),
                         "fp64_pipe_pct": round(a[M["fp64"]] / n, 1), "warps_active_pct": round(a[M["warps"]] / n, 1)}
        s = stages.setdefault(STAGE[name], {"ms": 0.0, "dram_bytes_per_step": 0.0})
        s["ms"] += ms
        s["dram_bytes_per_step"] += rd + wr
    for s in stages.values():
        s["ms"] = round(s["ms"], 4)
        s["dram_bytes_per_step"] = round(s["dram_bytes_per_step"], -5)
    out = {"command": "bash profiles/tools/capture.sh (ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,"
                      "smsp__inst_executed.sum,smsp__issue_active...,sm__pipe_fp64_cycles_active...,sm__warps_active... "
                      "--clock-control none python bench.py --profile-step --steps 2 --warmup 2)",
           "commit": commit,
           "workload": "4096 random 8-node paths, 1 B200",
           "note": "per-launch averages over the sampled steps; ncu serialises kernels and runs them cold, compare SHARES with "
                   "bench.py's CUDA-event stage times",
           "kernels": kernels, "stages": stages}
    json.dump(out, open(dst, "w"), indent=1)
    tot = sum(k["ms"] for k in kernels.values())
    for name, k in sorted(kernels.items(), key=lambda kv: -kv[1]["ms"]):
        print(f"{name:20s} {k['ms']:7.4f} ms  {100 * k['ms'] / tot:5.1f}%  {k['dram_GBps']:7.1f} GB/s  fp64 {k['fp64_pipe_pct']:5.1f}%")
    print("sum", round(tot, 3), "ms")


if __name__ == "__main__":
    main()
