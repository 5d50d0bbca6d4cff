"""Capture the hardware counters bench.py cannot read outside a profiler, ONE launch per shape, and cache them.

    python tools/measure_counters.py [--what spmm_c5w,spmm_c5w8,spmm_c4,eval_c5w,eval_c4] [--out gpurun_out/kernel_counters.json]

Runs `ncu --metrics ... --clock-control none -k regex:<kernel> --launch-skip <s> -c <n>` over the probe scripts (one GPU; never a bench number)
and writes, keyed the way bench.py looks them up (`profiles/kernel_counters.json` after the file is copied there):

  spmm:<workload>:<world>:<schedule>   (schedule = what DeviceCSR.schedule reports: auto, or spread for the blocks of >= 4 ranks) dram_read_bytes, dram_write_bytes, l2_to_sm_bytes, l2_hit_pct, duration_ms
  eval:<workload>:<world>              per scoring kernel: tensor-pipe cycles active as % of peak sustained ELAPSED, duration
"""
import argparse
import csv
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

SPMM_METRICS = "dram__bytes_read.sum,dram__bytes_write.sum,l1tex__m_xbar2l1tex_read_bytes.sum,lts__t_sector_hit_rate.pct,gpu__time_duration.sum"
EVAL_METRICS = ("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active,"
                "sm__cycles_active.avg,sm__cycles_elapsed.max,gpu__time_duration.sum")

JOBS = {
    # name: (cache key prefix, kernel regex, matching launches to skip, launches to capture, probe command)
    # spmm_probe.py first runs two reference propagations (no split plan, then the binned schedule): skipped.
    "spmm_c5w": ("spmm:c5w:1", "spmm_rows_async", 2, 1, ["tools/spmm_probe.py", "--shapes", "1250000x250000x125000000", "--schedules", "auto", "--splits", "auto", "--iters", "1"]),
    "spmm_c5w8": ("spmm:c5w:8", "spmm_rows_async", 0, 1, ["tools/shard_probe.py", "--schedules", "auto", "--splits", "auto", "--iters", "1"]),
    "spmm_c5w4": ("spmm:c5w:4", "spmm_rows_async", 0, 1, ["tools/shard_probe.py", "--world", "4", "--schedules", "auto", "--splits", "auto", "--iters", "1"]),
    "spmm_c5w2": ("spmm:c5w:2", "spmm_rows_async", 0, 1, ["tools/shard_probe.py", "--world", "2", "--schedules", "auto", "--splits", "auto", "--iters", "1"]),
    "spmm_c5w8s": ("spmm:c5w:8", "spmm_rows_async", 0, 1, ["tools/shard_probe.py", "--schedules", "spread", "--splits", "auto", "--iters", "1"]),
    "spmm_c5w4s": ("spmm:c5w:4", "spmm_rows_async", 0, 1, ["tools/shard_probe.py", "--world", "4", "--schedules", "spread", "--splits", "auto", "--iters", "1"]),
    "spmm_c4": ("spmm:c4:1", "spmm_rows_async", 2, 1, ["tools/spmm_probe.py", "--shapes", "52000x92000x3000000", "--schedules", "auto", "--splits", "auto", "--iters", "1"]),
    "eval_c5w": ("eval:c5w:1", "eval_scores", 0, 2, ["tools/eval_probe.py", "--shape", "c5e", "--users", "262144", "--iters", "1"]),
    "eval_c4": ("eval:c4:1", "eval_scores", 0, 2, ["tools/eval_probe.py", "--shape", "c4", "--iters", "1"]),
}


def to_number(value, unit):
    v = float(value.replace(",", ""))
    scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "ms": 1.0, "us": 1e-3, "ns": 1e-6, "s": 1e3}
    return v * scale.get(unit, 1.0)


def run_ncu(regex, skip, count, metrics, cmd):
    log = tempfile.NamedTemporaryFile(suffix=".csv", delete=False).name
    full = ["ncu", "--metrics", metrics, "--clock-control", "none", "-k", "regex:" + regex, "--launch-skip", str(skip), "-c", str(count),
            "--csv", "--log-file", log, sys.executable] + cmd
    subprocess.run(full, cwd=ROOT, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    rows = list(csv.reader(open(log, errors="replace")))
    hdr = next(k for k, r in enumerate(rows) if r and r[0] == "ID")
    cols = {name: k for k, name in enumerate(rows[hdr])}
    launches = {}
    for r in rows[hdr + 1:]:
        if len(r) <= cols["Metric Value"]:
            continue
        d = launches.setdefault((r[cols["ID"]], r[cols["Kernel Name"]]), {})
        d[r[cols["Metric Name"]]] = to_number(r[cols["Metric Value"]], r[cols["Metric Unit"]])
    return launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--what", default=",".join(JOBS))
    ap.add_argument("--merge", default=os.path.join(ROOT, "profiles", "kernel_counters.json"), help="existing cache to start from")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "kernel_counters.json"))
    args = ap.parse_args()
    out = {}
    for path in (args.merge, args.out):
        if path and os.path.exists(path):
            out.update(json.load(open(path)))
    for name in args.what.split(","):
        prefix, regex, skip, count, cmd = JOBS[name]
        launches = run_ncu(regex, skip, count, SPMM_METRICS if prefix.startswith("spmm") else EVAL_METRICS, cmd)
        src = "ncu --metrics (tools/measure_counters.py %s): %s" % (name, " ".join(cmd))
        if prefix.startswith("spmm"):
            (_, kname), m = next(iter(launches.items()))
            # the schedule `auto` resolves to for this shape (graph.work_schedule): windowed above a 64 MB table, else binned
            sched = cmd[cmd.index("--schedules") + 1] if "--schedules" in cmd else "auto"
            out["%s:%s" % (prefix, sched)] = {
                "kernel": kname.split("(")[0], "dram_read_bytes": m["dram__bytes_read.sum"], "dram_write_bytes": m["dram__bytes_write.sum"],
                "l2_to_sm_bytes": m["l1tex__m_xbar2l1tex_read_bytes.sum"], "l2_hit_pct": m["lts__t_sector_hit_rate.pct"],
                "duration_ms": m["gpu__time_duration.sum"], "source": src}
        else:
            ks = []
            for (_, kname), m in launches.items():
                ks.append({"kernel": kname.split("(")[0], "tensor_pipe_pct_elapsed": m["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed"],
                           "tensor_pipe_pct_active": m["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"],
                           "sm_cycles_active_avg": m["sm__cycles_active.avg"], "sm_cycles_elapsed_max": m["sm__cycles_elapsed.max"],
                           "duration_ms": m["gpu__time_duration.sum"]})
            out[prefix] = {"kernels": ks, "source": src}
        print(name, json.dumps(out.get(prefix) or out.get("%s:auto" % prefix))[:400], flush=True)
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
