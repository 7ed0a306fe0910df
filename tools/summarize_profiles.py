#!/usr/bin/env python
"""Condense the raw outputs of tools/profile_round.sh (gpurun_out/) into the tracked summaries under profiles/.

    python tools/summarize_profiles.py r01
"""
import collections
import csv
import io
import json
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = sys.argv[1] if len(sys.argv) > 1 else "r01"
O = os.path.join(ROOT, "gpurun_out")
P = os.path.join(ROOT, "profiles")
os.makedirs(P, exist_ok=True)

UNIT = {"ns": 1e-3, "nsecond": 1e-3, "us": 1.0, "usecond": 1.0, "ms": 1e3, "msecond": 1e3, "s": 1e6}


def launches():
    src = os.path.join(O, f"launches_{R}.csv")
    if not os.path.exists(src):
        return
    rows = list(csv.reader(open(src)))
    hdr = [i for i, r in enumerate(rows) if r and r[0] == "ID"][0]
    H = rows[hdr]
    ki, vi, ui = H.index("Kernel Name"), H.index("Metric Value"), H.index("Metric Unit")
    agg = collections.OrderedDict()
    for r in rows[hdr + 1:]:
        if len(r) <= vi:
            continue
        name = r[ki].split("(")[0].replace("void ", "").replace("ust::", "")
        us = float(r[vi].replace(",", "")) * UNIT.get(r[ui], 1.0)
        a = agg.setdefault(name, [0, 0.0])
        a[0] += 1
        a[1] += us
    tot = sum(v[1] for v in agg.values())
    with open(os.path.join(P, f"ncu_launches_{R}.txt"), "w") as f:
        f.write("# ncu --metrics gpu__time_duration.sum --clock-control none, first 6000 launches of\n"
                "#   python bench.py --n 256 --nfreq 2 --steps 1 --warmup 1 --no-cpu-baseline   (one B200)\n"
                "# per-launch times are cold-cache and serialised: compare SHARES, not absolutes\n")
        f.write(f"{'kernel':58s} {'launches':>8s} {'total_us':>11s} {'share':>7s} {'avg_us':>8s}\n")
        for k, v in sorted(agg.items(), key=lambda x: -x[1][1]):
            f.write(f"{k[:58]:58s} {v[0]:8d} {v[1]:11.1f} {v[1] / tot:7.3f} {v[1] / v[0]:8.2f}\n")


KEYS = [
    "gpu__time_duration.sum", "sm__cycles_elapsed.avg", "sm__cycles_active.avg", "sm__cycles_elapsed.avg.per_second",
    "launch__registers_per_thread", "launch__grid_size", "launch__block_size", "launch__shared_mem_per_block_dynamic",
    "dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
    "lts__throughput.avg.pct_of_peak_sustained_elapsed", "lts__t_sector_hit_rate.pct",
    "l1tex__throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum",
    "sm__mem_tensor_cycles_active.avg.pct_of_peak_sustained_active", "sm__mem_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed",
    "sm__mem_tensor_cycles_active.max.pct_of_peak_sustained_elapsed",
    "sm__inst_executed_pipe_tmem.avg.pct_of_peak_sustained_active", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
    "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__inst_executed.sum",
    "smsp__average_warps_issue_stalled_long_scoreboard_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_short_scoreboard_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio",
]


def ncu_rep(name, title):
    rep = os.path.join(O, f"{name}_{R}.ncu-rep")
    if not os.path.exists(rep):
        return
    out = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(out)))
    if len(rows) < 3:
        return
    H = rows[0]
    with open(os.path.join(P, f"ncu_{name.replace('prof_', '')}_{R}.txt"), "w") as f:
        f.write(f"# {title}\n# ncu --set full --clock-control none, one line per captured launch (values | unit)\n")
        ki = H.index("Kernel Name")
        for r in rows[2:]:
            f.write(f"kernel: {r[ki]}\n")
        for k in KEYS:
            if k in H:
                i = H.index(k)
                f.write(f"{k:82s} {rows[1][i]:12s} " + "  ".join(r[i] for r in rows[2:]) + "\n")


def copy(src, dst, header=None):
    s = os.path.join(O, src)
    if os.path.exists(s):
        with open(os.path.join(P, dst), "w") as f:
            if header:
                f.write(header)
            f.write(open(s).read())


def traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the captured kernels -> profiles/traffic.json (read by bench.py)."""
    out = {}
    for name, cls in (("prof_tc2_update", "gj_update"), ("prof_tc2_sweep", "sweep_gemm"), ("prof_gradient", "gradient"),
                      ("prof_assemble", "assemble"), ("prof_tc2_rowpanel", "gj_rowpanel")):
        rep = os.path.join(O, f"{name}_{R}.ncu-rep")
        if not os.path.exists(rep):
            continue
        rows = list(csv.reader(io.StringIO(subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout)))
        if len(rows) < 3:
            continue
        H = rows[0]
        try:
            ir, iw = H.index("dram__bytes_read.sum"), H.index("dram__bytes_write.sum")
        except ValueError:
            continue
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        vals = []
        for r in rows[2:]:
            vals.append(float(r[ir].replace(",", "")) * scale.get(rows[1][ir], 1.0) + float(r[iw].replace(",", "")) * scale.get(rows[1][iw], 1.0))
        out[cls] = max(vals)  # the fullest of the captured launches
    if out:
        json.dump(out, open(os.path.join(P, "traffic.json"), "w"), indent=1)


launches()
traffic()
ncu_rep("prof_tc2_sweep", "tc2_sweep_gemm_kernel at the benchmark configuration (512^2, 256 sources, 16 frequencies)")
ncu_rep("prof_tc2_update", "tc2_gj_update_kernel (rank-64 Gauss-Jordan update + look-ahead pivot CTAs) at the benchmark configuration")
ncu_rep("prof_tc2_rowpanel", "tc2_gj_rowpanel_kernel at the benchmark configuration")
ncu_rep("prof_gradient", "gradient_kernel at the benchmark configuration")
ncu_rep("prof_assemble", "assemble_kernel at the benchmark configuration")
copy(f"exp_update_trace_{R}.log", f"exp_update_trace_{R}.txt",
     "# python tools/exp_update_trace.py on one B200: every CTA of one rank-64 update launch (512^2, 16 frequencies), ns since the first CTA entered\n")
copy(f"exp_update_trace_f2_{R}.log", f"exp_update_trace_f2_{R}.txt",
     "# python tools/exp_update_trace.py --nfreq 2 on one B200: one rank-64 update launch with 2 frequencies (4 chains) on the GPU\n")
copy(f"exp_accuracy_{R}.log", f"exp_accuracy_{R}.txt",
     "# python tools/exp_accuracy.py 512 8 on one B200: interior wavefield error vs the complex128 oracle under environment toggles\n")
copy(f"pytest_gpu_{R}.log", f"pytest_gpu_{R}.txt", "# python -m pytest tests -m gpu -q -s on one B200\n")
copy(f"smoke_{R}.log", f"smoke_{R}.txt")
copy(f"gpu_{R}.txt", f"gpu_{R}.txt")
for tag in ("bench", "bench_final", "bench_simt", "bench_ref", "bench_cfg2", "bench_cfg4", "bench_cfg4_c128", "bench_f2", "bench_f4", "bench_f8", "bench_c128", "bench_g1",
            "bench_2gpu_strong", "bench_2gpu_cfg4", "bench_4gpu_strong", "bench_8gpu_strong", "cfg5_8gpu", "cpu_baseline"):
    s = os.path.join(O, f"{tag}_{R}.json")
    if os.path.exists(s):
        try:
            line = [l for l in open(s).read().splitlines() if l.startswith("{")][-1]
            json.dump(json.loads(line), open(os.path.join(P, f"{tag}_{R}.json"), "w"), indent=1)
        except Exception as e:  # noqa: BLE001
            print(tag, "unreadable:", e)
print(sorted(os.listdir(P)))
