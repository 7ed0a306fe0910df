#!/usr/bin/env python
"""In-situ phase timestamps of one rank-64 Gauss-Jordan update launch at the benchmark size (512^2, 16 frequencies):
every CTA of the launch for (step, k) dumps the 16 trace slots of tools/exp_tc2_trace.py, relative to the first CTA
entering the kernel.  Prints per-wave summaries.

    UST_TC2_TRACE_UPDATE=100,3 python tools/exp_update_trace.py
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if "UST_TC2_TRACE_UPDATE" not in os.environ:
    os.environ["UST_TC2_TRACE_UPDATE"] = "100,3"
env = dict(os.environ, UST_NO_GRAPHS="1")
r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline", "--groups", "1"] + sys.argv[1:],
                   env=env, capture_output=True, text=True)  # extra arguments go to bench.py (e.g. --nfreq 2)
rows = []
for line in r.stderr.splitlines():
    if line.startswith("upd cta"):
        parts = line.replace(":", "").split()
        rows.append((int(parts[2]), int(parts[4]), [int(x) for x in parts[5:]]))
if not rows:
    print(r.stderr[-2000:])
    raise SystemExit("no trace lines")
# keep only the first dump (the factor of the first step)
seen, first = set(), []
for b, sm, t in rows:
    if b in seen:
        break
    seen.add(b)
    first.append((b, sm, t))
first.sort(key=lambda x: x[2][0])
names = ["enter", "setup", "tma0", "land0", "mma0", "d1seen", "d1back", "mmasees", "lastback", "lastissue", "d2done", "staged", "written", "emitted", "freed", "stagedB", "pivdone"]
print("ctas", len(first), "kernel span", max(max(t[:17]) for _, _, t in first), "ns")
print("%5s %4s " % ("cta", "sm") + " ".join("%8s" % n for n in names))
for b, sm, t in first[:: max(1, len(first) // 48)]:
    print("%5d %4d " % (b, sm) + " ".join("%8d" % x for x in t[:17]))
piv = [r_ for r_ in first if r_[0] >= 1000]
if piv:
    print("look-ahead pivot CTAs (rows 1000 + chain): formed = 'staged', inversion done = 'pivdone'")
    for b, sm, t in piv:
        print("%5d %4d " % (b, sm) + " ".join("%8d" % x for x in t[:17]))
        if len(t) > 17:  # blocked inversion: start, then (diagonal block inverted, panels formed, update applied) x 4
            st = t[17:]
            print("       inversion phases [ns]: " + " | ".join("inv16 %d panels %d update %d" % (st[1 + 3 * q] - st[3 * q], st[2 + 3 * q] - st[1 + 3 * q], st[3 + 3 * q] - st[2 + 3 * q]) for q in range(4)))
import statistics
for i, n in enumerate(names[1:], 1):
    d = [t[i] - t[0] for _, _, t in first if t[i] > 0]
    if d:
        print("%-10s since enter: median %7d  p10 %7d  p90 %7d" % (n, statistics.median(d), sorted(d)[len(d) // 10], sorted(d)[9 * len(d) // 10]))
