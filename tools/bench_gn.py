"""Cost of one Gauss-Newton product (ust_fwi_gn_hvp) against one (loss, grad) evaluation on one GPU.

Workloads: BASELINE configs[2] (512 x 512, 256-element ring, 16 frequencies, complex64) and configs[3] (1024 x 1024,
1024-element ring, 1 frequency), built exactly as bench.py builds them (bench.workload / bench.Harness).  Both shapes are
warmed up (graph capture of the evaluation and of the product), then 5 evaluations and 5 products are timed alternately
with CUDA events around each call and the medians reported; one extra product and one extra evaluation run under
plan.profile for the per-class split.  The plan's device bytes are read before and after the products (the product
allocates nothing).  Card name, power limit and maximum SM clock come from a read-only nvidia-smi query.

    python tools/bench_gn.py --out DIR [--configs configs2,configs3]     -> DIR/bench_gn.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402

SHAPES = {"configs2": dict(n=512, nsrc=256, nfreq=16, shard="freq", name="configs[2]"),
          "configs3": dict(n=1024, nsrc=1024, nfreq=1, shard="source", name="configs[3]")}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def run_shape(torch, key, dtype, reps):
    s = SHAPES[key]
    a = types.SimpleNamespace(n=s["n"], nsrc=s["nsrc"], nfreq=s["nfreq"], scaling="strong", impl="ours", dtype=dtype,
                              engine="auto", shard=s["shard"], groups=0)
    geom, freqs, vel_true, vel0 = bench.workload(a)
    h = bench.Harness(a, torch, None, geom, freqs, vel_true, vel0, 0, 1, 0)
    plan = h.eng.plan
    v = torch.as_tensor((1.0 / vel_true - 1.0 / vel0).astype(plan.real)).to(h.dv)
    ev = lambda: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def timed(fn):
        e0, e1 = ev()
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for _ in range(2):  # warm-up: both graphs captured, modules loaded
        h.step_dev()
        plan.gn_hvp(v)
    torch.cuda.synchronize()
    bytes_before = plan.device_bytes
    t_eval, t_prod = [], []
    for _ in range(reps):
        t, (loss, grad) = timed(h.step_dev)
        t_eval.append(t)
        t, (hv, jv2) = timed(lambda: plan.gn_hvp(v))
        t_prod.append(t)
    bytes_after = plan.device_bytes
    vhv = float(torch.sum(v.double() * hv.double()))
    plan.profile(True)
    plan.gn_hvp(v)
    prof_prod = plan.get_profile()
    h.step_dev()
    prof_eval = plan.get_profile()
    plan.profile(False)
    me, mp = statistics.median(t_eval), statistics.median(t_prod)
    nz = lambda p: {k: [round(v[0], 3), v[1]] for k, v in p.items() if v[1]}
    out = {"config": s["name"], "workload": f"{s['n']}x{s['n']} grid, {geom.tx_include.size} transmitters, {len(freqs)} frequencies, {dtype}",
           "evaluation_ms": t_eval, "product_ms": t_prod, "evaluation_median_ms": me, "product_median_ms": mp,
           "product_over_evaluation": mp / me, "jv2": float(jv2[0]), "v_dot_hv": vhv, "loss": float(loss),
           "device_bytes_before": bytes_before, "device_bytes_after": bytes_after,
           "profile_product_ms_launches": nz(prof_prod), "profile_evaluation_ms_launches": nz(prof_eval)}
    print(f"{s['name']}: evaluation {me:.1f} ms, product {mp:.1f} ms, ratio {mp / me:.3f}", flush=True)
    h.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default="configs2,configs3")
    ap.add_argument("--dtype", default="c64", choices=["c64", "c128"])
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_gn.py needs a CUDA device")
    import __graft_entry__  # noqa: F401  (puts the repository on sys.path)
    res = {"gpu": card(), "dtype": a.dtype, "timing": f"CUDA events around each call, median of {a.reps}, evaluations and products alternating",
           "shapes": [run_shape(torch, k, a.dtype, a.reps) for k in a.configs.split(",")]}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_gn.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu",)}))


if __name__ == "__main__":
    main()
