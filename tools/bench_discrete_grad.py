"""Cost of the discrete gradient mode (ust_plan_set_gradient(UST_GRAD_DISCRETE), DESIGN.md section 7f) against the reference
mode on one GPU: the (loss, grad) evaluation, the NCG line search and the Gauss-Newton product.

Workloads: BASELINE configs[2] (512 x 512, 256-element ring, 16 frequencies) and configs[3] (1024 x 1024, 1024-element ring,
1 frequency), complex64, built exactly as bench.py builds them (bench.workload / bench.Harness).  Every call of both modes is
warmed up (graph capture), then 5 rounds time evaluation, line search and product of the reference mode and of the discrete
mode alternately, with CUDA events around each call; medians are reported.  Per-class kernel times come from separate
profiled calls (plan.profile): the gradient kernel is the "gradient" class of an evaluation, the perturbation right-hand side
the "receiver" class of a discrete-mode line search (its only member there; the reference right-hand side is not profiled).
Rates use the algorithmic bytes of the reference kernels: gradient 2 complex reads per (pixel, source, frequency),
right-hand side one complex read and one write.  The copy bandwidth is a device-to-device copy of 4 GiB (read + write
counted), timed the same way.  Card name, power limit and maximum SM clock come from a read-only nvidia-smi query in the same
call.

    python tools/bench_discrete_grad.py --out DIR [--configs configs2,configs3]     -> DIR/bench_discrete_grad.json
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

import bench  # noqa: E402

SHAPES = {"configs2": dict(n=512, nsrc=256, nfreq=16, shard="freq", name="configs[2]"),
          "configs3": dict(n=1024, nsrc=1024, nfreq=1, shard="source", name="configs[3]")}
MODES = ("reference", "discrete")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def timed(torch, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def copy_bandwidth(torch, reps):
    """Bytes per second of a device-to-device copy of 4 GiB (read + write), median of ``reps``."""
    a = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    ts = [timed(torch, lambda: b.copy_(a))[0] for _ in range(reps)]
    del a, b
    return 2.0 * (1 << 32) / (statistics.median(ts) * 1e-3)


def run_shape(torch, key, reps, copy_bw):
    s = SHAPES[key]
    a = types.SimpleNamespace(n=s["n"], nsrc=s["nsrc"], nfreq=s["nfreq"], scaling="strong", impl="ours", dtype="c64",
                              engine="auto", shard=s["shard"], groups=0)
    geom, freqs, vel_true, vel0 = bench.workload(a)
    h = bench.Harness(a, torch, None, geom, freqs, vel_true, vel0, 0, 1, 0)
    plan = h.eng.plan
    v = torch.as_tensor((1.0 / vel_true - 1.0 / vel0).astype(plan.real)).to(h.dv)
    calls = {"evaluation": h.step_dev, "linesearch": lambda: plan.ncg_linesearch(v), "product": lambda: plan.gn_hvp(v)}
    for _ in range(2):  # warm-up: the graphs of both modes captured, modules loaded
        for mode in MODES:
            plan.set_gradient(mode)
            for fn in calls.values():
                fn()
    torch.cuda.synchronize()
    bytes_before = plan.device_bytes
    t = {m: {c: [] for c in calls} for m in MODES}
    for _ in range(reps):
        for mode in MODES:
            plan.set_gradient(mode)
            for c, fn in calls.items():
                t[mode][c].append(timed(torch, fn)[0])
    prof = {}
    for mode in MODES:
        plan.set_gradient(mode)
        plan.profile(True)
        prof[mode] = {}
        for c, fn in calls.items():
            fn()
            torch.cuda.synchronize()
            prof[mode][c] = {k: [round(x[0], 4), x[1]] for k, x in plan.get_profile().items() if x[1]}
        plan.profile(False)
    plan.set_gradient("reference")
    bytes_after = plan.device_bytes
    N, nt, nf = geom.Nx * geom.Ny, geom.tx_include.size, len(h.eng.local_freqs)
    grad_bytes = 16.0 * N * nt * nf  # reference gradient kernel: u and lambda, 8 B each per (pixel, source, frequency)
    rhs_bytes = 16.0 * N * nt * nf   # reference right-hand side: read u, write the right-hand side
    med = {m: {c: statistics.median(x) for c, x in t[m].items()} for m in MODES}
    kern = {}
    for m in MODES:
        g_ms = prof[m]["evaluation"]["gradient"][0]
        kern[m] = {"gradient_ms": g_ms, "gradient_bytes_per_s": grad_bytes / (g_ms * 1e-3),
                   "gradient_over_copy_bw": grad_bytes / (g_ms * 1e-3) / copy_bw}
    r_ms = prof["discrete"]["linesearch"]["receiver"][0]
    kern["discrete"].update(rhs_ms=r_ms, rhs_bytes_per_s=rhs_bytes / (r_ms * 1e-3), rhs_over_copy_bw=rhs_bytes / (r_ms * 1e-3) / copy_bw)
    out = {"config": s["name"], "workload": f"{s['n']}x{s['n']} grid, {nt} transmitters, {nf} frequencies, c64",
           "call_ms": t, "call_median_ms": med,
           "discrete_over_reference": {c: med["discrete"][c] / med["reference"][c] for c in calls},
           "kernels": kern, "gradient_kernel_discrete_over_reference": kern["discrete"]["gradient_ms"] / kern["reference"]["gradient_ms"],
           "algorithmic_bytes": {"gradient": grad_bytes, "rhs": rhs_bytes},
           "device_bytes_before": bytes_before, "device_bytes_after": bytes_after, "profile_ms_launches": prof}
    print(f"{s['name']}: " + ", ".join(f"{c} {med['reference'][c]:.2f} -> {med['discrete'][c]:.2f} ms" for c in calls)
          + f"; gradient kernel {kern['reference']['gradient_ms']:.3f} -> {kern['discrete']['gradient_ms']:.3f} ms"
          + f", discrete rhs kernel {kern['discrete']['rhs_ms']:.3f} ms", flush=True)
    h.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--configs", default="configs2,configs3")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_discrete_grad.py needs a CUDA device")
    import __graft_entry__  # noqa: F401  (puts the repository on sys.path)
    bw = copy_bandwidth(torch, a.reps)
    res = {"gpu": card(), "dtype": "c64", "copy_bandwidth_bytes_per_s": bw,
           "timing": f"CUDA events around each call, median of {a.reps}, reference and discrete modes alternating",
           "shapes": [run_shape(torch, k, a.reps, bw) for k in a.configs.split(",")]}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_discrete_grad.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"gpu": res["gpu"], "copy_bandwidth_TB_s": bw / 1e12}))


if __name__ == "__main__":
    main()
