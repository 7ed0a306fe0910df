"""Cost of the lossy line search (ust_ncg_linesearch_lossy) and the lossy Gauss-Newton product (ust_fwi_gn_hvp_lossy), each
beside its lossless counterpart and both against one (loss, grad) evaluation, on one GPU.

Workloads: BASELINE configs[2] (512 x 512, 256-element ring, 16 frequencies, complex64) and configs[3] (1024 x 1024,
1024-element ring, 1 frequency), built exactly as bench.py builds them (bench.workload / bench.Harness).  Every graph is
captured in a warm-up, then the six calls -- lossless evaluation, line search, product; lossy evaluation, line search,
product -- run in that order 5 times, timed with CUDA events around each call, and the medians are reported.  The plan's
device bytes are read before and after the timed calls (the line search and the product allocate nothing) and compared with
the bytes the plan would have without the two buffers this change adds (vk_in, hv_kappa_out: Ny*Nx reals each).  Card name,
power limit and maximum SM clock come from a read-only nvidia-smi query in the same run.

    python tools/bench_joint_gn.py --out DIR [--configs configs2,configs3]     -> DIR/bench_joint_gn.json
"""
import argparse
import json
import os
import statistics
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
from bench_gn import SHAPES, card  # noqa: E402


def run_shape(torch, key, dtype, reps):
    from waveforminversionust_b200 import geometry as G
    s = SHAPES[key]
    a = types.SimpleNamespace(n=s["n"], nsrc=s["nsrc"], nfreq=s["nfreq"], scaling="strong", impl="ours", dtype=dtype,
                              engine="auto", shard=s["shard"], groups=0)
    geom, freqs, vel_true, vel0 = bench.workload(a)
    h = bench.Harness(a, torch, None, geom, freqs, vel_true, vel0, 0, 1, 0)
    eng, plan = h.eng, h.eng.plan
    vs = torch.as_tensor((1.0 / vel_true - 1.0 / vel0).astype(plan.real)).to(h.dv)
    kappa = torch.as_tensor(G.attenuation_blob_model(geom, alpha0=0.25, dalpha=0.5).astype(plan.real)).to(h.dv)
    vk = torch.as_tensor(G.attenuation_blob_model(geom, alpha0=0.0, dalpha=0.25, seed=7).astype(plan.real)).to(h.dv)
    calls = {"evaluation": h.step_dev, "linesearch": lambda: plan.ncg_linesearch(vs), "product": lambda: plan.gn_hvp(vs),
             "lossy_evaluation": lambda: eng.loss_grad_lossy_device(h.slow0, kappa, h.rec_local),
             "lossy_linesearch": lambda: plan.ncg_linesearch_lossy(vs, vk), "lossy_product": lambda: plan.gn_hvp_lossy(vs, vk)}

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for _ in range(2):  # warm-up: all six graphs captured, modules loaded
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    bytes_before = plan.device_bytes
    t = {k: [] for k in calls}
    for _ in range(reps):
        for k, fn in calls.items():
            t[k].append(timed(fn)[0])
    bytes_after = plan.device_bytes
    prof = {}
    plan.profile(True)
    for k in ("product", "lossy_product"):
        calls["evaluation" if k == "product" else "lossy_evaluation"]()
        plan.get_profile()
        calls[k]()
        prof[k] = plan.get_profile()
    plan.profile(False)
    med = {k: statistics.median(v) for k, v in t.items()}
    nz = lambda p: {c: [round(v[0], 3), v[1]] for c, v in p.items() if v[1]}
    new_bytes = 2 * geom.Nx * geom.Ny * np.dtype(plan.real).itemsize
    out = {"config": s["name"], "workload": f"{s['n']}x{s['n']} grid, {geom.tx_include.size} transmitters, {len(freqs)} frequencies, {dtype}",
           "ms": t, "median_ms": med,
           "lossy_over_lossless": {k: med["lossy_" + k] / med[k] for k in ("evaluation", "linesearch", "product")},
           "over_evaluation": {k: med[k] / med["evaluation"] for k in ("linesearch", "product")},
           "lossy_over_lossy_evaluation": {k: med["lossy_" + k] / med["lossy_evaluation"] for k in ("linesearch", "product")},
           "gradient_kernel_ms": {k: round(prof[k]["gradient"][0], 4) for k in prof},
           "device_bytes_before": bytes_before, "device_bytes_after": bytes_after,
           "device_bytes_added_by_vk_in_and_hv_kappa_out": new_bytes,
           "profile_ms_launches": {k: nz(v) for k, v in prof.items()}}
    print(f"{s['name']}: " + ", ".join(f"{k} {v:.1f} ms" for k, v in med.items()) +
          "; lossy/lossless " + ", ".join(f"{k} {v:.3f}" for k, v in out["lossy_over_lossless"].items()), flush=True)
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
        raise SystemExit("bench_joint_gn.py needs a CUDA device")
    import __graft_entry__  # noqa: F401  (puts the repository on sys.path)
    res = {"gpu": card(), "dtype": a.dtype,
           "timing": f"CUDA events around each call, median of {a.reps}; lossless and lossy evaluation, line search and product alternating",
           "shapes": [run_shape(torch, k, a.dtype, a.reps) for k in a.configs.split(",")]}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_joint_gn.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu",)}))


if __name__ == "__main__":
    main()
