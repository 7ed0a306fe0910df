"""Cost of one lossy (loss, grad_s, grad_kappa) evaluation (ust_fwi_loss_grad_lossy) against one lossless (loss, grad)
evaluation (ust_fwi_loss_grad) on one GPU.

Workloads: BASELINE configs[2] (512 x 512, 256-element ring, 16 frequencies, complex64) and configs[3] (1024 x 1024,
1024-element ring, 1 frequency), built exactly as bench.py builds them (bench.workload / bench.Harness); the lossy
evaluation adds an attenuation map of ~0.5 dB/(cm MHz) blobs on a 0.25 dB/(cm MHz) background.  Both evaluations are warmed
up (graph capture of both keys), then 5 of each are timed alternately with CUDA events around each call and the medians
reported.  Separate profiled runs (plan.profile: per-launch events, no graph) give the per-class split; the assembly and
gradient classes, the only ones whose kernels differ, are profiled 3 times each.  The plan's device bytes are read before
and after.  Card name, power limit and maximum SM clock come from a read-only nvidia-smi query.

    python tools/bench_joint.py --out DIR [--configs configs2,configs3]     -> DIR/bench_joint.json
"""
import argparse
import json
import os
import statistics
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

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
    kappa = torch.as_tensor(G.attenuation_blob_model(geom, alpha0=0.25, dalpha=0.5).astype(plan.real)).to(h.dv)
    lossy = lambda: eng.loss_grad_lossy_device(h.slow0, kappa, h.rec_local)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for _ in range(2):  # warm-up: both graphs captured, modules loaded
        h.step_dev()
        lossy()
    torch.cuda.synchronize()
    bytes_before = plan.device_bytes
    t_ll, t_ly = [], []
    for _ in range(reps):
        t, (loss0, _) = timed(h.step_dev)
        t_ll.append(t)
        t, (loss1, grad) = timed(lossy)
        t_ly.append(t)
    bytes_after = plan.device_bytes
    gk_max = float(torch.abs(grad[1]).max())
    prof = {"lossless": [], "lossy": []}
    plan.profile(True)
    for _ in range(3):
        for name, fn in (("lossless", h.step_dev), ("lossy", lossy)):
            fn()
            prof[name].append(plan.get_profile())
    plan.profile(False)
    nz = lambda p: {k: [round(v[0], 3), v[1]] for k, v in p.items() if v[1]}
    cls = lambda name, c: [round(p[c][0], 4) for p in prof[name]]
    ml, my = statistics.median(t_ll), statistics.median(t_ly)
    out = {"config": s["name"], "workload": f"{s['n']}x{s['n']} grid, {geom.tx_include.size} transmitters, {len(freqs)} frequencies, {dtype}",
           "lossless_ms": t_ll, "lossy_ms": t_ly, "lossless_median_ms": ml, "lossy_median_ms": my, "lossy_over_lossless": my / ml,
           "assemble_ms_lossless": cls("lossless", "assemble"), "assemble_ms_lossy": cls("lossy", "assemble"),
           "gradient_ms_lossless": cls("lossless", "gradient"), "gradient_ms_lossy": cls("lossy", "gradient"),
           "loss_lossless": float(loss0), "loss_lossy": float(loss1), "grad_kappa_max_abs": gk_max,
           "device_bytes_before": bytes_before, "device_bytes_after": bytes_after,
           "profile_lossless_ms_launches": nz(prof["lossless"][0]), "profile_lossy_ms_launches": nz(prof["lossy"][0])}
    print(f"{s['name']}: lossless {ml:.1f} ms, lossy {my:.1f} ms, ratio {my / ml:.4f}; gradient kernel {out['gradient_ms_lossless']} vs "
          f"{out['gradient_ms_lossy']} ms; assembly {out['assemble_ms_lossless']} vs {out['assemble_ms_lossy']} ms", flush=True)
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
        raise SystemExit("bench_joint.py needs a CUDA device")
    res = {"gpu": card(), "dtype": a.dtype,
           "timing": f"CUDA events around each call, median of {a.reps}, lossless and lossy evaluations alternating",
           "shapes": [run_shape(torch, k, a.dtype, a.reps) for k in a.configs.split(",")]}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_joint.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"gpu": res["gpu"]}))


if __name__ == "__main__":
    main()
