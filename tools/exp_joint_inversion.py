"""Sound-speed-only against joint sound-speed + attenuation L-BFGS on lossy data.

256 x 256 grid, 256-element ring, 4 frequencies of the band bench.py uses at this grid; blob truths for the sound speed
(geometry.blob_model) and the attenuation (geometry.attenuation_blob_model: ~0.5 dB/(cm MHz) blobs); observed data from the
complex128 lossy forward model on the GPU.  Both runs start at c = 1480 m/s (and kappa = 0) and get the same budget of
objective evaluations (one factorisation each, complex64; gtol = 0, so that only the budget or L-BFGS-B's own line-search /
relative-reduction tests end a run):
  (a) run_lbfgs_fwi on the slowness alone (the lossless model fitted to lossy data);
  (b) run_lbfgs_joint_fwi on [slowness, kappa] with kappa >= 0.
Reported per run: the sound-speed RMS error (m/s) and the attenuation RMS error (dB/(cm MHz)) inside the ring, and the loss,
at the evaluation with the lowest loss within the budget, plus the error trace.

    python tools/exp_joint_inversion.py --out DIR [--evals 40]     -> DIR/exp_joint_inversion.txt
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


class Budget(Exception):
    pass


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--evals", type=int, default=40)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("exp_joint_inversion.py needs a CUDA device")
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import geometry as G
    n = a.n
    geom = G.ring_geometry(n, 256)
    f_hi = G.frequency_for_grid(n)
    freqs = np.linspace(f_hi * 300.0 / 596.0, f_hi, 4)
    vel_true = G.blob_model(geom)
    kappa_true = G.attenuation_blob_model(geom, dalpha=0.5)
    amp = G.source_amplitudes(geom.tx_include.size)
    src = geom.dense_src(np.complex128)
    rec = np.stack([w.solve_helmholtz(geom.xi, geom.yi, vel_true, src, f, geom.a0, geom.L_PML, False, dtype="c128", kappa=kappa_true)
                    [geom.y_idx, geom.x_idx, :].T * amp[:, None] for f in freqs])
    w.clear_plans()
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64))
    inside = X ** 2 + Y ** 2 < 0.1 ** 2  # inside the 110 mm ring, clear of the elements
    c_err = lambda c: float(np.sqrt(np.mean((c[inside] - vel_true[inside]) ** 2)))
    k_err = lambda k: float(np.sqrt(np.mean(G.kappa_to_db_cm_mhz(k[inside] - kappa_true[inside]) ** 2)))
    fargs = (geom.xi, geom.yi, rec, geom.dense_src(), freqs, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab,
             geom.mask_indices, geom.num_elements)
    dargs = (geom.xi, geom.yi, None, None, geom.tx_include, geom.ind_matlab, 1480.0, freqs, geom.a0, geom.L_PML, geom.mask_indices)
    lines = [f"# tools/exp_joint_inversion.py: {n}x{n} grid, 256-element ring, frequencies {[round(f / 1e3, 1) for f in freqs]} kHz, "
             f"complex64, budget {a.evals} evaluations per run", f"# card: {card()}",
             f"# truth: sound speed {vel_true[inside].min():.1f}..{vel_true[inside].max():.1f} m/s, attenuation "
             f"{G.kappa_to_db_cm_mhz(kappa_true[inside]).min():.3f}..{G.kappa_to_db_cm_mhz(kappa_true[inside]).max():.3f} dB/(cm MHz); "
             f"errors are RMS over the disc r < 100 mm",
             f"# start: c = 1480 m/s (error {c_err(np.full((n, n), 1480.0)):.3f} m/s), kappa = 0 (error {k_err(np.zeros((n, n))):.4f} dB/(cm MHz))"]
    results = {}
    for name in ("a_sound_speed_only", "b_joint"):
        trace = []

        def record(loss, c, k):
            trace.append((float(loss), c_err(c), k_err(k)))
            if len(trace) >= a.evals:
                raise Budget()

        if name == "a_sound_speed_only":
            def loss_grad(slow):
                loss, grad = w.fwi_loss_function(slow.astype(np.float32), *fargs, dtype="c64")
                record(loss, 1.0 / slow, np.zeros((n, n)))
                return loss, grad
            run = lambda: w.run_lbfgs_fwi(*dargs, maxiter=10 * a.evals, tol=0.0, dtype="c64", loss_grad=loss_grad)
        else:
            def loss_grad(params):
                loss, grad = w.fwi_joint_loss_function(params.astype(np.float32), *fargs, dtype="c64")
                record(loss, 1.0 / params[0], params[1])
                return loss, grad
            run = lambda: w.run_lbfgs_joint_fwi(*dargs, kappa_init=0.0, maxiter=10 * a.evals, tol=0.0, dtype="c64", loss_grad=loss_grad)
        t0 = time.perf_counter()
        try:
            run()
        except Budget:
            pass
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = min(range(len(trace)), key=lambda i: trace[i][0])
        results[name] = trace[best]
        lines.append(f"{name}: {len(trace)} evaluations in {dt:.2f} s; lowest loss at evaluation {best}: loss {trace[best][0]:.6e}, "
                     f"c RMS error {trace[best][1]:.3f} m/s, attenuation RMS error {trace[best][2]:.4f} dB/(cm MHz)")
        lines.append("  trace (evaluation: loss, c error m/s, attenuation error dB/(cm MHz)): " +
                     "; ".join(f"{i}: {l:.4e}, {ce:.3f}, {ke:.4f}" for i, (l, ce, ke) in enumerate(trace)))
        w.clear_plans()
    ra, rb = results["a_sound_speed_only"], results["b_joint"]
    lines.append(f"joint vs sound-speed-only at equal budget: c RMS error {rb[1]:.3f} vs {ra[1]:.3f} m/s, attenuation RMS error "
                 f"{rb[2]:.4f} vs {ra[2]:.4f} dB/(cm MHz), loss {rb[0]:.4e} vs {ra[0]:.4e}")
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "exp_joint_inversion.txt"), "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
