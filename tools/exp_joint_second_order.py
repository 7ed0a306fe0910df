"""Joint sound-speed + attenuation inversion with second-order information: joint NCG, joint Gauss-Newton and joint L-BFGS at
equal factorisation budgets.

The case of tools/exp_joint_inversion.py: 256 x 256 grid, 256-element ring, 4 frequencies of the band bench.py uses at this
grid, blob truths for both maps, observed data from the complex128 lossy forward model on the GPU, start c = 1480 m/s and
kappa = 0, complex64, each block scaled as in run_lbfgs_joint_fwi (kappa_scale = 0.5 dB/(cm MHz), pert_scale = 1e-2).  Each run
gets the same budget of objective evaluations (one factorisation each):
  (a) nonlinear_conjugate_gradient_joint: one evaluation and one lossy line search per iteration;
  (b) gauss_newton_joint_fwi with cg_iters = 4: evaluations for the trials, lossy products for the CG steps;
  (c) run_lbfgs_joint_fwi (gtol = 0, so that only the budget or L-BFGS-B's own tests end it).
Reported per run, per evaluation: wall time since the start (with a device synchronise), loss, sound-speed RMS error (m/s) and
attenuation RMS error (dB/(cm MHz)) over the disc r < 100 mm, and the products / line searches so far.

    python tools/exp_joint_second_order.py --out DIR [--evals 40]     -> DIR/exp_joint_second_order.txt
"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from exp_joint_inversion import Budget, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--evals", type=int, default=40)
    ap.add_argument("--cg-iters", type=int, default=4)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("exp_joint_second_order.py needs a CUDA device")
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import api
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
    src1 = w.OneHotSources(geom.src_lin, (n, n, geom.tx_include.size))  # sparse one-hot sources: no dense scan per call
    dargs = (geom.xi, geom.yi, geom.num_elements, rec, src1, geom.tx_include, geom.ind_matlab, 1480.0, freqs)
    tail = (geom.a0, geom.L_PML, geom.mask_indices)
    lines = [f"# tools/exp_joint_second_order.py: {n}x{n} grid, 256-element ring, frequencies {[round(f / 1e3, 1) for f in freqs]} kHz, "
             f"complex64, budget {a.evals} evaluations (factorisations) per run, Gauss-Newton cg_iters = {a.cg_iters}",
             f"# card: {card()}",
             f"# truth: sound speed {vel_true[inside].min():.1f}..{vel_true[inside].max():.1f} m/s, attenuation "
             f"{G.kappa_to_db_cm_mhz(kappa_true[inside]).min():.3f}..{G.kappa_to_db_cm_mhz(kappa_true[inside]).max():.3f} dB/(cm MHz); "
             f"errors are RMS over the disc r < 100 mm",
             f"# start: c = 1480 m/s (error {c_err(np.full((n, n), 1480.0)):.3f} m/s), kappa = 0 (error {k_err(np.zeros((n, n))):.4f} dB/(cm MHz))"]
    results = {}
    for name in ("a_ncg", "b_gauss_newton", "c_lbfgs"):
        lg0, ls0, hvp0 = api._gpu_callables(True, *dargs[:7], freqs, *tail, "c64", None, "python", 0, "auto")
        trace, count = [], {"products": 0, "linesearches": 0}
        t0 = [0.0]

        def record(loss, x):
            torch.cuda.synchronize()
            trace.append((time.perf_counter() - t0[0], float(loss), c_err(1.0 / x[0]), k_err(x[1]), count["products"],
                          count["linesearches"]))

        def loss_grad(x):
            if len(trace) >= a.evals:
                raise Budget()
            loss, grad = lg0(x)
            record(loss, x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x))
            return loss, grad

        def linesearch(sd):
            count["linesearches"] += 1
            return ls0(sd)

        def hvp(v):
            count["products"] += 1
            return hvp0(v)

        def lbfgs_loss_grad(params):
            loss, grad = loss_grad(torch.as_tensor(params))
            return loss, grad.double().cpu().numpy()

        kw = dict(kappa_init=0.0, dtype="c64")
        if name == "a_ncg":
            run = lambda: w.nonlinear_conjugate_gradient_joint(*dargs, a.evals, *tail, loss_grad=loss_grad, linesearch=linesearch, **kw)
        elif name == "b_gauss_newton":
            run = lambda: w.gauss_newton_joint_fwi(*dargs, 10 * a.evals, *tail, cg_iters=a.cg_iters, loss_grad=loss_grad, hvp=hvp, **kw)
        else:
            run = lambda: w.run_lbfgs_joint_fwi(geom.xi, geom.yi, None, None, geom.tx_include, geom.ind_matlab, 1480.0, freqs, *tail,
                                                maxiter=10 * a.evals, tol=0.0, loss_grad=lbfgs_loss_grad, **kw)
        lg0(torch.as_tensor(np.stack([np.full((n, n), 1 / 1480.0), np.zeros((n, n))])))  # warm-up: plan, graphs, modules
        if name != "c_lbfgs":
            (ls0 if name == "a_ncg" else hvp0)(torch.zeros((2, n, n), dtype=torch.float64) + 1e-9)
        torch.cuda.synchronize()
        t0[0] = time.perf_counter()
        try:
            run()
        except Budget:
            pass
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0[0]
        best = min(range(len(trace)), key=lambda i: trace[i][1])
        results[name] = trace
        tb = trace[best]
        lines.append(f"{name}: {len(trace)} evaluations, {count['products']} products, {count['linesearches']} line searches in {dt:.2f} s; "
                     f"lowest loss at evaluation {best} ({tb[0]:.2f} s): loss {tb[1]:.6e}, c RMS error {tb[2]:.3f} m/s, attenuation RMS "
                     f"error {tb[3]:.4f} dB/(cm MHz); lowest attenuation error {min(t[3] for t in trace):.4f} at evaluation "
                     f"{min(range(len(trace)), key=lambda i: trace[i][3])}")
        lines.append("  trace (evaluation: s, loss, c error m/s, attenuation error dB/(cm MHz), products, line searches): " +
                     "; ".join(f"{i}: {t:.2f}, {l:.4e}, {ce:.3f}, {ke:.4f}, {p}, {q}" for i, (t, l, ce, ke, p, q) in enumerate(trace)))
        w.clear_plans()
    for k in (10, 20, a.evals):
        row = []
        for name, tr in results.items():
            if len(tr) >= k:
                b = min(tr[:k], key=lambda t: t[1])
                row.append(f"{name} loss {b[1]:.4e} c {b[2]:.3f} m/s att {b[3]:.4f} dB/(cm MHz) ({tr[k - 1][0]:.2f} s)")
        lines.append(f"after {k} evaluations (lowest-loss point so far): " + " | ".join(row))
    tmin = min(tr[-1][0] for tr in results.values())
    row = []
    for name, tr in results.items():
        b = min((t for t in tr if t[0] <= tmin), key=lambda t: t[1])
        row.append(f"{name} loss {b[1]:.4e} c {b[2]:.3f} m/s att {b[3]:.4f} dB/(cm MHz)")
    lines.append(f"within {tmin:.2f} s (the shortest run's wall time, lowest-loss point so far): " + " | ".join(row))
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "exp_joint_second_order.txt"), "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
