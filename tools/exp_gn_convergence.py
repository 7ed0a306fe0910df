"""NCG, L-BFGS and truncated Gauss-Newton on one small inversion: loss and model error against the truth as a function of
factorisations (one per (loss, grad) evaluation; Gauss-Newton products need none) and of wall time.

256 x 256 grid, 256-element ring (all elements transmit), 4 frequencies in the lower half of the grid's band, complex64,
truth = geometry.blob_model, start = its 1500 m/s background.  Observed data come from this solver at the truth.
NCG is api.nonlinear_conjugate_gradient (re-run for each iteration count, since it returns the final model only);
L-BFGS (api.run_lbfgs_fwi) and Gauss-Newton (api.gauss_newton_fwi) get recording wrappers of the public
fwi_loss_function / fwi_gauss_newton_product.  Times are host wall clock around calls that end in a device synchronise.

    python tools/exp_gn_convergence.py --out DIR        -> DIR/exp_gn_convergence.txt
"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--budget", type=int, default=20, help="factorisations per method")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("exp_gn_convergence.py needs a CUDA device")
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import api
    from waveforminversionust_b200 import geometry as G
    n, dtype = 256, "c64"
    geom = G.ring_geometry(n, 256)
    f_hi = G.frequency_for_grid(n)
    freqs = np.linspace(0.25, 0.5, 4) * f_hi
    vel_true = G.blob_model(geom)
    c_init = 1500.0
    dv = torch.device("cuda:0")
    src = w.OneHotSources(geom.src_lin, (n, n, geom.tx_include.size))
    nt = geom.tx_include.size
    # observed data: amp_t * u_t(element e) of this solver at the truth, every frequency
    plan = api.get_plan(n, n, dtype, 0, freqs.size, nt, "python", True)
    plan.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
    plan.set_acquisition(geom.src_lin, (geom.y_idx * n + geom.x_idx).astype(np.int32), geom.mask_indices)
    rec = torch.zeros((freqs.size, nt, geom.num_elements), dtype=plan.tcplx, device=dv)
    plan.fwi_loss_grad(torch.as_tensor((1.0 / vel_true).astype(np.float32)).to(dv), rec, freqs)
    amp = torch.as_tensor(G.source_amplitudes(nt)).to(dv, plan.tcplx)
    rx = torch.as_tensor((geom.y_idx * n + geom.x_idx).astype(np.int64)).to(dv)
    for i in range(freqs.size):
        rec[i] = plan.wavefield(i).reshape(n * n, nt)[rx, :].T * amp[:, None]
    torch.cuda.synchronize()
    fargs = (geom.xi, geom.yi, rec, src, freqs, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab, geom.mask_indices,
             geom.num_elements)
    rms = lambda vel: float(np.sqrt(np.mean((np.asarray(vel, dtype=np.float64) - vel_true) ** 2)))
    lines = [f"# {n}x{n} grid, {nt}-element ring, frequencies {', '.join(f'{f / 1e3:.1f}' for f in freqs)} kHz, {dtype}, "
             f"truth geometry.blob_model, start {c_init} m/s (model RMS error {rms(np.full((n, n), c_init)):.3f} m/s)",
             f"# card: {_card()}"]

    # warm-up of every path (graph capture, module load)
    s0 = torch.full((n, n), 1.0 / c_init, dtype=torch.float32, device=dv)
    api.fwi_loss_function(s0, *fargs, dtype=dtype)
    api.fwi_gauss_newton_product(s0, s0 * 1e-3, *fargs, dtype=dtype)
    plan.ncg_linesearch(s0)
    torch.cuda.synchronize()

    rows = []  # (method, factorisations, products, wall_s, loss, rms)

    # NCG: one factorisation per iteration; the driver returns the final model only, so it is re-run per iteration count
    for k in range(1, a.budget + 1):
        hist = []
        t0 = time.perf_counter()
        vel = api.nonlinear_conjugate_gradient(geom.xi, geom.yi, geom.num_elements, rec, src, geom.tx_include, geom.ind_matlab, c_init,
                                               freqs, k, geom.a0, geom.L_PML, geom.mask_indices, dtype=dtype, history=hist,
                                               return_fields=False)[0]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        loss, _ = api.fwi_loss_function(torch.as_tensor(1.0 / vel).to(dv), *fargs, dtype=dtype)
        rows.append(("ncg", k, 0, dt, float(loss), rms(vel)))

    def recorder(method):
        st = {"t0": time.perf_counter(), "evals": 0, "prods": 0}

        def loss_grad(slow):
            s = torch.as_tensor(np.asarray(slow)) if not torch.is_tensor(slow) else slow
            st["slow"] = s.to(dv, torch.float32).contiguous()
            loss, grad = api.fwi_loss_function(st["slow"], *fargs, dtype=dtype)
            loss = float(loss)
            st["evals"] += 1
            rows.append((method, st["evals"], st["prods"], time.perf_counter() - st["t0"], loss, rms(1.0 / st["slow"].double().cpu().numpy())))
            return loss, grad if torch.is_tensor(slow) else grad.double().cpu().numpy()

        def hvp(v):
            st["prods"] += 1
            return api.fwi_gauss_newton_product(st["slow"], v.to(dv, torch.float32).contiguous(), *fargs, dtype=dtype)

        return loss_grad, hvp

    lg, _ = recorder("lbfgs")
    api.run_lbfgs_fwi(geom.xi, geom.yi, None, None, geom.tx_include, geom.ind_matlab, c_init, freqs, geom.a0, geom.L_PML, geom.mask_indices,
                      maxiter=a.budget, tol=0.0, dtype=dtype, loss_grad=lg)
    for cg in (4, 8):
        lg, hvp = recorder(f"gn(cg_iters={cg})")
        ghist = []
        api.gauss_newton_fwi(geom.xi, geom.yi, geom.num_elements, None, None, geom.tx_include, geom.ind_matlab, c_init, freqs, a.budget,
                             geom.a0, geom.L_PML, geom.mask_indices, cg_iters=cg, dtype=dtype, history=ghist, loss_grad=lg, hvp=hvp)
        for h in ghist:
            lines.append(f"# gn(cg_iters={cg}) outer {h['it']}: cg {h['cg_iters']}, step {h['step']}, evals {h['evals']}, products {h['products']}"
                         + (f", stop: {h['stop']}" if "stop" in h else ""))

    lines.append(f"{'method':<16} {'factorisations':>14} {'products':>9} {'wall_s':>8} {'loss':>14} {'rms_m_s':>9}")
    for r in rows:
        if r[1] <= a.budget:
            lines.append(f"{r[0]:<16} {r[1]:>14d} {r[2]:>9d} {r[3]:>8.3f} {r[4]:>14.6e} {r[5]:>9.3f}")
    best = {}
    for r in rows:
        if r[1] <= a.budget:
            best[r[0]] = min(best.get(r[0], (np.inf,)), (r[5], r[1], r[3], r[4]))
    lines.append("# lowest model RMS error within the budget: " + "; ".join(
        f"{m} {b[0]:.3f} m/s at {b[1]} factorisations, {b[2]:.2f} s" for m, b in best.items()))
    txt = "\n".join(lines) + "\n"
    print(txt)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "exp_gn_convergence.txt"), "w") as fh:
        fh.write(txt)


def _card():
    import subprocess
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


if __name__ == "__main__":
    main()
