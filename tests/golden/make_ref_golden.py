"""Reference-EXECUTED fixtures: runs the reference's own, unmodified source text and stores what it returns.

    python tests/golden/make_ref_golden.py            # needs /root/reference (this container only)

``/root/reference/Final_python/{solve_helmholtz,nonlinearcg,fwi_loss_function,fwi_script}.py`` are imported as they lie
(nothing is copied or edited) on top of ``oracle/jax_shim.py``, a NumPy-backed stand-in for the few dozen ``jax`` names they
use (JAX itself is not installable here: no network).  The sparse solve is the reference's own ``scipy_solve`` ->
``scipy.sparse.linalg.spsolve`` (SuperLU).  Two arithmetic modes, both legitimate JAX configurations:
  * ``x32``: x64 disabled (the reference's default): float32 / complex64 throughout;
  * ``x64``: ``jax.config.update("jax_enable_x64", True)``: float64 assembly and SuperLU, the reference's explicit
    ``complex64`` casts (``solve_helmholtz.py:79, 87``) still applied.  This mode sits ~1e-7 from exact arithmetic, far
    below the complex64 SuperLU noise floor (1e-5), so it pins the ALGORITHM (stencil, index conventions, conjugations,
    reshape orders, NCG update) tightly; the x32 mode pins the reference's actual single-precision outputs.
Outputs: tests/golden/ref_*.npz, consumed by tests/test_ref_pin.py (CPU: oracle vs these) and tests/test_gpu_parity.py
(CUDA path vs these).
"""
import importlib
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
REF = "/root/reference/Final_python"
HERE = os.path.dirname(os.path.abspath(__file__))

from oracle import jax_shim  # noqa: E402
from waveforminversionust_b200.matfile import load_mat73  # noqa: E402


def _mat73_like(path):
    """What ``mat73.loadmat`` returns for RecordedData.mat: vectors squeezed to 1-D, scalars to float."""
    d = load_mat73(os.path.join(REF, os.path.basename(path)))
    out = {}
    for k, v in d.items():
        v = np.asarray(v)
        out[k] = float(v.ravel()[0]) if v.size == 1 else (v.ravel() if 1 in v.shape else v)
    return out


def load_reference(x64):
    jax = jax_shim.install(mat_loader=_mat73_like)
    jax.config.update("jax_enable_x64", x64)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    mods = {}
    for name in ("solve_helmholtz", "nonlinearcg", "fwi_loss_function", "fwi_script"):
        sys.modules.pop(name, None)
    for name in ("solve_helmholtz", "nonlinearcg", "fwi_loss_function", "fwi_script"):
        mods[name] = importlib.import_module(name)
        assert mods[name].__file__.startswith(REF), mods[name].__file__
    return jax, mods


def ring_inputs(jnp, n, nelem, seed, pml_cells, real):
    """Inputs built the way ``fwi_script.py:31-85`` builds them, on a small synthetic ring (tests/common.small_case)."""
    from common import bde_for, observed_data, small_case
    geom, f, vel_true = small_case(n, nelem, seed=seed, pml_cells=pml_cells)
    rec = observed_data(geom, f, vel_true, bde=bde_for(geom, vel_true, f))  # complex128 "measured" data
    cplx = np.complex64  # fwi_script.py:26 casts REC_DATA to complex64 in both modes
    xi = jnp.array(geom.xi.astype(real))
    yi = jnp.array(geom.yi.astype(real))
    SRC = jnp.zeros((geom.Ny, geom.Nx, geom.tx_include.size), dtype=jnp.complex64)  # :72-74
    for i, t in enumerate(geom.tx_include):
        SRC = SRC.at[geom.y_idx[t], geom.x_idx[t], i].set(1.0)
    return geom, f, vel_true, rec, dict(
        xi=xi, yi=yi, REC_DATA=jnp.array(rec.astype(cplx)), SRC=SRC, tx_include=jnp.array(geom.tx_include),
        ind_matlab=jnp.array(geom.ind_matlab), mask_indices=jnp.array(geom.mask_indices), f=jnp.array(real(f)))


def np_(a):
    return np.asarray(jax_shim._unwrap(a))


def case_solve(mode, n=44, nelem=16, seed=2, pml_cells=6.0, nrhs=3):
    """solve_helmholtz: CSR matrix the reference hands to SuperLU (forward and adjoint), b/d/e, wavefields."""
    x64 = mode == "x64"
    jax, m = load_reference(x64)
    jnp = jax.numpy
    real = np.float64 if x64 else np.float32
    geom, f, vel_true, rec, inp = ring_inputs(jnp, n, nelem, seed, pml_cells, real)
    sh = m["solve_helmholtz"]
    captured = []
    orig = sh.scipy_solve

    def spy(data, indices, indptr, rhs_np, shape):
        captured.append((np.array(data), np.array(indices), np.array(indptr)))
        return orig(data, indices, indptr, rhs_np, shape)

    sh.scipy_solve = spy
    vel = jnp.array(vel_true.astype(real))
    rng = np.random.default_rng(5)
    dense = (rng.standard_normal((n, n, nrhs)) + 1j * rng.standard_normal((n, n, nrhs))).astype(np.complex64)
    dense[0] = dense[-1] = 0  # the FWI loop never puts a right-hand side on the Dirichlet ring
    dense[:, 0] = dense[:, -1] = 0
    onehot = np_(inp["SRC"])[:, :, :nrhs]
    out = {}
    for tag, src in (("onehot", onehot), ("dense", dense)):
        for adj in (False, True):
            u = sh.solve_helmholtz(inp["xi"], inp["yi"], vel, jnp.array(src), inp["f"], geom.a0, geom.L_PML, adj)
            out["wv_%s_%s" % (tag, "adj" if adj else "fwd")] = np_(u)
    sh.scipy_solve = orig
    h = jnp.mean(jnp.diff(inp["xi"]))
    g = jnp.mean(jnp.diff(inp["yi"])) / h
    b, d, e = sh.stencil_opt_params(jnp.min(vel), jnp.max(vel), inp["f"], h, g)
    fwd, adj = captured[0], captured[1]
    np.savez_compressed(
        os.path.join(HERE, "ref_solve_%s.npz" % mode), mode=mode, n=n, nelem=nelem, seed=seed, pml_cells=pml_cells, f=f,
        vel=vel_true, dense_src=dense, nrhs=nrhs, bde=np.array([float(b), float(np_(d)), float(np_(e))]),
        csr_data=fwd[0], csr_indices=fwd[1], csr_indptr=fwd[2], csr_adj_data=adj[0], csr_adj_indices=adj[1],
        csr_adj_indptr=adj[2], **out)
    print("ref_solve_%s: bde" % mode, float(b), float(np_(d)), float(np_(e)), "dtype", out["wv_onehot_fwd"].dtype, fwd[0].dtype)


def case_ncg(mode, n=48, nelem=16, seed=0, pml_cells=4.0, niter=2):
    """nonlinear_conjugate_gradient_vectorized (2 iterations), the loop form (1 iteration) and fwi_loss_function."""
    x64 = mode == "x64"
    jax, m = load_reference(x64)
    jnp = jax.numpy
    real = np.float64 if x64 else np.float32
    geom, f, vel_true, rec, inp = ring_inputs(jnp, n, nelem, seed, pml_cells, real)
    ncg = m["nonlinearcg"]
    args = (inp["xi"], inp["yi"], geom.num_elements, inp["REC_DATA"], inp["SRC"], inp["tx_include"], inp["ind_matlab"],
            1480.0, inp["f"], niter, geom.a0, geom.L_PML, inp["mask_indices"])
    VEL, sd, grad, ADJ_WV, WV = ncg.nonlinear_conjugate_gradient_vectorized(*args)
    a1 = list(args)
    a1[9] = 1
    VEL1, sd1, grad1, ADJ1, WV1 = ncg.nonlinear_conjugate_gradient_vectorized(*a1)
    VELl, sdl, gradl, ADJl, WVl = ncg.nonlinear_conjugate_gradient(*a1)  # loop form (what fwi_script.py:115 calls)
    lf = m["fwi_loss_function"]
    params = 1.0 / (1480.0 * jnp.ones((n, n)))  # fwi_loss_function.py:110-111 (2-D init_params)
    loss = lf.fwi_loss_function(params, inp["xi"], inp["yi"], inp["REC_DATA"], inp["SRC"], inp["f"], geom.a0, geom.L_PML,
                                inp["tx_include"], inp["ind_matlab"], inp["mask_indices"], geom.num_elements)
    np.savez_compressed(
        os.path.join(HERE, "ref_ncg_%s.npz" % mode), mode=mode, n=n, nelem=nelem, seed=seed, pml_cells=pml_cells, f=f,
        niter=niter, rec=rec, vel_true=vel_true, loss0=float(np_(loss)),
        VEL=np_(VEL), sd=np_(sd), grad=np_(grad), ADJ_WV=np_(ADJ_WV)[:, :, :2], WV=np_(WV)[:, :, :2],
        VEL1=np_(VEL1), sd1=np_(sd1), grad1=np_(grad1), ADJ_WV1=np_(ADJ1)[:, :, :2], WV1=np_(WV1)[:, :, :2],
        VEL1_loop=np_(VELl), grad1_loop=np_(gradl))
    print("ref_ncg_%s: loss0 %.9e |grad1| %.6e |grad| %.6e VEL [%.3f, %.3f]; loop vs vectorised grad rel %.2e" % (
        mode, float(np_(loss)), np.linalg.norm(np_(grad1)), np.linalg.norm(np_(grad)), np_(VEL).min(), np_(VEL).max(),
        np.linalg.norm(np_(gradl) - np_(grad1)) / np.linalg.norm(np_(grad1))))


def case_script():
    """BASELINE configs[0]: ``fwi_script.main()`` itself on the shipped RecordedData.mat (x64 disabled, Niter = 1, loop-form
    NCG as ``fwi_script.py:115`` calls it).  The call into nonlinearcg is observed, not altered."""
    jax, m = load_reference(False)
    fs = m["fwi_script"]
    seen = {}
    orig = fs.nonlinear_conjugate_gradient

    def spy(*a):
        seen["args"] = a
        seen["out"] = orig(*a)
        return seen["out"]

    fs.nonlinear_conjugate_gradient = spy
    t0 = time.time()
    fs.main()
    fs.nonlinear_conjugate_gradient = orig
    a = seen["args"]
    VEL, sd, grad, ADJ_WV, WV = (np_(v) for v in seen["out"])
    xi, ind_matlab, mask = np_(a[0]), np_(a[6]), np_(a[12])
    print("fwi_script.main(): %.0f s; grid %d, |grad| %.6e, VEL [%.3f, %.3f]" % (
        time.time() - t0, xi.size, np.linalg.norm(grad), VEL.min(), VEL.max()))
    # receivers-only slices keep the fixture small (under 1 MB): the scaled forward field and the adjoint field at the element
    # nodes, for every 4th source
    yx = (ind_matlab % xi.size, ind_matlab // xi.size)  # ind_matlab = x_idx*Nxi + y_idx (fwi_script.py:68)
    np.savez_compressed(
        os.path.join(HERE, "ref_script_cfg1.npz"), xi=xi, ind_matlab=ind_matlab, mask_indices=mask.astype(np.int16),
        f=float(np_(a[8])), c_init=float(a[7]), a0=float(a[10]), L_PML=float(a[11]), grad_norm=float(np.linalg.norm(grad)),
        VEL_dec2=VEL[::2, ::2], grad_dec2=grad[::2, ::2], sd_dec2=sd[::2, ::2], vel_min=float(VEL.min()), vel_max=float(VEL.max()),
        WV_at_elements=WV[yx[0], yx[1], ::4], ADJ_WV_at_elements=ADJ_WV[yx[0], yx[1], ::4], grad_sum=float(grad.sum()),
        grad_abs_sum=float(np.abs(grad).sum()))


if __name__ == "__main__":
    which = sys.argv[1:] or ["solve", "ncg", "script"]
    if "solve" in which:
        for mode in ("x32", "x64"):
            case_solve(mode)
    if "ncg" in which:
        for mode in ("x32", "x64"):
            case_ncg(mode)
    if "script" in which:
        case_script()
    jax_shim.uninstall()
