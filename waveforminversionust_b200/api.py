"""Reference-facing surface: the same names, argument order and meaning as the reference's
``solve_helmholtz.py``, ``fwi_loss_function.py`` and ``nonlinearcg.py``, running on libustfwi.so.

    solve_helmholtz(x, y, vel, src, f, a0, L_PML, adjoint)            solve_helmholtz.py:21-101
    fwi_loss_function(params, xi, yi, REC_DATA, SRC, f, a0, L_PML,
                      tx_include, ind_matlab, mask_indices, num_elements) -> (loss, grad)
                                                                       fwi_loss_function.py:29-103
    nonlinear_conjugate_gradient[_vectorized](xi, yi, numElements, REC_DATA, SRC, tx_include,
                      ind_matlab, c_init, f, Niter, a0, L_PML, mask_indices)
                                                                       nonlinearcg.py:41-308

Inputs may be NumPy arrays (host buffers: copies happen inside the C call) or torch CUDA tensors
(device buffers: zero-copy).  There is no CPU fallback: without the CUDA library / a GPU these raise.
Extensions over the reference (keyword-only): ``dtype`` ("c64" default = the reference's precision,
or "c128"), ``engine`` ("auto" | "simt" | "tc2": block-GEMM engine; tcgen05 is complex64 only), ``bde`` (inject the stencil weights), ``stencil`` ("python" | "matlab"), and ``f`` /
``REC_DATA`` may carry a leading frequency axis for the joint multi-frequency objective.

Attenuation (not in the reference): ``kappa`` (attenuation slowness, s/m) makes the medium lossy with complex slowness
``1/c - i kappa`` (``solve_helmholtz``, ``time_domain_simulation``); ``fwi_joint_loss_function`` and ``run_lbfgs_joint_fwi``
invert sound speed and attenuation together (DESIGN.md section 7d); ``fwi_joint_gauss_newton_product``,
``nonlinear_conjugate_gradient_joint``, ``gauss_newton_joint_fwi`` and ``joint_frequency_continuation`` add the joint
Gauss-Newton product, NCG and truncated Gauss-Newton (section 7e).

Exact derivative (not in the reference): ``gradient="discrete"`` on every gradient-based function and driver builds the
gradient, the line search and the Gauss-Newton product from the exact derivative of the discrete forward map at fixed stencil
weights instead of the reference's virtual source (DESIGN.md section 7f).  The default ``"reference"`` keeps the reference's.
"""
from __future__ import annotations

import hashlib
import math

import numpy as np

from .plan import HelmholtzPlan

_PLANS = {}


def _is_torch(a):
    return type(a).__module__.startswith("torch")


def _to_np(a):
    if _is_torch(a):
        return a.detach().cpu().numpy()
    return np.asarray(a)


def _device_of(*arrs):
    for a in arrs:
        if _is_torch(a) and a.is_cuda:
            return a.device.index
    return 0


def get_plan(nx, ny, dtype, device, max_freq, max_nrhs, stencil, fwi_buffers, engine="auto"):
    """Plan cache: plans are reused (and grown) per (grid, precision, device, stencil, engine)."""
    key = (nx, ny, dtype, device, stencil, engine)
    p = _PLANS.get(key)
    if p is not None and (p.max_freq < max_freq or p.max_nrhs < max_nrhs or (fwi_buffers and not p.fwi_buffers)):
        max_freq, max_nrhs = max(max_freq, p.max_freq), max(max_nrhs, p.max_nrhs)
        fwi_buffers = fwi_buffers or p.fwi_buffers
        p.close()
        p = None
    if p is None:
        p = HelmholtzPlan(nx, ny, dtype=dtype, max_freq=max_freq, max_nrhs=max_nrhs, device=device,
                          stencil=stencil, fwi_buffers=fwi_buffers, engine=engine)
        p.fwi_buffers = bool(fwi_buffers)
        _PLANS[key] = p
    return p


def clear_plans():
    for p in _PLANS.values():
        p.close()
    _PLANS.clear()


def _fingerprint(*parts):
    h = hashlib.blake2b(digest_size=16)
    for q in parts:
        if isinstance(q, np.ndarray):
            h.update(np.ascontiguousarray(q).tobytes())
        else:
            h.update(repr(q).encode())
    return h.digest()


def solve_helmholtz(x, y, vel, src, f, a0, L_PML, adjoint, *, dtype="c64", bde=None, stencil="python", engine="auto",
                    kappa=None):
    """Solve H(vel, f) u = src (or conj(H)^T u = src when ``adjoint``) for every column of ``src``.

    ``src`` is (Ny, Nx, nrhs) (anything that reshapes C-order to (Ny*Nx, nrhs), solve_helmholtz.py:78);
    returns (Ny, Nx, nrhs) complex (solve_helmholtz.py:101).  The factorisation is cached and reused
    while (vel, f, grid, PML, weights, kappa) stay the same, so the forward / adjoint / perturbation solves of
    one iteration (nonlinearcg.py:213,263,279) factorise once instead of three times.

    ``kappa`` ((Ny, Nx) attenuation slowness, s/m, >= 0): lossy medium with complex slowness ``1/vel - i kappa``, amplitude
    attenuation ``2 pi f kappa`` Np/m (``geometry.db_cm_mhz_to_kappa`` converts from dB/(cm MHz)).  NumPy inputs then go
    through device tensors; the result is NumPy as for the lossless call.
    """
    xh, yh = _to_np(x).astype(np.float64).ravel(), _to_np(y).astype(np.float64).ravel()
    nx, ny = xh.size, yh.size
    f = float(np.asarray(_to_np(f)).reshape(-1)[0])
    adjoint = bool(np.asarray(_to_np(adjoint)).reshape(-1)[0]) if not isinstance(adjoint, bool) else adjoint
    nrhs = int(np.prod(src.shape)) // (nx * ny)
    dev = _device_of(src, vel, kappa)
    plan = get_plan(nx, ny, dtype, dev, 1, nrhs, stencil, False, engine)
    plan.set_grid(xh, yh, float(a0), float(L_PML))
    on_dev = _is_torch(src) and src.is_cuda
    if on_dev or kappa is not None:
        import torch
        dv = src.device if on_dev else torch.device(f"cuda:{dev}")
        velt = vel if _is_torch(vel) else torch.as_tensor(_to_np(vel))
        velt = velt.to(device=dv, dtype=plan.treal).reshape(ny, nx).contiguous()
        parts = (velt.cpu().numpy(), f, None if bde is None else np.asarray(bde, dtype=np.float64))
        kapt = None
        if kappa is not None:
            kapt = (kappa if _is_torch(kappa) else torch.as_tensor(_to_np(kappa))).to(device=dv, dtype=plan.treal).reshape(ny, nx).contiguous()
            parts += ("kappa", kapt.cpu().numpy())
        key = _fingerprint(*parts)
        if plan._factor_key != key:
            plan.factor(velt, [f], bde=None if bde is None else [bde], kappa=kapt)
            plan._factor_key = key
        srct = src if _is_torch(src) else torch.as_tensor(_to_np(src))
        out = srct.to(device=dv, dtype=plan.tcplx).reshape(ny * nx, nrhs).contiguous().clone()
        plan.solve(out, 0, adjoint)
        out = out.reshape(ny, nx, nrhs)
        return out if on_dev else out.cpu().numpy()
    velh = _to_np(vel).astype(plan.real)
    key = _fingerprint(velh, f, None if bde is None else np.asarray(bde, dtype=np.float64))
    refactor = plan._factor_key != key
    out = plan.solve_helmholtz_host(velh, _to_np(src), f, adjoint=adjoint, bde=bde, refactor=refactor)
    plan._factor_key = key
    return out


def _acquisition(SRC, ind_matlab, mask_indices, nx, ny):
    """Convert the reference's arrays to what the C ABI takes: one-hot source nodes and row-major
    receiver nodes.  ``ind_matlab`` indexes the column-major (order='F') flattening of a (Ny, Nx) field
    (nonlinearcg.py:220-222): p = x*Ny + y."""
    ind = _to_np(ind_matlab).astype(np.int64).ravel()
    xr, yr = ind // ny, ind % ny
    rx_lin = (yr * nx + xr).astype(np.int32)
    mask = _to_np(mask_indices).astype(np.int32)
    if hasattr(SRC, "src_lin"):
        src_lin = np.asarray(SRC.src_lin, dtype=np.int32)
    else:
        S = _to_np(SRC)
        nt = S.shape[2]
        flat = S.reshape(ny * nx, nt)
        nz_row, nz_col = np.nonzero(flat)
        if nz_col.size != nt or not np.array_equal(np.sort(nz_col), np.arange(nt)) or not np.allclose(flat[nz_row, nz_col], 1.0):
            raise NotImplementedError("fwi_loss_function: SRC must be one-hot unit sources (fwi_script.py:72-74)")
        src_lin = np.empty(nt, dtype=np.int32)
        src_lin[nz_col] = nz_row
    return src_lin, rx_lin, mask


class OneHotSources:
    """Sparse stand-in for the reference's dense (Ny, Nx, Nt) one-hot ``SRC`` array."""

    def __init__(self, src_lin, shape):
        self.src_lin = np.asarray(src_lin, dtype=np.int32)
        self.shape = tuple(shape)


def _fwi_plan(xi, yi, REC_DATA, SRC, f, a0, L_PML, ind_matlab, mask_indices, dtype, stencil, device, engine="auto",
              gradient="reference"):
    """The cached plan of this problem with its grid, acquisition and gradient mode set.  Plans are shared, so the mode is set
    on every call rather than left from an earlier one."""
    xh, yh = _to_np(xi).astype(np.float64).ravel(), _to_np(yi).astype(np.float64).ravel()
    nx, ny = xh.size, yh.size
    freqs = np.atleast_1d(np.asarray(_to_np(f), dtype=np.float64)).ravel()
    src_lin, rx_lin, mask = _acquisition(SRC, ind_matlab, mask_indices, nx, ny)
    plan = get_plan(nx, ny, dtype, device, freqs.size, src_lin.size, stencil, True, engine)
    plan.set_grid(xh, yh, float(a0), float(L_PML))
    plan.set_acquisition(src_lin, rx_lin, mask)
    plan.set_gradient(gradient)
    return plan, freqs


def fwi_loss_function(params, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices,
                      num_elements, *, dtype="c64", bde=None, stencil="python", engine="auto", gradient="reference"):
    """(loss, grad): loss of fwi_loss_function.py:29-103 and the adjoint-state gradient with respect to
    the slowness ``params`` (nonlinearcg.py:243-265), ``grad.shape == params.shape``.

    ``gradient``: ``"reference"`` builds the gradient from the reference's virtual source ``2 w^2 s alpha u``;
    ``"discrete"`` from the exact derivative of the discrete forward map at fixed stencil weights (the 9-point mass stencil
    and the PML factor, DESIGN.md section 7f), so that it is the derivative of the returned loss.  The loss is the same.

    With ``f`` of length Nf and ``REC_DATA`` of shape (Nf, Nt, E) the joint objective sum_f loss_f is
    returned.  Usable as ``jaxopt.LBFGS(fun, value_and_grad=True)`` / ``scipy.optimize.minimize(jac=True)``.
    """
    return _loss_function(False, params, xi, yi, REC_DATA, SRC, f, a0, L_PML, ind_matlab, mask_indices, dtype, bde, stencil,
                          engine, gradient)


def fwi_joint_loss_function(params, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements,
                            *, dtype="c64", bde=None, stencil="python", engine="auto", gradient="reference"):
    """(loss, grad) of the joint sound-speed and attenuation problem: ``params`` is (2, Ny, Nx) = [slowness s (s/m),
    attenuation slowness kappa (s/m)] of the complex slowness ``s - i kappa``, and ``grad`` has ``params``' shape
    ([dloss/ds, dloss/dkappa]).  The other arguments and the loss are those of ``fwi_loss_function``; the gradients use the
    same linearisation (source estimates held fixed, DESIGN.md section 7d) and ``gradient`` mode.  The ``value_and_grad`` contract of
    ``fwi_loss_function``: torch CUDA in -> torch out (device buffers), NumPy in -> NumPy out (host buffers)."""
    return _loss_function(True, params, xi, yi, REC_DATA, SRC, f, a0, L_PML, ind_matlab, mask_indices, dtype, bde, stencil,
                          engine, gradient)


def _loss_function(lossy, params, xi, yi, REC_DATA, SRC, f, a0, L_PML, ind_matlab, mask_indices, dtype, bde, stencil, engine,
                   gradient):
    """The body of ``fwi_loss_function`` (``lossy``: of ``fwi_joint_loss_function``, ``params`` = [s, kappa])."""
    dev = _device_of(params, REC_DATA)
    plan, freqs = _fwi_plan(xi, yi, REC_DATA, SRC, f, a0, L_PML, ind_matlab, mask_indices, dtype, stencil, dev, engine, gradient)
    if lossy and tuple(params.shape) != (2, plan.ny, plan.nx):
        raise ValueError(f"params must have shape (2, {plan.ny}, {plan.nx}) = [slowness, kappa]")
    if _is_torch(params) and params.is_cuda:
        import torch
        rec = REC_DATA.to(plan.tcplx).reshape(freqs.size, plan.nt, plan.nelem).contiguous()
        p = params.to(plan.treal)
        maps = (p[0].contiguous(), p[1].contiguous()) if lossy else (p.reshape(plan.ny, plan.nx).contiguous(), None)
        loss, *grads = plan._loss_grad(*maps, rec, freqs, bde)
        loss, grad, shape = loss[0], torch.stack(grads) if lossy else grads[0], params.shape
    else:
        p = np.asarray(_to_np(params), dtype=plan.real)
        maps = (p[0], p[1]) if lossy else (p.reshape(plan.ny, plan.nx), None)
        loss, *grads = plan._loss_grad_host(*maps, _to_np(REC_DATA), freqs, bde, None)
        grad, shape = np.stack(grads) if lossy else grads[0], p.shape
    plan._eval_key = _eval_key(params, REC_DATA, freqs, bde, lossy, gradient)
    return loss, grad.reshape(shape)


def _eval_key(params, REC_DATA, freqs, bde, lossy=False, gradient="reference"):
    """What identifies an evaluation's state on the plan: device inputs are kept as copies (compared on the device), host
    inputs as a hash.  The key of a lossy evaluation is tagged, so that it never matches a lossless one, and so is the key of
    the discrete gradient mode, so that an evaluation in one mode is never reused for a product in the other."""
    b = None if bde is None else np.asarray(bde, dtype=np.float64)
    tag = ("-lossy" if lossy else "") + ("-discrete" if gradient == "discrete" else "")
    if _is_torch(params) and params.is_cuda:
        rec = REC_DATA.detach().clone() if _is_torch(REC_DATA) else _fingerprint(np.asarray(REC_DATA))
        return ("dev" + tag, params.detach().clone(), rec, _fingerprint(freqs, b))
    return ("host" + tag, _fingerprint(np.asarray(_to_np(params)), np.asarray(_to_np(REC_DATA)), freqs, b))


def _same_eval(a, b):
    import torch
    if a is None or b is None or a[0] != b[0] or len(a) != len(b):
        return False
    for x, y in zip(a[1:], b[1:]):
        if _is_torch(x) != _is_torch(y):
            return False
        if _is_torch(x):
            if x.shape != y.shape or x.dtype != y.dtype or x.device != y.device or not torch.equal(x, y):
                return False
        elif x != y:
            return False
    return True


def fwi_gauss_newton_product(params, v, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements,
                             *, dtype="c64", bde=None, stencil="python", engine="auto", gradient="reference"):
    """Gauss-Newton Hessian-vector product ``H_GN v = Re(J^H J v)`` of the objective of ``fwi_loss_function`` at slowness
    ``params``, returned with ``params``' shape (NumPy in, NumPy out; a CUDA tensor ``v`` gives a CUDA tensor).

    ``J`` is the linearisation the gradient is built from (``nonlinearcg.py:258,279``): the perturbation solve with virtual
    source ``-2 w^2 s alpha u v``, gathered at the kept receivers, with the source estimates ``alpha`` held fixed, so that the
    gradient is ``Re(J^H residual)``.  The virtual source leaves out the stencil's mass weights and the PML factor, as the
    reference does: ``J`` is not the exact derivative of the discrete forward map (DESIGN.md section 7c).  With
    ``gradient="discrete"`` it is, at fixed stencil weights (section 7f), and the gradient of
    ``fwi_loss_function(..., gradient="discrete")`` is ``Re(J^H residual)`` of that ``J``.

    A product costs two all-source sweeps on the factorisation the last evaluation left on the plan; when the last
    ``fwi_loss_function`` on this plan had other ``(params, REC_DATA, f, bde)``, the evaluation runs first.
    """
    return _gauss_newton_product(False, params, v, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices,
                                 num_elements, dtype, bde, stencil, engine, gradient)


def fwi_joint_gauss_newton_product(params, v, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices,
                                   num_elements, *, dtype="c64", bde=None, stencil="python", engine="auto", gradient="reference"):
    """Gauss-Newton product ``H_GN v = Re(J^H J v)`` of the joint objective of ``fwi_joint_loss_function``: ``params`` and
    ``v`` are (2, Ny, Nx) = [slowness, kappa] blocks, and so is the result (NumPy in, NumPy out; a CUDA tensor ``v`` gives a
    CUDA tensor).

    With the complex slowness ``sigma = s - i kappa`` and the source estimates held fixed, ``J [v_s; v_kappa]`` is the
    perturbation solve with virtual source ``-2 w^2 sigma alpha u (v_s - i v_kappa)`` gathered at the kept receivers, the
    linearisation the joint gradient is built from (DESIGN.md section 7e).  Because ``J_kappa = -i J_s``, the blocks satisfy
    ``H_kk = H_ss`` and ``H_ks = -H_sk``; both hold in the ``gradient="discrete"`` mode too (section 7f).

    A product costs two all-source sweeps on the factorisation the last evaluation left on the plan; when the last
    ``fwi_joint_loss_function`` on this plan had other ``(params, REC_DATA, f, bde)`` (or the last evaluation was lossless),
    the evaluation runs first.
    """
    return _gauss_newton_product(True, params, v, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices,
                                 num_elements, dtype, bde, stencil, engine, gradient)


def _gauss_newton_product(lossy, params, v, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices,
                          num_elements, dtype, bde, stencil, engine, gradient):
    """The body of ``fwi_gauss_newton_product`` (``lossy``: of ``fwi_joint_gauss_newton_product``)."""
    import torch
    dev = _device_of(params, REC_DATA, v)
    plan, freqs = _fwi_plan(xi, yi, REC_DATA, SRC, f, a0, L_PML, ind_matlab, mask_indices, dtype, stencil, dev, engine, gradient)
    if lossy and tuple(v.shape) != (2, plan.ny, plan.nx):
        raise ValueError(f"v must have shape (2, {plan.ny}, {plan.nx}) = [slowness, kappa] directions")
    if not _same_eval(plan._eval_key, _eval_key(params, REC_DATA, freqs, bde, lossy, gradient)):
        # looked up at call time: tests record the evaluation points by replacing these module functions
        evaluate = fwi_joint_loss_function if lossy else fwi_loss_function
        evaluate(params, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements, dtype=dtype,
                 bde=bde, stencil=stencil, engine=engine, gradient=gradient)
    on_device = _is_torch(v) and v.is_cuda
    if on_device:
        vt = v.detach().to(plan.treal)
    else:
        vt = torch.as_tensor(np.ascontiguousarray(np.asarray(_to_np(v), dtype=plan.real))).to(f"cuda:{plan.device}")
    dirs = (vt[0].contiguous(), vt[1].contiguous()) if lossy else (vt.reshape(plan.ny, plan.nx).contiguous(), None)
    hv, _ = plan._gn_hvp(*dirs, False)
    hv = hv.reshape(np.shape(params))
    return hv if on_device else hv.cpu().numpy()


def nonlinear_conjugate_gradient(xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, Niter,
                                 a0, L_PML, mask_indices, *, dtype="c64", bde=None, stencil="python",
                                 device=0, history=None, return_fields=True, engine="auto", gradient="reference"):
    """The reference's NCG loop (nonlinearcg.py:41-180 / 184-308: Hestenes-Stiefel beta, forced to 0 at
    the first iteration; linearised exact step) on the GPU path: per iteration one factorisation,
    forward + adjoint + perturbation sweeps, all on device.

    Returns (VEL, sd, grad, ADJ_WV, WV) as NumPy arrays like the reference; ADJ_WV / WV (each
    (Ny, Nx, Nt) complex, WV scaled by the source estimates, nonlinearcg.py:227) are only materialised
    when ``return_fields`` and refer to the last iteration / first frequency.  ``gradient``: the gradient and line-search
    linearisation, ``"reference"`` or ``"discrete"`` (``fwi_loss_function``).
    """
    import torch
    plan, freqs = _fwi_plan(xi, yi, REC_DATA, SRC, f, a0, L_PML, ind_matlab, mask_indices, dtype, stencil, device, engine,
                            gradient)
    dv = torch.device(f"cuda:{device}")
    ny, nx = plan.ny, plan.nx
    rec = torch.as_tensor(_to_np(REC_DATA)).to(device=dv, dtype=plan.tcplx).reshape(freqs.size, plan.nt, plan.nelem).contiguous()
    VEL = (torch.as_tensor(np.asarray(_to_np(c_init), dtype=np.float64)) * torch.ones((ny, nx), dtype=torch.float64)).to(dv, plan.treal)
    SLOW = (1.0 / VEL).contiguous()
    sd = torch.zeros((ny, nx), dtype=plan.treal, device=dv)
    gprev = torch.zeros_like(sd)
    grad = torch.zeros_like(sd)
    for it in range(int(Niter)):
        loss, grad = plan.fwi_loss_grad(SLOW, rec, freqs, bde=bde)  # nonlinearcg.py:213-265
        dg = grad - gprev  # :268
        if it == 0:  # :274
            beta = torch.zeros((), dtype=plan.treal, device=dv)
        else:
            beta = torch.sum(grad * dg) / torch.sum(sd * dg)  # :270-272
        sd = (beta * sd - grad).contiguous()  # :276
        if return_fields and it == int(Niter) - 1:
            ADJ_WV = plan.adjoint_wavefield(0)  # before the perturbation solve reuses the buffer
        nd = plan.ncg_linesearch(sd)  # :279-298, :24-27
        step = (nd[0] / nd[1]).to(plan.treal)  # :28
        SLOW = (SLOW + step * sd).contiguous()  # :29
        VEL = 1.0 / SLOW  # :30
        if history is not None:
            history.append(dict(it=it, loss=float(loss[0]), grad_norm=float(torch.linalg.norm(grad.double())),
                                beta=float(beta), step=float(step), vel_min=float(VEL.min()), vel_max=float(VEL.max())))
        gprev = grad
    out_adj = out_wv = None
    if return_fields and int(Niter) > 0:
        alpha = torch.as_tensor(plan.src_est(0)).to(dv)
        out_wv = (plan.wavefield(0) * alpha[None, None, :]).cpu().numpy()
        out_adj = ADJ_WV.cpu().numpy()
    return VEL.cpu().numpy(), sd.cpu().numpy(), grad.cpu().numpy(), out_adj, out_wv


nonlinear_conjugate_gradient_vectorized = nonlinear_conjugate_gradient


def run_lbfgs_fwi(xi, yi, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, a0, L_PML, mask_indices, *, maxiter=1, tol=1e-5,
                  history_size=10, dtype="c64", bde=None, stencil="python", engine="auto", history=None, loss_grad=None,
                  pert_scale=1e-2, gradient="reference"):
    """``run_lbfgs_fwi`` of the reference (``fwi_loss_function.py:106-132``): L-BFGS on the slowness map, returning the
    final sound speed ``(Ny, Nx)``.  The reference wires ``jaxopt.LBFGS(fun=loss_fn, maxiter=1, tol=1e-5)`` around a
    loss-only function (which JAX cannot differentiate through ``pure_callback``); here the objective is this package's
    ``fwi_loss_function -> (loss, grad)`` (the ``value_and_grad=True`` contract: ``grad.shape == params.shape``, also for the
    2-D ``init_params`` of ``:110-111``) and the optimiser is SciPy's L-BFGS (jaxopt is not installable in this image; with
    jaxopt present use ``jaxopt.LBFGS(fun, value_and_grad=True, jit=False)`` on the same function).

    Deliberate deviation (SURVEY.md section 8b): in the reference's units ``|grad| ~ 3e-11`` and useful steps are ``~3e7``, so
    ``tol=1e-5`` would stop at iteration 0.  The problem is non-dimensionalised: the unknown is the relative slowness
    perturbation ``p = (s / s0 - 1) / pert_scale`` (a unit step is a ``pert_scale`` = 1 % change) and the objective
    ``loss / loss(s0)``; ``tol`` applies to the projected gradient of that scaled problem.

    ``loss_grad(slow_2d) -> (loss, grad_2d)`` replaces the objective (the parity test drives the same optimiser with the
    oracle's); ``history`` receives ``(loss, params.copy())`` of every evaluation.  ``gradient`` is the gradient mode of
    ``fwi_loss_function``.
    """
    ny, nx = _to_np(yi).size, _to_np(xi).size
    num_elements = int(SRC.shape[2]) if SRC is not None else 0  # unused when ``loss_grad`` is injected
    c0 = np.asarray(_to_np(c_init), dtype=np.float64)
    s0 = 1.0 / float(c0.mean())
    real = np.float32 if dtype == "c64" else np.float64
    if loss_grad is None:
        def loss_grad(slow):
            return fwi_loss_function(slow.astype(real), xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices,
                                     num_elements, dtype=dtype, bde=bde, stencil=stencil, engine=engine, gradient=gradient)

    slow, = _lbfgs_blocks(loss_grad, [_slowness_block(c0, s0, pert_scale, ny, nx)], ny, nx, maxiter, tol, history_size, history)
    return 1.0 / slow


def _slowness_block(c0, s0, pert_scale, ny, nx):
    """The slowness block of the L-BFGS drivers: ``s = (1 + pert_scale p) s0``, starting at ``1 / c0``."""
    p0 = ((np.ones((ny, nx)) / (c0 * s0) - 1.0) / pert_scale).ravel()
    return (lambda p: (1.0 + pert_scale * p) * s0), s0 * pert_scale, p0, None


def _lbfgs_blocks(loss_grad, blocks, ny, nx, maxiter, tol, history_size, history):
    """SciPy's L-BFGS-B on a model of one (Ny, Nx) map or a stack of several, each non-dimensionalised on its own: block
    ``(to_model, dmodel_dp, p0, lower_bound)`` maps its part ``p`` of the unknown to its map ``to_model(p)``, starts at ``p0``
    and is bounded below by ``lower_bound`` (None: unbounded).  The objective is ``loss / loss(start)``.  ``history``
    receives ``(loss, model.copy())`` of every evaluation.  Returns the final maps."""
    from scipy.optimize import minimize
    n = ny * nx
    state = {"loss0": None}

    def maps(p):
        return [to_model(p[i * n:(i + 1) * n].reshape(ny, nx)) for i, (to_model, _, _, _) in enumerate(blocks)]

    def fun(p):
        m = maps(p)
        model = m[0] if len(m) == 1 else np.stack(m)
        loss, grad = loss_grad(model)
        if np.shape(grad) != model.shape:
            raise ValueError(f"loss_grad must return a gradient with the shape of its argument {model.shape}")
        if state["loss0"] is None:
            state["loss0"] = float(loss)
        if history is not None:
            history.append((float(loss), model.copy()))
        scale = 1.0 / state["loss0"]
        g = np.asarray(grad, dtype=np.float64).reshape(len(blocks), n)
        return float(loss) * scale, np.concatenate([g[i] * (dmodel_dp * scale) for i, (_, dmodel_dp, _, _) in enumerate(blocks)])

    p0 = np.concatenate([b[2] for b in blocks])
    bounds = None if all(b[3] is None for b in blocks) else [(b[3], None) for b in blocks for _ in range(n)]
    res = minimize(fun, p0, jac=True, method="L-BFGS-B", bounds=bounds,
                   options=dict(maxiter=int(maxiter), maxcor=int(history_size), gtol=float(tol)))
    return maps(res.x)


def run_lbfgs_joint_fwi(xi, yi, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, a0, L_PML, mask_indices, *, kappa_init=0.0,
                        kappa_scale=None, maxiter=1, tol=1e-5, history_size=10, dtype="c64", bde=None, stencil="python",
                        engine="auto", history=None, loss_grad=None, pert_scale=1e-2, gradient="reference"):
    """L-BFGS on sound speed and attenuation together (``fwi_joint_loss_function``); returns ``(c, kappa)``, both (Ny, Nx).

    SciPy's L-BFGS-B with the bound ``kappa >= 0``, on the problem non-dimensionalised per block: the slowness as in
    ``run_lbfgs_fwi`` (``p_s = (s / s0 - 1) / pert_scale``), the attenuation as ``p_kappa = kappa / kappa_scale`` (default
    ``kappa_scale``: the kappa of 0.5 dB/(cm MHz), ``geometry.db_cm_mhz_to_kappa(0.5)``), and the objective
    ``loss / loss(start)``; ``tol`` applies to the projected gradient of that scaled problem.  ``kappa_init`` is a scalar or an
    (Ny, Nx) map.

    ``loss_grad(params) -> (loss, grad)`` with ``params`` (2, Ny, Nx) float64 = [slowness, kappa] replaces the objective (the
    parity test drives the same optimiser with the oracle's); ``history`` receives ``(loss, params.copy())`` of every
    evaluation.  ``gradient`` is the gradient mode of ``fwi_joint_loss_function``.
    """
    from .geometry import db_cm_mhz_to_kappa
    ny, nx = _to_np(yi).size, _to_np(xi).size
    num_elements = int(SRC.shape[2]) if SRC is not None else 0  # unused when ``loss_grad`` is injected
    c0 = np.asarray(_to_np(c_init), dtype=np.float64)
    s0 = 1.0 / float(c0.mean())
    ks = float(db_cm_mhz_to_kappa(0.5) if kappa_scale is None else kappa_scale)
    real = np.float32 if dtype == "c64" else np.float64
    if loss_grad is None:
        def loss_grad(params):
            return fwi_joint_loss_function(params.astype(real), xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab,
                                           mask_indices, num_elements, dtype=dtype, bde=bde, stencil=stencil, engine=engine,
                                           gradient=gradient)

    kappa_block = (lambda p: ks * p), ks, (np.asarray(_to_np(kappa_init), dtype=np.float64) * np.ones((ny, nx)) / ks).ravel(), 0.0
    slow, kappa = _lbfgs_blocks(loss_grad, [_slowness_block(c0, s0, pert_scale, ny, nx), kappa_block], ny, nx, maxiter, tol,
                                history_size, history)
    return 1.0 / slow, kappa


def gauss_newton_fwi(xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, Niter, a0, L_PML, mask_indices, *,
                     cg_iters=8, cg_tol=1e-2, damping=0.0, max_backtracks=4, dtype="c64", bde=None, stencil="python", device=0,
                     engine="auto", history=None, loss_grad=None, hvp=None, gradient="reference"):
    """Truncated Gauss-Newton FWI on the slowness, with the arguments of ``nonlinear_conjugate_gradient``; returns the sound
    speed (Ny, Nx) as a NumPy array.

    Per outer iteration: conjugate gradients from ``p = 0`` on ``(H_GN + mu I) p = -g`` with at most ``cg_iters`` Gauss-Newton
    products (``fwi_gauss_newton_product``), stopped early when ``|r| <= cg_tol |g|`` or the curvature is not positive;
    ``mu = damping * <g, H_GN g> / <g, g>`` comes from the first product.  Then ``s + p`` is tried and the step halved up to
    ``max_backtracks`` times until the loss decreases; without a decrease the driver stops.  One evaluation (one
    factorisation) per trial; the products reuse the factorisation of the accepted trial.  With ``cg_iters=1`` and
    ``damping=0`` the first iteration is the reference NCG's first iteration (steepest descent with the linearised exact step,
    ``nonlinearcg.py:268-301``).

    ``loss_grad(slow) -> (loss, grad)`` and ``hvp(v) -> hv`` (products at the point of the last ``loss_grad`` call) replace
    the GPU objective; they receive (Ny, Nx) float64 torch tensors and may return tensors or NumPy arrays.  The vector
    algebra is float64 torch on the device of the first gradient.  ``history`` (a list) receives one dict per outer
    iteration: loss, CG iterations, the quadratic-model value ``q(p_k) = <g,p_k>/2 - <p_k,r_k>/2`` of every CG iterate, mu,
    the accepted step, cumulative evaluation and product counts, the velocity range, and ``stop`` when the driver stops.
    ``gradient``: the linearisation of the gradient and the products, ``"reference"`` or ``"discrete"``
    (``fwi_gauss_newton_product``).
    """
    import torch
    ny, nx = _to_np(yi).size, _to_np(xi).size
    if loss_grad is None or hvp is None:
        loss_grad, _, hvp = _gpu_callables(False, xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, f, a0, L_PML,
                                           mask_indices, dtype, bde, stencil, device, engine, gradient)
    c0 = np.asarray(_to_np(c_init), dtype=np.float64) * np.ones((ny, nx))
    s = _gauss_newton_loop(torch.as_tensor(1.0 / c0), loss_grad, hvp, Niter, cg_iters, cg_tol, damping, max_backtracks, history,
                           slow_of=lambda x: x)
    return (1.0 / s).cpu().numpy()


def _f64(a, dv):
    import torch
    return a.detach().to(dv, torch.float64) if torch.is_tensor(a) else torch.as_tensor(np.asarray(a, dtype=np.float64)).to(dv)


def _gauss_newton_loop(x, loss_grad, hvp, Niter, cg_iters, cg_tol, damping, max_backtracks, history, slow_of, scale=None,
                       project=None):
    """The outer loop of ``gauss_newton_fwi`` and ``gauss_newton_joint_fwi`` on the model ``x`` (float64 torch): CG on
    ``(D H_GN D + mu I) p = -D g`` in the scaled variables, trial ``project(x + step D p)`` with step halving.  ``scale`` is
    ``D`` (a tensor of ``x``'s shape; None: the identity, no arithmetic), ``project(x) -> (x, clipped node count)`` (None: no
    projection), ``slow_of(x)`` the slowness map whose range the history reports.  Returns the final ``x``."""
    import torch
    shape = tuple(x.shape)
    D = (lambda a: a) if scale is None else (lambda a: scale * a)
    loss, g = loss_grad(x)
    dv = g.device if torch.is_tensor(g) else torch.device("cpu")
    x, g, loss = x.to(dv), _f64(g, dv).reshape(shape), float(loss)
    if scale is not None:
        scale = scale.to(dv)
    nevals, nprods = 1, 0
    dot = lambda a, b: float(torch.sum(a * b))
    for it in range(int(Niter)):
        rec = dict(it=it, loss=loss)
        gs = D(g)
        gg = dot(gs, gs)
        p = torch.zeros_like(g)
        r, d, rr = -gs, -gs, gg
        qs, mu, k = [], 0.0, 0
        while k < int(cg_iters):
            Hd = D(_f64(hvp(D(d)), dv).reshape(shape))
            nprods += 1
            if k == 0:
                mu = float(damping) * dot(d, Hd) / gg  # d = -D g
            Ad = Hd + mu * d
            curv = dot(d, Ad)
            if not curv > 0:
                break
            a = rr / curv
            p = p + a * d
            r = r - a * Ad
            k += 1
            qs.append(0.5 * dot(gs, p) - 0.5 * dot(p, r))
            rr_new = dot(r, r)
            if math.sqrt(rr_new) <= float(cg_tol) * math.sqrt(gg):
                break
            d = r + (rr_new / rr) * d
            rr = rr_new
        rec.update(cg_iters=k, q=qs, mu=mu)
        step, accepted, clipped = 1.0, False, 0
        if k > 0:
            dp = D(p)
            for _ in range(int(max_backtracks) + 1):
                trial = x + step * dp
                if project is not None:
                    trial, clipped = project(trial)
                lt, gt = loss_grad(trial)
                nevals += 1
                if float(lt) < loss:
                    x, loss, g, accepted = trial, float(lt), _f64(gt, dv).reshape(shape), True
                    break
                step *= 0.5
        s = slow_of(x)
        rec.update(step=step if accepted else 0.0, evals=nevals, products=nprods, vel_min=float(1.0 / s.max()),
                   vel_max=float(1.0 / s.min()))
        if project is not None:
            rec["clipped"] = clipped
        if not accepted:
            rec["stop"] = ("no positive curvature along -g" if k == 0 else
                           f"no loss decrease after {int(max_backtracks)} step halvings")
        if history is not None:
            history.append(rec)
        if not accepted:
            break
    return x


def _joint_setup(ny, nx, c_init, kappa_init, kappa_scale, pert_scale):
    """Start model x0 (2, Ny, Nx) = [1/c_init, kappa_init] and the block scaling D = diag(s0 pert_scale, kappa_scale) of
    ``run_lbfgs_joint_fwi``, both float64 torch (CPU)."""
    import torch
    from .geometry import db_cm_mhz_to_kappa
    c0 = np.asarray(_to_np(c_init), dtype=np.float64) * np.ones((ny, nx))
    s0 = 1.0 / float(c0.mean())
    ks = float(db_cm_mhz_to_kappa(0.5) if kappa_scale is None else kappa_scale)
    k0 = np.asarray(_to_np(kappa_init), dtype=np.float64) * np.ones((ny, nx))
    x0 = torch.as_tensor(np.stack([1.0 / c0, k0]))
    D = torch.as_tensor(np.stack([np.full((ny, nx), s0 * float(pert_scale)), np.full((ny, nx), ks)]))
    return x0, D


def _project_kappa(x):
    """kappa <- max(kappa, 0) on a (2, Ny, Nx) model; returns (model, number of clipped nodes)."""
    import torch
    neg = x[1] < 0
    return torch.stack([x[0], torch.clamp(x[1], min=0.0)]), int(neg.sum())


def _gpu_callables(lossy, xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, f, a0, L_PML, mask_indices, dtype, bde,
                   stencil, device, engine, gradient="reference"):
    """GPU objective of the drivers on float64 torch models, (Ny, Nx) slowness maps or, ``lossy``, (2, Ny, Nx) = [s, kappa]:
    loss_grad(x), and the line search and the Gauss-Newton product at the point of the last loss_grad call."""
    import torch
    freqs = np.atleast_1d(np.asarray(_to_np(f), dtype=np.float64)).ravel()
    dv = torch.device(f"cuda:{device}")
    real = torch.float32 if dtype == "c64" else torch.float64
    rec = torch.as_tensor(_to_np(REC_DATA)).to(dv).reshape(freqs.size, len(_to_np(tx_include)), -1).contiguous()
    state = {}
    fargs = (xi, yi, rec, SRC, freqs, a0, L_PML, tx_include, ind_matlab, mask_indices, numElements)
    kw = dict(dtype=dtype, bde=bde, stencil=stencil, engine=engine, gradient=gradient)

    # the module functions are looked up at call time: tests record the evaluation points by replacing them
    def loss_grad(x):
        state["x"] = x.to(dv, real).contiguous()
        loss, grad = (fwi_joint_loss_function if lossy else fwi_loss_function)(state["x"], *fargs, **kw)
        return float(loss), grad

    def linesearch(sd):
        plan, _ = _fwi_plan(xi, yi, rec, SRC, freqs, a0, L_PML, ind_matlab, mask_indices, dtype, stencil, device, engine, gradient)
        sdt = sd.to(dv, real)
        nd = plan._linesearch(*((sdt[0].contiguous(), sdt[1].contiguous()) if lossy else (sdt.contiguous(), None)))
        return float(nd[0]), float(nd[1])

    def hvp(v):
        product = fwi_joint_gauss_newton_product if lossy else fwi_gauss_newton_product
        return product(state["x"], v.to(dv, real).contiguous(), *fargs, **kw)

    return loss_grad, linesearch, hvp


def nonlinear_conjugate_gradient_joint(xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, Niter, a0, L_PML,
                                       mask_indices, *, kappa_init=0.0, kappa_scale=None, pert_scale=1e-2, dtype="c64", bde=None,
                                       stencil="python", device=0, engine="auto", history=None, loss_grad=None,
                                       linesearch=None, gradient="reference"):
    """The reference's NCG loop (``nonlinear_conjugate_gradient``) on sound speed and attenuation together; returns ``(c,
    kappa)`` as NumPy (Ny, Nx) arrays.

    It works on the block-scaled variables of ``run_lbfgs_joint_fwi``, ``x = D x~`` with ``D = diag(s0 pert_scale,
    kappa_scale)``: Hestenes-Stiefel on the scaled gradient ``g~ = D g`` (beta = 0 at the first iteration, as in the
    reference), the physical direction ``sd = D d~``, the linearised exact step ``num / den`` of the joint line search
    (``ust_ncg_linesearch_lossy``: ``num = -<sd, g>``, ``den = |J sd|^2``), and ``kappa <- max(kappa, 0)`` after every
    step.  One evaluation (one factorisation) and one line search per iteration.

    ``loss_grad(x) -> (loss, grad)`` and ``linesearch(sd) -> (num, den)`` (at the point of the last ``loss_grad`` call)
    replace the GPU objective; they receive (2, Ny, Nx) float64 torch tensors = [slowness, kappa].  ``history`` (a list)
    receives one dict per iteration: loss, gradient norm, beta, step, velocity range, largest kappa and clipped nodes.
    ``gradient`` is the linearisation of the gradient and the line search (``fwi_joint_loss_function``).
    """
    import torch
    ny, nx = _to_np(yi).size, _to_np(xi).size
    if loss_grad is None or linesearch is None:
        loss_grad, linesearch, _ = _gpu_callables(True, xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, f, a0, L_PML,
                                                  mask_indices, dtype, bde, stencil, device, engine, gradient)
    x, D = _joint_setup(ny, nx, c_init, kappa_init, kappa_scale, pert_scale)
    dot = lambda a, b: float(torch.sum(a * b))
    d = gprev = None
    for it in range(int(Niter)):
        loss, g = loss_grad(x)
        if it == 0:
            dv = g.device if torch.is_tensor(g) else torch.device("cpu")
            x, D = x.to(dv), D.to(dv)
        gt = D * _f64(g, dv).reshape(2, ny, nx)  # scaled gradient
        if it == 0:
            beta = 0.0
        else:
            dg = gt - gprev
            beta = dot(gt, dg) / dot(d, dg)
        d = -gt if it == 0 else beta * d - gt
        sd = D * d
        num, den = linesearch(sd)
        step = float(num) / float(den)
        x, clipped = _project_kappa(x + step * sd)
        if history is not None:
            history.append(dict(it=it, loss=float(loss), grad_norm=math.sqrt(dot(gt, gt)), beta=beta, step=step,
                                vel_min=float(1.0 / x[0].max()), vel_max=float(1.0 / x[0].min()), kappa_max=float(x[1].max()),
                                clipped=clipped))
        gprev = gt
    x = x.cpu().numpy()
    return 1.0 / x[0], x[1]


def gauss_newton_joint_fwi(xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, Niter, a0, L_PML, mask_indices, *,
                           kappa_init=0.0, kappa_scale=None, pert_scale=1e-2, cg_iters=8, cg_tol=1e-2, damping=0.0,
                           max_backtracks=4, dtype="c64", bde=None, stencil="python", device=0, engine="auto", history=None,
                           loss_grad=None, hvp=None, gradient="reference"):
    """Truncated Gauss-Newton on sound speed and attenuation together; returns ``(c, kappa)`` as NumPy (Ny, Nx) arrays.

    The outer loop of ``gauss_newton_fwi`` on the block-scaled variables of ``run_lbfgs_joint_fwi`` (``D = diag(s0 pert_scale,
    kappa_scale)``): CG on ``(D H_GN D + mu I) p~ = -D g`` with the joint products (``fwi_joint_gauss_newton_product``), whose
    off-diagonal blocks ``H_s,kappa`` couple the two maps from the first product; the trial ``x + step D p~`` has kappa
    clipped at 0 and is backtracked as in ``gauss_newton_fwi``.  With ``cg_iters=1`` and ``damping=0`` an iteration is the
    first iteration of ``nonlinear_conjugate_gradient_joint``.

    ``loss_grad(x) -> (loss, grad)`` and ``hvp(v) -> hv`` (at the point of the last ``loss_grad`` call) replace the GPU
    objective; they receive (2, Ny, Nx) float64 torch tensors = [slowness, kappa].  ``history`` receives the records of
    ``gauss_newton_fwi`` plus ``clipped``, the number of kappa nodes clipped in the last trial.  ``gradient`` is the
    linearisation of the gradient and the products (``fwi_joint_gauss_newton_product``).
    """
    import torch
    ny, nx = _to_np(yi).size, _to_np(xi).size
    if loss_grad is None or hvp is None:
        loss_grad, _, hvp = _gpu_callables(True, xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, f, a0, L_PML,
                                           mask_indices, dtype, bde, stencil, device, engine, gradient)
    x0, D = _joint_setup(ny, nx, c_init, kappa_init, kappa_scale, pert_scale)
    x = _gauss_newton_loop(x0, loss_grad, hvp, Niter, cg_iters, cg_tol, damping, max_backtracks, history, slow_of=lambda x: x[0],
                           scale=D, project=_project_kappa)
    x = x.cpu().numpy()
    return 1.0 / x[0], x[1]


# -------------------------------------------------------------------------------------------------
# SURVEY section 8(f) rank 4: time-domain synthesis and the low-to-high frequency schedule
# -------------------------------------------------------------------------------------------------
def hanning(n):
    """MATLAB ``hanning(n)`` (symmetric Hann window without the zero end points), the frequency response of
    ``Lecture19_Fwi/TimeDomainSimulation.m:33``."""
    k = np.arange(1, int(n) + 1, dtype=np.float64)
    return 0.5 * (1.0 - np.cos(2.0 * np.pi * k / (int(n) + 1)))


def idtft(WVFIELD_F, f, resp_freq, time, df=None, *, device=0):
    """Inverse discrete-time Fourier transform of a stack of frequency-domain wavefields on an arbitrary time axis
    (``TimeDomainSimulation.m:54-56``; not an inverse FFT): ``WVFIELD_F`` (Ny, Nx, Nf) complex -> (Ny, Nx, Nt) with
    ``out[..., t] = sum_k exp(2j*pi*f[k]*time[t]) * df * resp_freq[k] * WVFIELD_F[..., k]`` (``ust_idtft``).

    A torch CUDA tensor in gives a torch CUDA tensor out (a permuted view of the (Nt, Ny*Nx) result); NumPy in, NumPy out.
    """
    import ctypes as C
    import torch
    from . import _lib
    f = np.ascontiguousarray(np.asarray(_to_np(f), dtype=np.float64).ravel())
    tm = np.ascontiguousarray(np.asarray(_to_np(time), dtype=np.float64).ravel())
    resp = np.ascontiguousarray(np.asarray(_to_np(resp_freq), dtype=np.float64).ravel())
    if resp.size != f.size:
        raise ValueError("resp_freq and f must have the same length")
    if df is None:
        df = float(f[1] - f[0]) if f.size > 1 else 1.0
    on_dev = _is_torch(WVFIELD_F) and WVFIELD_F.is_cuda
    W = WVFIELD_F if on_dev else torch.as_tensor(_to_np(WVFIELD_F)).to(f"cuda:{device}")
    if W.dtype not in (torch.complex64, torch.complex128):
        W = W.to(torch.complex64)
    ny, nx, nf = W.shape
    if nf != f.size:
        raise ValueError("last axis of WVFIELD_F must match f")
    U = W.permute(2, 0, 1).reshape(nf, ny * nx).contiguous()  # frequency-major stack
    out = torch.empty((tm.size, ny * nx), dtype=U.dtype, device=U.device)
    pd = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    with torch.cuda.device(U.device):
        rc = _lib.lib().ust_idtft(0 if U.dtype == torch.complex64 else 1, C.c_void_p(U.data_ptr()), nf, ny * nx, pd(f), pd(resp),
                                  float(df), pd(tm), tm.size, C.c_void_p(out.data_ptr()),
                                  C.c_void_p(torch.cuda.current_stream(U.device).cuda_stream))
    _lib.check(rc, "ust_idtft")
    res = out.reshape(tm.size, ny, nx).permute(1, 2, 0)
    return res if on_dev else res.cpu().numpy()


def time_domain_simulation(xi, yi, C_map, src, f, resp_freq, time, a0, L_PML, *, dtype="c64", stencil="python",
                           engine="auto", device=0, batch=16, kappa=None):
    """``Lecture19_Fwi/TimeDomainSimulation.m:36-56`` on the GPU path: one forward solve per frequency for the source
    ``src`` (Ny, Nx) of one transmitting element, ``batch`` frequencies factorised per launch sequence, then the inverse
    discrete-time Fourier transform to the time axis ``time``.  Returns NumPy ``(WVFIELD_F (Ny, Nx, Nf), WVFIELD_T (Ny, Nx, Nt))``.
    ``kappa`` ((Ny, Nx) attenuation slowness, s/m): lossy medium, attenuation linear in frequency (``solve_helmholtz``).
    """
    import torch
    xh, yh = _to_np(xi).astype(np.float64).ravel(), _to_np(yi).astype(np.float64).ravel()
    nx, ny = xh.size, yh.size
    f = np.asarray(_to_np(f), dtype=np.float64).ravel()
    batch = max(1, min(int(batch), f.size))
    plan = get_plan(nx, ny, dtype, device, batch, 1, stencil, False, engine)
    plan.set_grid(xh, yh, float(a0), float(L_PML))
    plan._factor_key = None
    dv = torch.device(f"cuda:{device}")
    vel = torch.as_tensor(_to_np(C_map)).to(device=dv, dtype=plan.treal).reshape(ny, nx).contiguous()
    kap = None if kappa is None else torch.as_tensor(_to_np(kappa)).to(device=dv, dtype=plan.treal).reshape(ny, nx).contiguous()
    rhs0 = torch.as_tensor(_to_np(src)).to(device=dv, dtype=plan.tcplx).reshape(ny * nx, 1).contiguous()
    U = torch.empty((f.size, ny * nx), dtype=plan.tcplx, device=dv)
    for k0 in range(0, f.size, batch):
        fb = f[k0:k0 + batch]
        plan.factor(vel, fb, kappa=kap)
        for i in range(fb.size):
            X = rhs0.clone()
            plan.solve(X, i, False)
            U[k0 + i] = X[:, 0]
    WF = U.reshape(f.size, ny, nx).permute(1, 2, 0)
    WT = idtft(WF, f, resp_freq, time)
    return WF.cpu().numpy(), WT.cpu().numpy()


def channel_data(WVFIELD_T, x_idx, y_idx):
    """``channelData(t, e) = WVFIELD_T(y_idx(e), x_idx(e), t)`` (``TimeDomainSimulation.m:72-75``; 0-based indices)."""
    W = _to_np(WVFIELD_T)
    return W[np.asarray(y_idx), np.asarray(x_idx), :].T


def continuation_stages(f, nstages):
    """Low-to-high frequency schedule: ``nstages`` contiguous groups of ascending frequency (index arrays into ``f``).
    The reference states the rule only (``SimulateData.m:29-30`` "Use 0.1-0.6 MHz ... cycle skipping"; slides p.24)."""
    order = np.argsort(np.asarray(_to_np(f), dtype=np.float64), kind="stable")
    return [np.sort(g) for g in np.array_split(order, int(nstages)) if g.size]


def frequency_continuation(xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, stages, Niter,
                           a0, L_PML, mask_indices, *, dtype="c64", stencil="python", device=0, engine="auto", history=None,
                           method="ncg", gradient="reference"):
    """Multi-frequency FWI by frequency continuation: for every stage (an index array into ``f``, see
    ``continuation_stages``) ``Niter`` NCG iterations (``nonlinear_conjugate_gradient``; ``method="gn"``: ``Niter`` outer
    iterations of ``gauss_newton_fwi`` with its default settings) on the joint objective of that stage's frequencies, each
    stage starting from the sound speed the previous one ended with.  ``REC_DATA`` is (Nf, Nt, E).  Returns the final sound
    speed (Ny, Nx); ``history`` (a list) receives one list of per-iteration records per stage.  ``gradient`` is passed to
    the stage driver.
    """
    if method not in ("ncg", "gn"):
        raise ValueError("method must be 'ncg' or 'gn'")

    def stage(vel, rec, f, h):
        if method == "gn":
            return gauss_newton_fwi(xi, yi, numElements, rec, SRC, tx_include, ind_matlab, vel, f, Niter, a0, L_PML, mask_indices,
                                    dtype=dtype, stencil=stencil, device=device, engine=engine, history=h, gradient=gradient)
        return nonlinear_conjugate_gradient(xi, yi, numElements, rec, SRC, tx_include, ind_matlab, vel, f, Niter, a0, L_PML,
                                            mask_indices, dtype=dtype, stencil=stencil, device=device, history=h,
                                            return_fields=False, engine=engine, gradient=gradient)[0]

    return _continuation(REC_DATA, f, stages, history, c_init, stage)


def _continuation(REC_DATA, f, stages, history, model, stage):
    """The stage loop of the continuation drivers: ``model = stage(model, REC_DATA[idx], f[idx], h)`` for every stage ``idx``,
    with ``h`` the stage's history list (None without ``history``).  Returns the final model."""
    f = np.asarray(_to_np(f), dtype=np.float64).ravel()
    rec = _to_np(REC_DATA)
    if rec.ndim != 3 or rec.shape[0] != f.size:
        raise ValueError("REC_DATA must be (Nf, Nt, E) with Nf == len(f)")
    prev = None
    for st in stages:
        idx = np.asarray(st, dtype=np.int64).ravel()
        if prev is not None and prev != idx.size:
            clear_plans()  # a plan is sized for its number of frequencies; do not keep two factor stores alive
        prev = idx.size
        h = [] if history is not None else None
        model = stage(model, rec[idx], f[idx], h)
        if history is not None:
            history.append(h)
    return model


def joint_frequency_continuation(xi, yi, numElements, REC_DATA, SRC, tx_include, ind_matlab, c_init, f, stages, Niter, a0, L_PML,
                                 mask_indices, *, kappa_init=0.0, dtype="c64", stencil="python", device=0, engine="auto",
                                 history=None, method="ncg", gradient="reference"):
    """``frequency_continuation`` for sound speed and attenuation together: per stage ``Niter`` iterations of
    ``nonlinear_conjugate_gradient_joint`` (``method="ncg"``), outer iterations of ``gauss_newton_joint_fwi`` (``"gn"``) or
    L-BFGS-B iterations of ``run_lbfgs_joint_fwi`` (``"lbfgs"``), each with its default settings and each stage starting
    from the maps the previous one ended with.  Returns ``(c, kappa)``; ``history`` (a list) receives one list of records per
    stage (for ``"lbfgs"``, ``(loss, params)`` of every evaluation).  ``gradient`` is passed to the stage driver.
    """
    if method not in ("ncg", "gn", "lbfgs"):
        raise ValueError("method must be 'ncg', 'gn' or 'lbfgs'")

    def stage(model, rec, f, h):
        vel, kap = model
        if method == "lbfgs":
            return run_lbfgs_joint_fwi(xi, yi, rec, SRC, tx_include, ind_matlab, vel, f, a0, L_PML, mask_indices, kappa_init=kap,
                                       maxiter=Niter, dtype=dtype, stencil=stencil, engine=engine, history=h, gradient=gradient)
        drv = gauss_newton_joint_fwi if method == "gn" else nonlinear_conjugate_gradient_joint
        return drv(xi, yi, numElements, rec, SRC, tx_include, ind_matlab, vel, f, Niter, a0, L_PML, mask_indices, kappa_init=kap,
                   dtype=dtype, stencil=stencil, device=device, engine=engine, history=h, gradient=gradient)

    return _continuation(REC_DATA, f, stages, history, (c_init, kappa_init), stage)
