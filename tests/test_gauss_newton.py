"""Gauss-Newton Hessian-vector products H_GN v = Re(J^H J v) and the truncated Gauss-Newton driver.

J is the linearisation the gradient is built from (nonlinearcg.py:258,279; source estimates held fixed), so the gradient is
Re(J^H diff) and the NCG line-search scalars are den = |J sd|^2, num = -<sd, grad>.  The CPU tests pin these identities on
the oracle and drive the one driver with oracle callables; the GPU tests compare the device product with the oracle and with
the device's own gradient and line search."""
import numpy as np
import pytest

from common import bde_for, observed_data, rel, small_case
from oracle import fwi as ofwi
from oracle import helmholtz as oh
from oracle.helmholtz import _CPLX, _REAL

GRAD_TOL = 1e-4


def gn_hvp_ref(params, v, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements,
               dtype="c64", bde=None, stencil="python", threads=1, return_jv=False):
    """Reference Gauss-Newton product ``H_GN v = Re(J^H J v)`` for one frequency, with ``params``' shape, built from the
    oracle's pieces and the lines of ``oracle.fwi.fwi_loss_and_grad``.

    ``(J v)_t`` is the perturbation solve ``H^-1(-VIRT_t * v)`` (``nonlinearcg.py:279-281``) gathered at the kept receivers,
    with ``VIRT_t = 2 w^2 s alpha_t u_t`` (``:258``) and the source estimate ``alpha`` held fixed; ``J^H r`` is the gradient's
    adjoint-source scatter and adjoint solve (``:248-265``), so ``fwi_loss_and_grad``'s gradient is ``Re(J^H diff)``.
    ``return_jv`` also returns ``J v`` (Nt, Nmask) in mask order.
    """
    R, Cx = _REAL[dtype], _CPLX[dtype]
    Nyi, Nxi = np.asarray(yi).size, np.asarray(xi).size
    Nt = np.asarray(tx_include).size
    params = np.asarray(params, dtype=R)
    SLOW = params.reshape(Nyi, Nxi)
    V = np.asarray(v, dtype=R).reshape(Nyi, Nxi)
    VEL = (R(1) / SLOW).astype(R)
    REC_DATA = np.asarray(REC_DATA).astype(Cx)
    solve = ofwi._solver(xi, yi, VEL, f, a0, L_PML, dtype, bde, stencil, True, threads)

    WV = solve(SRC, False)  # fwi_loss_function.py:53
    rec_sim, global_inds = ofwi.receiver_gather(WV, ind_matlab, mask_indices)
    rec = np.take_along_axis(REC_DATA, mask_indices, axis=1)
    SRC_EST = ofwi.estimate_src_strength_batched(rec_sim, rec)  # :78
    WV = (WV * SRC_EST[None, None, :]).astype(Cx)  # :81
    w = R(2 * np.pi) * R(f)
    VIRT = (R(2) * w**2) * SLOW[:, :, None] * WV  # nonlinearcg.py:258

    PERT = solve((-VIRT * V[:, :, None]).astype(Cx), False)  # :279-281
    jv, _ = ofwi.receiver_gather(PERT, ind_matlab, mask_indices)  # :284-293
    flat_adj = np.zeros((Nt, Nyi * Nxi), dtype=Cx)
    flat_adj[np.arange(Nt)[:, None], global_inds] = jv  # :249-250
    ADJ_SRC = np.transpose(flat_adj.reshape(Nt, Nxi, Nyi), (2, 1, 0))
    ADJ_WV = solve(ADJ_SRC, True)  # :263
    hv = np.sum(-np.real(np.conj(VIRT) * ADJ_WV), axis=2).astype(R).reshape(params.shape)  # :264-265
    return (hv, jv) if return_jv else hv


def _case(n=48, nelem=32):
    geom, f, vel_true = small_case(n, nelem)
    c0 = np.full((n, n), 1480.0)
    bde = bde_for(geom, c0, f)
    rec = observed_data(geom, f, vel_true, bde=bde_for(geom, vel_true, f))
    args = (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab,
            geom.mask_indices, geom.num_elements)
    return geom, f, c0, bde, rec, args


def _perturbations(geom, c0, seeds=(5, 6)):
    """Model-like slowness perturbations: smooth blobs of the kind an FWI update has."""
    from waveforminversionust_b200 import geometry as G
    return [1.0 / G.blob_model(geom, c0=float(c0.mean()), dc=20.0, seed=s) - 1.0 / c0 for s in seeds]


# ---------------------------------------------------------------------------------------------------------------------
# oracle identities (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_adjoint_identity():
    """Re<J w, diff> = <w, grad>: the gradient is J^H applied to the residual, for the J of gn_hvp_ref."""
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    loss, grad, fl = ofwi.fwi_loss_and_grad(slow, *args, dtype="c128", bde=bde, return_fields=True)
    diff = fl["rec_sim"] - np.take_along_axis(rec, geom.mask_indices, axis=1)
    for w in _perturbations(geom, c0):
        _, jw = gn_hvp_ref(slow, w, *args, dtype="c128", bde=bde, return_jv=True)
        lhs, rhs = float(np.real(np.vdot(jw, diff))), float(np.sum(w * grad))
        print(f"Re<Jw, diff> = {lhs:.15e}, <w, grad> = {rhs:.15e}")
        assert abs(lhs - rhs) <= 1e-10 * abs(rhs)


def test_oracle_symmetry_and_positive_semidefinite():
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    v, w = _perturbations(geom, c0)
    hv, jv = gn_hvp_ref(slow, v, *args, dtype="c128", bde=bde, return_jv=True)
    hw = gn_hvp_ref(slow, w, *args, dtype="c128", bde=bde)
    a, b = float(np.sum(w * hv)), float(np.sum(v * hw))
    assert abs(a - b) <= 1e-10 * max(abs(a), abs(b))
    vhv, jv2 = float(np.sum(v * hv)), float(np.vdot(jv, jv).real)
    assert jv2 > 0 and abs(vhv - jv2) <= 1e-10 * jv2


def test_oracle_jv_against_finite_differences():
    """J v against the central difference of alpha P u(s +- eps v) (alpha fixed), v supported inside the PML-free interior.
    J's virtual source 2 w^2 s alpha u leaves out the stencil's mass weights and the PML factor C (as the reference's gradient
    does), so J is not the derivative of the discrete forward map.  Inside the interior the gap is almost exactly one complex
    scale factor (measured: 1.1233 + 0.0004i with 6.4e-5 left after it, 12.3 % rel-L2 without it, on this 48 x 48 case);
    the asserted bounds record that."""
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64))
    v = np.exp(-(X ** 2 + Y ** 2) / (2 * 0.015 ** 2)) * slow * 1e-2
    _, jv = gn_hvp_ref(slow, v, *args, dtype="c128", bde=bde, return_jv=True)
    _, _, fl = ofwi.fwi_loss_and_grad(slow, *args, dtype="c128", bde=bde, return_fields=True)
    alpha = fl["SRC_EST"]

    def apu(s):
        fac = oh.HelmholtzFactor(geom.xi, geom.yi, 1.0 / s, f, geom.a0, geom.L_PML, "c128", bde=bde)
        return ofwi.receiver_gather(fac.solve(geom.dense_src(np.complex128)) * alpha[None, None, :], geom.ind_matlab,
                                    geom.mask_indices)[0]

    eps = 1e-3
    fd = (apu(slow + eps * v) - apu(slow - eps * v)) / (2 * eps)
    c = np.vdot(fd, jv) / np.vdot(fd, fd)
    e_raw, e_scaled = rel(jv, fd), rel(jv, c * fd)
    print(f"J v vs central difference: rel-L2 {e_raw:.3e}; best complex scale {c:.6f}, rel-L2 after it {e_scaled:.3e}")
    assert e_raw < 0.15 and abs(c - 1.1233) < 5e-3 and e_scaled < 1e-3


# ---------------------------------------------------------------------------------------------------------------------
# the driver with injected oracle callables (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_callables(args, bde, dtype="c128", points=None):
    st = {}

    def loss_grad(slow):
        st["slow"] = slow.cpu().numpy()
        if points is not None:
            points.append(st["slow"].copy())
        return ofwi.fwi_loss_and_grad(st["slow"], *args, dtype=dtype, bde=bde)

    def hvp(v):
        return gn_hvp_ref(st["slow"], v.cpu().numpy(), *args, dtype=dtype, bde=bde)

    return loss_grad, hvp


def _driver_args(geom, f, rec, niter):
    return (geom.xi, geom.yi, geom.num_elements, rec, geom.dense_src(), geom.tx_include, geom.ind_matlab, 1480.0, f, niter,
            geom.a0, geom.L_PML, geom.mask_indices)


def test_driver_with_one_cg_step_is_the_ncg_first_iteration():
    """The first CG iterate -(<g,g>/<g,Hg>) g is the reference NCG's linearised exact step along -g."""
    from waveforminversionust_b200 import api
    geom, f, c0, bde, rec, args = _case()
    VELo = ofwi.nonlinear_conjugate_gradient_vectorized(*_driver_args(geom, f, rec, 1), dtype="c128", bde=bde)[0]
    lg, hvp = _oracle_callables(args, bde)
    hist = []
    vel = api.gauss_newton_fwi(*_driver_args(geom, f, None, 1), cg_iters=1, damping=0.0, dtype="c128", history=hist,
                               loss_grad=lg, hvp=hvp)
    print(hist)
    assert hist[0]["cg_iters"] == 1 and hist[0]["step"] == 1.0 and hist[0]["products"] == 1
    assert rel(vel, VELo) < 1e-9


def test_driver_quadratic_model_decreases():
    from waveforminversionust_b200 import api
    geom, f, c0, bde, rec, args = _case()
    lg, hvp = _oracle_callables(args, bde)
    hist = []
    api.gauss_newton_fwi(*_driver_args(geom, f, None, 2), cg_iters=4, cg_tol=1e-6, dtype="c128", history=hist,
                         loss_grad=lg, hvp=hvp)
    for h in hist:
        print({k: h[k] for k in ("it", "loss", "cg_iters", "q", "step", "evals", "products")})
        q = h["q"]
        assert len(q) >= 2 and q[0] < 0 and all(b < a for a, b in zip(q, q[1:]))
    assert hist[1]["loss"] < hist[0]["loss"]


def test_frequency_continuation_rejects_an_unknown_method():
    from waveforminversionust_b200 import api
    with pytest.raises(ValueError, match="method"):
        api.frequency_continuation(None, None, 0, None, None, None, None, 1480.0, [1.0], [[0]], 1, 0.0, 0.0, None, method="lbfgs")


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_():
    import torch
    return torch


def _dev_case(torch_, n, nelem, dtype):
    import waveforminversionust_b200 as w
    geom, f, c0, bde, rec, args = _case(n, nelem)
    real = np.float32 if dtype == "c64" else np.float64
    slow = (1.0 / c0).astype(real)
    v = _perturbations(geom, c0, seeds=(5,))[0].astype(real)
    st = torch_.as_tensor(slow).cuda()
    rt = torch_.as_tensor(rec).cuda()
    loss, grad = w.fwi_loss_function(st, geom.xi, geom.yi, rt, *args[3:], dtype=dtype, bde=bde)
    plan = w.api.get_plan(n, n, dtype, 0, 1, geom.tx_include.size, "python", True)
    return geom, f, c0, bde, rec, args, slow, v, st, rt, grad, plan


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
@pytest.mark.parametrize("n,nelem", [(48, 32), (90, 64)])
def test_product_against_the_oracle(torch_, dtype, n, nelem):
    import waveforminversionust_b200 as w
    geom, f, c0, bde, rec, args, slow, v, st, rt, grad, plan = _dev_case(torch_, n, nelem, dtype)
    hv_t, jv_t = gn_hvp_ref(slow.astype(np.float64), v.astype(np.float64), *args, dtype="c128", bde=bde, return_jv=True)
    hv = w.fwi_gauss_newton_product(st, torch_.as_tensor(v).cuda(), geom.xi, geom.yi, rt, *args[3:], dtype=dtype, bde=bde)
    hv2, jv2, jv = plan.gn_hvp(torch_.as_tensor(v).cuda(), jv=True)
    hv, hv2, jv = hv.cpu().numpy(), hv2.cpu().numpy(), jv.cpu().numpy()[0]
    vhv = float(np.sum(v.astype(np.float64) * hv))
    e_hv, e_jv, e_j2 = rel(hv, hv_t), rel(jv, jv_t), abs(float(jv2[0]) - vhv) / vhv
    print(f"{dtype} n={n}: hv rel-L2 {e_hv:.3e}, J v rel-L2 {e_jv:.3e}, |jv2 - <v,hv>|/<v,hv> {e_j2:.3e}")
    tol = 1e-8 if dtype == "c128" else GRAD_TOL
    assert np.array_equal(hv, hv2)
    assert e_hv < tol and e_jv < tol and e_j2 < (1e-10 if dtype == "c128" else 1e-4)
    # the NumPy surface gives the same product
    hv_np = w.fwi_gauss_newton_product(slow, v, *args, dtype=dtype, bde=bde)
    assert rel(hv_np, hv) < (1e-12 if dtype == "c128" else 1e-6)
    w.clear_plans()


@pytest.mark.gpu
def test_joint_product_is_the_sum_over_frequencies_and_groups_are_bit_identical(torch_):
    import waveforminversionust_b200 as w
    n, nelem = 56, 32
    geom, f0, vel_true = small_case(n, nelem)
    freqs = [0.8 * f0, f0, 1.1 * f0]
    c0 = np.full((n, n), 1490.0)
    bde = np.array([bde_for(geom, c0, f) for f in freqs])
    recs = np.stack([observed_data(geom, f, vel_true, seed=11 + i) for i, f in enumerate(freqs)])
    slow = 1.0 / c0
    v = _perturbations(geom, c0, seeds=(3,))[0]
    tail = (geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab, geom.mask_indices, geom.num_elements)
    st, rt, vt = (torch_.as_tensor(a).cuda() for a in (slow, recs, v))
    hv = w.fwi_gauss_newton_product(st, vt, geom.xi, geom.yi, rt, geom.dense_src(), freqs, *tail, dtype="c128", bde=bde)
    ho = sum(gn_hvp_ref(slow, v, geom.xi, geom.yi, r, geom.dense_src(), fr, *tail, dtype="c128", bde=b)
             for fr, r, b in zip(freqs, recs, bde))
    e = rel(hv.cpu().numpy(), ho)
    print(f"3-frequency product vs sum of oracle products: {e:.3e}")
    assert e < 1e-8
    plan = w.api.get_plan(n, n, "c128", 0, 3, geom.tx_include.size, "python", True)
    plan.set_groups(1)
    h1 = plan.gn_hvp(vt)[0]
    plan.set_groups(2)
    h2 = plan.gn_hvp(vt)[0]
    assert torch_.equal(h1, hv) and torch_.equal(h2, hv)
    w.clear_plans()


@pytest.mark.gpu
def test_product_is_consistent_with_gradient_and_line_search(torch_):
    """ncg_linesearch(v) = (num, den) with den = |J v|^2 and num = -<v, grad>; Re<J v, diff> = <v, grad>."""
    geom, f, c0, bde, rec, args, slow, v, st, rt, grad, plan = _dev_case(torch_, 48, 32, "c128")
    vt = torch_.as_tensor(v).cuda()
    nd = plan.ncg_linesearch(vt).cpu().numpy()
    hv, jv2, jv = plan.gn_hvp(vt, jv=True)
    jv2, jv, g = float(jv2[0]), jv.cpu().numpy()[0], grad.cpu().numpy()
    vg = float(np.sum(v * g))
    U = plan.wavefield(0).cpu().numpy()
    nodes = np.take(geom.ind_matlab, geom.mask_indices)  # column-major flat index x * Ny + y
    sim = U[nodes % 48, nodes // 48, np.arange(geom.tx_include.size)[:, None]] * plan.src_est(0)[:, None]
    diff = sim - np.take_along_axis(rec, geom.mask_indices, axis=1)
    print(f"den {nd[1]:.15e} jv2 {jv2:.15e}; num {nd[0]:.15e} -<v,g> {-vg:.15e}; Re<Jv,diff> {np.real(np.vdot(jv, diff)):.15e}")
    assert abs(nd[1] - jv2) <= 1e-10 * jv2
    assert abs(nd[0] + vg) <= 1e-10 * abs(vg)
    assert abs(np.real(np.vdot(jv, diff)) - vg) <= 1e-10 * abs(vg)
    import waveforminversionust_b200 as w
    w.clear_plans()


@pytest.mark.gpu
def test_plan_state(torch_):
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import _lib
    from waveforminversionust_b200.plan import HelmholtzPlan
    geom, f, c0, bde, rec, args, slow, v, st, rt, grad, plan = _dev_case(torch_, 48, 32, "c64")
    vt = torch_.as_tensor(v).cuda()
    nd0 = plan.ncg_linesearch(vt)
    a, b = plan.gn_hvp(vt), plan.gn_hvp(vt)
    # hv is bit-identical; jv2 and the line-search scalars are FP64 atomics over CTAs (like the loss), so they agree to the
    # last bits only
    close = lambda x, y: bool(torch_.all(torch_.abs(x - y) <= 1e-13 * torch_.abs(y)))
    assert torch_.equal(a[0], b[0]) and close(a[1], b[1])
    assert close(plan.ncg_linesearch(vt), nd0)
    # replaced factors: the line search refuses, after a factorisation and after a refactorising host solve; the next
    # evaluation makes it run again
    rt1 = rt.to(plan.tcplx).reshape(1, plan.nt, plan.nelem).contiguous()
    replace = (lambda: plan.factor(torch_.as_tensor(c0.astype(np.float32)).cuda(), [f]),
               lambda: plan.solve_helmholtz_host(c0.astype(np.float32), np.zeros((48, 48, 1), np.complex64), f, refactor=True))
    for r in replace:
        r()
        with pytest.raises(_lib.UstError, match="replaced"):
            plan.ncg_linesearch(vt)
        plan.fwi_loss_grad(st, rt1, [f], bde=bde)
        assert close(plan.ncg_linesearch(vt), nd0)
    # replaced factors: the product refuses ...
    plan.factor(torch_.as_tensor(c0.astype(np.float32)).cuda(), [f])
    with pytest.raises(_lib.UstError, match="replaced"):
        plan.gn_hvp(vt)
    # ... and the API surface evaluates again
    hv = w.fwi_gauss_newton_product(st, vt, geom.xi, geom.yi, rt, *args[3:], dtype="c64", bde=bde)
    assert torch_.equal(hv, a[0])
    # no evaluation yet on a fresh plan
    p2 = HelmholtzPlan(48, 48, dtype="c64", max_nrhs=geom.tx_include.size, fwi_buffers=True)
    p2.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
    rx = (geom.y_idx * 48 + geom.x_idx).astype(np.int32)
    p2.set_acquisition(geom.src_lin, rx, geom.mask_indices)
    with pytest.raises(_lib.UstError, match="ust_fwi_loss_grad first"):
        p2.gn_hvp(vt)
    p2.close()
    w.clear_plans()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
def test_gpu_driver_one_cg_step_matches_gpu_ncg(torch_, dtype):
    import waveforminversionust_b200 as w
    geom, f, c0, bde, rec, args = _case(64, 32)
    VELn = w.nonlinear_conjugate_gradient(*_driver_args(geom, f, rec, 1), dtype=dtype, bde=bde, return_fields=False)[0]
    w.clear_plans()
    hist = []
    vel = w.gauss_newton_fwi(*_driver_args(geom, f, rec, 1), cg_iters=1, dtype=dtype, bde=bde, history=hist)
    e = rel(vel, VELn)
    print(f"{dtype}: GN(cg_iters=1) vs NCG(Niter=1) velocity rel {e:.3e}; {hist}")
    assert e < (1e-9 if dtype == "c128" else 1e-4)
    w.clear_plans()


@pytest.mark.gpu
def test_gpu_driver_matches_the_driver_on_the_oracle(torch_, monkeypatch):
    """Two outer iterations, cg_iters=4 (complex128): every evaluation point of the GPU run equals the oracle run's."""
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import api
    geom, f, c0, bde, rec, args = _case()
    pts_o, ho = [], []
    lg, hvp = _oracle_callables(args, bde, points=pts_o)
    vel_o = api.gauss_newton_fwi(*_driver_args(geom, f, None, 2), cg_iters=4, dtype="c128", history=ho, loss_grad=lg, hvp=hvp)
    pts_g, hg = [], []
    orig = api.fwi_loss_function

    def recording(params, *a, **k):
        pts_g.append(params.detach().cpu().numpy().astype(np.float64).copy())
        return orig(params, *a, **k)

    monkeypatch.setattr(api, "fwi_loss_function", recording)
    vel_g = api.gauss_newton_fwi(*_driver_args(geom, f, rec, 2), cg_iters=4, dtype="c128", bde=bde, history=hg)
    for a, b in zip(ho, hg):
        print(a, "\n", b)
    assert len(pts_g) == len(pts_o) and [h["cg_iters"] for h in hg] == [h["cg_iters"] for h in ho]
    errs = [rel(a, b) for a, b in zip(pts_g, pts_o)]
    print("evaluation points rel:", errs)
    assert max(errs) < 1e-9 and rel(vel_g, vel_o) < 1e-9
    w.clear_plans()


@pytest.mark.gpu
@pytest.mark.parametrize("shard", ["freq", "source"])
def test_sharded_products_sum_to_the_whole(torch_, shard):
    from waveforminversionust_b200.distributed import ShardedFWI
    n, nelem = 60, 32
    geom, f0, vel_true = small_case(n, nelem)
    freqs = np.array([0.8, 0.9, 1.0, 1.1]) * f0
    rec_all = torch_.as_tensor(np.ascontiguousarray(np.stack([observed_data(geom, f, vel_true, seed=7 + i) for i, f in enumerate(freqs)])
                                                    .astype(np.complex128))).cuda()
    c0 = np.full((n, n), 1485.0)
    slow = torch_.as_tensor(1.0 / c0).cuda()
    v = torch_.as_tensor(_perturbations(geom, c0, seeds=(4,))[0]).cuda()
    whole = ShardedFWI(geom, freqs, dtype="c128", rank=0, world=1)
    whole.loss_grad_device(slow, rec_all)
    h_all, j_all = whole.gn_hvp_device(v)
    h_all, j_all = h_all.clone(), float(j_all)
    whole.close()
    h_sum, j_sum = torch_.zeros_like(h_all), 0.0
    for r in range(3):
        part = ShardedFWI(geom, freqs, dtype="c128", rank=r, world=3, shard=shard)
        part.loss_grad_device(slow, part.local_rec(rec_all).contiguous())
        h, j = part.gn_hvp_device(v)
        h_sum += h; j_sum += float(j)
        part.close()
    e = rel(h_sum.cpu().numpy(), h_all.cpu().numpy())
    print(f"{shard}: sharded product parts vs whole {e:.3e}, jv2 {abs(j_sum - j_all) / j_all:.3e}")
    assert e < 1e-12 and abs(j_sum - j_all) <= 1e-12 * j_all
    assert abs(j_all - float(torch_.sum(v * h_all))) <= 1e-10 * j_all


@pytest.mark.gpu
def test_product_parity_at_256_with_the_tcgen05_engine(torch_):
    """256 x 256, 32 transmitters of a 256-element ring, complex64 on the tcgen05 engine, against the complex128 oracle."""
    import os
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import geometry as G
    n = 256
    geom = G.ring_geometry(n, 256, dwnsmp=8)
    f = G.frequency_for_grid(n)
    vel_true = G.blob_model(geom)
    c0 = G.blob_model(geom, dc=15.0, seed=99)
    thr = max(1, min(16, os.cpu_count() or 1))
    rec = observed_data(geom, f, vel_true, bde=bde_for(geom, vel_true, f))
    slow32 = (1.0 / c0).astype(np.float32)
    vel32 = (np.float32(1.0) / slow32).astype(np.float32)
    bde = bde_for(geom, vel32, f)
    v = (1.0 / G.blob_model(geom, dc=20.0, seed=5) - 1.0 / c0).astype(np.float32)
    args = (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab, geom.mask_indices,
            geom.num_elements)
    hv_t = gn_hvp_ref(slow32.astype(np.float64), v.astype(np.float64), *args, dtype="c128", bde=bde, threads=thr)
    src = w.OneHotSources(geom.src_lin, (n, n, geom.tx_include.size))
    hv = w.fwi_gauss_newton_product(slow32, v, geom.xi, geom.yi, rec, src, f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab,
                                    geom.mask_indices, geom.num_elements, dtype="c64", bde=bde, engine="tc2")
    e = rel(hv, hv_t)
    print(f"256^2 x 32 sources, c64 tcgen05 product vs c128 oracle: rel-L2 {e:.3e}")
    assert e < GRAD_TOL
    w.clear_plans()
