"""Joint sound-speed and attenuation NCG and Gauss-Newton: the complex perturbation source (DESIGN.md section 7e).

With the complex slowness sigma = s - i kappa and the source estimates held fixed, a joint direction [v_s; v_kappa] has
J [v_s; v_kappa] = P H^-1(-2 w^2 sigma alpha u (v_s - i v_kappa)), and J^H r is the pair of lossy gradients formed from the
adjoint field of r.  The reference product and line search below are built from the lossy reference of test_attenuation.

CPU: the reference product's symmetry, semi-definiteness and block identities (J_kappa = -i J_s), the line-search scalars, and
the joint NCG and Gauss-Newton drivers on the reference callables.  GPU: the lossy product and line search through the C ABI
against the complex128 reference, kappa = 0 against the lossless entry points, the plan-state guards, the Python surfaces,
both drivers, sharding and frequency continuation."""
import ctypes as C

import numpy as np
import pytest

from common import bde_for, rel, small_case
from oracle import fwi as ofwi
from test_attenuation import LossyFactor, _case, _multi, _plan, jv_ref, lossy_loss_and_grad, lossy_observed_data
from waveforminversionust_b200 import geometry as G

GRAD_TOL = 1e-4


# ---------------------------------------------------------------------------------------------------------------------
# reference product and line search
# ---------------------------------------------------------------------------------------------------------------------
def lossy_state(slow, kappa, args, bde, threads=1):
    """Fields of the lossy reference evaluation at (slow, kappa) and its factorisation, shared by the products and line
    searches at that point."""
    xi, yi, rec, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements = args
    loss, gs, gk, fl = lossy_loss_and_grad(slow, *args, dtype="c128", bde=bde, kappa=kappa, return_fields=True, threads=threads)
    fl.update(loss=loss, grad=np.stack([gs, gk]), threads=threads,
              fac=LossyFactor(xi, yi, 1.0 / np.asarray(slow, dtype=np.float64), f, a0, L_PML, kappa, "c128", bde=bde))
    return fl


def _lossy_jv(st, args, v):
    """J [v_s; v_kappa]: the perturbation solve with RHS -(VIRT_s v_s + VIRT_kappa v_kappa) = -2 w^2 sigma alpha u (v_s - i v_kappa)
    gathered at the kept receivers (mask order)."""
    ind_matlab, mask_indices = args[8], args[9]
    v = np.asarray(v, dtype=np.float64)
    rhs = -(st["VIRT"] * v[0][:, :, None] + st["VIRT_K"] * v[1][:, :, None])
    return ofwi.receiver_gather(st["fac"].solve(rhs.astype(np.complex128), False, threads=st["threads"]), ind_matlab, mask_indices)[0]


def lossy_gn_hvp_ref(st, args, v):
    """Reference joint Gauss-Newton product Re(J^H J v) (2, Ny, Nx) and J v, at the point of ``st`` (``lossy_state``): J v
    scattered back as the adjoint source, the adjoint solve, then both lossy gradient formulas of ``lossy_loss_and_grad``."""
    xi, yi, rec, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements = args
    Nt, ny, nx = np.asarray(tx_include).size, np.asarray(yi).size, np.asarray(xi).size
    jv = _lossy_jv(st, args, v)
    _, inds = ofwi.receiver_gather(st["WV"], ind_matlab, mask_indices)
    flat = np.zeros((Nt, ny * nx), dtype=np.complex128)
    flat[np.arange(Nt)[:, None], inds] = jv
    ADJ = st["fac"].solve(np.transpose(flat.reshape(Nt, nx, ny), (2, 1, 0)), True, threads=st["threads"])
    hv = np.stack([np.sum(-np.real(np.conj(st["VIRT"]) * ADJ), axis=2), np.sum(-np.real(np.conj(st["VIRT_K"]) * ADJ), axis=2)])
    return hv, jv


def lossy_linesearch_ref(st, args, sd):
    """Reference joint line-search scalars (num, den) = (Re<J sd, REC_DATA - REC_SIM>, |J sd|^2) (nonlinearcg.py:22-28)."""
    rec, mask_indices = args[2], args[9]
    jsd = _lossy_jv(st, args, sd)
    diff = st["rec_sim"] - np.take_along_axis(np.asarray(rec, dtype=np.complex128), mask_indices, axis=1)
    return -float(np.real(np.vdot(jsd, diff))), float(np.sum(np.abs(jsd) ** 2))


def _directions(geom, seeds=(5, 6)):
    """Joint directions [v_s; v_kappa] of the size of a model update: smooth blobs in both maps."""
    out = []
    for s in seeds:
        vs = 1.0 / G.blob_model(geom, c0=1480.0, dc=20.0, seed=s) - 1.0 / 1480.0
        vk = G.attenuation_blob_model(geom, alpha0=0.0, dalpha=10.0, seed=s + 50)
        out.append(np.stack([vs, vk]))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# reference identities (CPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref48():
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    st = lossy_state(1.0 / c0, k0, args, bde)
    return geom, f, c0, k0, bde, rec, args, st


def test_reference_product_symmetric_psd_and_jv2(ref48):
    geom, f, c0, k0, bde, rec, args, st = ref48
    v, w = _directions(geom)
    hv, jv = lossy_gn_hvp_ref(st, args, v)
    hw, jw = lossy_gn_hvp_ref(st, args, w)
    wHv, vHw = float(np.sum(w * hv)), float(np.sum(v * hw))
    vHv, wHw = float(np.sum(v * hv)), float(np.sum(w * hw))
    jv2 = float(np.sum(np.abs(jv) ** 2))
    print(f"<w,Hv> {wHv:.15e} <Hw,v> {vHw:.15e}; <v,Hv> {vHv:.15e} |Jv|^2 {jv2:.15e}")
    assert abs(wHv - vHw) <= 1e-10 * np.sqrt(vHv * wHw)
    assert vHv > 0 and wHw > 0 and wHv ** 2 <= vHv * wHw * (1 + 1e-10)
    assert abs(vHv - jv2) <= 1e-10 * jv2
    # the lossy J of a pure slowness direction is jv_ref's
    assert rel(_lossy_jv(st, args, np.stack([v[0], 0 * v[0]])), jv_ref(1.0 / c0, k0, v[0], "s", args, bde)) < 1e-12


def test_reference_block_identities(ref48):
    """J_kappa = -i J_s, so H_kk = H_ss and H_ks = -H_sk."""
    geom, f, c0, k0, bde, rec, args, st = ref48
    w = _directions(geom, seeds=(7,))[0][0]
    z = np.zeros_like(w)
    h_s, _ = lossy_gn_hvp_ref(st, args, np.stack([w, z]))  # [H_ss w, H_ks w]
    h_k, _ = lossy_gn_hvp_ref(st, args, np.stack([z, w]))  # [H_sk w, H_kk w]
    e_diag, e_off = rel(h_k[1], h_s[0]), rel(h_s[1], -h_k[0])
    print(f"|H_kk w - H_ss w| {e_diag:.2e}, |H_ks w + H_sk w| {e_off:.2e}")
    assert e_diag < 1e-10 and e_off < 1e-10


def test_reference_linesearch_scalars(ref48):
    geom, f, c0, k0, bde, rec, args, st = ref48
    sd = _directions(geom, seeds=(8,))[0]
    num, den = lossy_linesearch_ref(st, args, sd)
    hv, jv = lossy_gn_hvp_ref(st, args, sd)
    sg = float(np.sum(sd * st["grad"]))
    print(f"num {num:.15e} -<sd,g> {-sg:.15e}; den {den:.15e} |J sd|^2 {np.sum(np.abs(jv) ** 2):.15e}")
    assert abs(num + sg) <= 1e-10 * abs(sg)
    assert abs(den - float(np.sum(np.abs(jv) ** 2))) <= 1e-12 * den


def _ref_callables(args, bde, points=None):
    """Reference objective, line search and product for the joint drivers (they pass (2, Ny, Nx) float64 torch tensors)."""
    st = {}

    def loss_grad(x):
        x = x.cpu().numpy()
        if points is not None:
            points.append(x.copy())
        st["s"] = lossy_state(x[0], x[1], args, bde)
        return st["s"]["loss"], st["s"]["grad"]

    def linesearch(sd):
        return lossy_linesearch_ref(st["s"], args, sd.cpu().numpy())

    def hvp(v):
        return lossy_gn_hvp_ref(st["s"], args, v.cpu().numpy())[0]

    return loss_grad, linesearch, hvp


def _driver_args(geom, f, rec, niter):
    return (geom.xi, geom.yi, geom.num_elements, rec, geom.dense_src(), geom.tx_include, geom.ind_matlab, 1480.0, f, niter,
            geom.a0, geom.L_PML, geom.mask_indices)


def test_gn_with_one_cg_step_is_the_joint_ncg_first_iteration(ref48):
    from waveforminversionust_b200 import api
    geom, f, c0, k0, bde, rec, args, st = ref48
    ks = float(G.db_cm_mhz_to_kappa(20.0))
    k_init = float(k0[0, 0])  # off the bound
    lg, ls, hvp = _ref_callables(args, bde)
    hn, hg = [], []
    cn, kn = api.nonlinear_conjugate_gradient_joint(*_driver_args(geom, f, None, 1), kappa_init=k_init, kappa_scale=ks, dtype="c128",
                                                    history=hn, loss_grad=lg, linesearch=ls)
    cg, kg = api.gauss_newton_joint_fwi(*_driver_args(geom, f, None, 1), kappa_init=k_init, kappa_scale=ks, cg_iters=1, damping=0.0,
                                        dtype="c128", history=hg, loss_grad=lg, hvp=hvp)
    print(hn, "\n", hg)
    assert hg[0]["cg_iters"] == 1 and hg[0]["step"] == 1.0 and hg[0]["products"] == 1
    assert hn[0]["clipped"] == 0 and hg[0]["clipped"] == 0
    assert rel(cg, cn) < 1e-12 and rel(kg, kn) < 1e-9
    assert np.max(np.abs(kg - k_init)) > 1e-3 * k_init  # the attenuation moved


def test_gn_quadratic_model_decreases_and_kappa_stays_feasible(ref48):
    from waveforminversionust_b200 import api
    geom, f, c0, k0, bde, rec, args, st = ref48
    pts = []
    lg, ls, hvp = _ref_callables(args, bde, points=pts)
    hist = []
    c, k = api.gauss_newton_joint_fwi(*_driver_args(geom, f, None, 2), kappa_init=0.0, kappa_scale=float(G.db_cm_mhz_to_kappa(20.0)),
                                      cg_iters=4, cg_tol=1e-6, dtype="c128", history=hist, loss_grad=lg, hvp=hvp)
    for h in hist:
        print({q: h[q] for q in ("it", "loss", "cg_iters", "q", "step", "evals", "products", "clipped")})
        q = h["q"]
        assert len(q) >= 2 and q[0] < 0 and all(b < a for a, b in zip(q, q[1:]))
    assert hist[1]["loss"] < hist[0]["loss"]
    assert all(np.all(p[1] >= 0) for p in pts) and np.all(k >= 0)
    assert len(pts) == hist[-1]["evals"]


def test_joint_frequency_continuation_rejects_an_unknown_method():
    from waveforminversionust_b200 import api
    with pytest.raises(ValueError, match="method"):
        api.joint_frequency_continuation(None, None, 0, None, None, None, None, 1480.0, [1.0], [[0]], 1, 0.0, 0.0, None,
                                         method="newton")


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_():
    import torch
    return torch


def _lossy_parity(torch_, geom, f, c0, k0, rec, dtype, engine="auto", threads=1):
    """Device lossy product and line search vs the complex128 reference on identical float32 (complex64) inputs."""
    plan = _plan(geom, dtype, engine=engine)
    slow_r = (1.0 / c0).astype(plan.real)
    vel_r = (plan.real(1.0) / slow_r).astype(plan.real)
    kap_r = k0.astype(plan.real)
    bde = bde_for(geom, vel_r, f)
    args = (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab, geom.mask_indices,
            geom.num_elements)
    v, sd = (d.astype(plan.real) for d in _directions(geom))
    st = lossy_state(1.0 / vel_r.astype(np.float64), kap_r.astype(np.float64), args, bde, threads=threads)
    hv_t, jv_t = lossy_gn_hvp_ref(st, args, v.astype(np.float64))
    nd_t = np.array(lossy_linesearch_ref(st, args, sd.astype(np.float64)))
    cu = lambda a: torch_.as_tensor(np.ascontiguousarray(a)).cuda()
    plan.fwi_loss_grad_lossy(cu(slow_r), cu(kap_r), cu(rec.astype(plan.cplx)[None]), [f], bde=[bde])
    hv, jv2, jv = plan.gn_hvp_lossy(cu(v[0]), cu(v[1]), jv=True)
    nd = plan.ncg_linesearch_lossy(cu(sd[0]), cu(sd[1])).cpu().numpy()
    hv, jv2, jv = hv.cpu().numpy(), float(jv2[0]), jv.cpu().numpy()[0]
    jv2_t = float(np.sum(np.abs(jv_t) ** 2))
    e = dict(hv_s=rel(hv[0], hv_t[0]), hv_k=rel(hv[1], hv_t[1]), jv=rel(jv, jv_t), jv2=abs(jv2 - jv2_t) / jv2_t,
             num=abs(nd[0] - nd_t[0]) / abs(nd_t[0]), den=abs(nd[1] - nd_t[1]) / nd_t[1])
    print(f"{dtype} {engine} n={geom.Nx}: " + ", ".join(f"{k} {x:.2e}" for k, x in e.items()))
    assert plan.status() == 0
    plan.close()
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
@pytest.mark.parametrize("n,nelem", [(48, 32), (90, 64)])
def test_lossy_product_and_linesearch_parity(torch_, dtype, n, nelem):
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case(n, nelem)
    e = _lossy_parity(torch_, geom, f, c0, k0, rec, dtype)
    tol = GRAD_TOL if dtype == "c64" else 1e-10
    assert all(x < tol for x in e.values()), e


@pytest.mark.gpu
def test_lossy_product_parity_at_256_with_the_tcgen05_engine(torch_):
    """256 x 256, 32 transmitters of a 256-element ring, complex64 on the tcgen05 engine, against the complex128 reference."""
    import os
    n = 256
    geom = G.ring_geometry(n, 256, dwnsmp=8)
    f = G.frequency_for_grid(n)
    vel_true = G.blob_model(geom)
    kappa_true = G.attenuation_blob_model(geom, alpha0=0.25, dalpha=0.5)
    c0 = G.blob_model(geom, dc=15.0, seed=99)
    k0 = G.attenuation_blob_model(geom, alpha0=0.25, dalpha=0.25, seed=98)
    thr = max(1, min(16, os.cpu_count() or 1))
    fac = LossyFactor(geom.xi, geom.yi, vel_true, f, geom.a0, geom.L_PML, kappa_true, "c128", bde=bde_for(geom, vel_true, f))
    amp = G.source_amplitudes(geom.tx_include.size, 1234)
    rec = fac.solve(geom.dense_src(np.complex128), threads=thr)[geom.y_idx, geom.x_idx, :].T * amp[:, None]
    del fac
    e = _lossy_parity(torch_, geom, f, c0, k0, rec, "c64", engine="tc2", threads=thr)
    assert all(x < GRAD_TOL for x in e.values()), e


def _dev(torch_, a):
    return torch_.as_tensor(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
def test_kappa_zero_is_the_lossless_product_and_linesearch(torch_, dtype):
    """At kappa = 0 and v_kappa = 0 the lossy product and line search reproduce the lossless ones: hv_s and J v bit for bit.
    jv2 and the line-search scalars are sums of FP64 atomics over CTAs (like the loss), so two runs of the same entry point
    agree to the last bits only; they are held to that."""
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    plan = _plan(geom, dtype)
    slow = _dev(torch_, (1.0 / c0).astype(plan.real))
    zero = torch_.zeros_like(slow)
    rt = _dev(torch_, rec.astype(plan.cplx)[None])
    v = _dev(torch_, _directions(geom)[0][0].astype(plan.real))
    plan.fwi_loss_grad(slow, rt, [f], bde=[bde])
    nd0 = plan.ncg_linesearch(v).clone()
    hv0, j0, jv0 = (x.clone() for x in plan.gn_hvp(v, jv=True))
    plan.fwi_loss_grad_lossy(slow, zero, rt, [f], bde=[bde])
    nd1 = plan.ncg_linesearch_lossy(v, zero)
    hv1, j1, jv1 = plan.gn_hvp_lossy(v, zero, jv=True)
    print(f"{dtype}: line search {nd0.tolist()} vs {nd1.tolist()}; jv2 {float(j0):.17e} vs {float(j1):.17e}")
    assert torch_.equal(hv1[0], hv0) and torch_.equal(jv1, jv0)
    close = lambda x, y: bool(torch_.all(torch_.abs(x - y) <= 1e-13 * torch_.abs(y)))
    assert close(nd1, nd0) and close(j1, j0)
    assert bool(torch_.isfinite(hv1[1]).all()) and float(torch_.abs(hv1[1]).max()) > 0
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
def test_block_identities_and_consistency_on_the_device(torch_, dtype):
    """H_kk = H_ss and H_ks = -H_sk (J_kappa = -i J_s); <v, Hv> = jv2; the line search of sd = v has den = jv2 and num = -<v, g>."""
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    plan = _plan(geom, dtype)
    cu = lambda a: _dev(torch_, np.asarray(a).astype(plan.real))
    _, gs, gk = plan.fwi_loss_grad_lossy(cu(1.0 / c0), cu(k0), _dev(torch_, rec.astype(plan.cplx)[None]), [f], bde=[bde])
    g = torch_.stack([gs, gk]).double().cpu().numpy()
    w = cu(_directions(geom, seeds=(7,))[0][0])
    z = torch_.zeros_like(w)
    h_s = plan.gn_hvp_lossy(w, z)[0].double().cpu().numpy()
    h_k = plan.gn_hvp_lossy(z, w)[0].double().cpu().numpy()
    e_diag, e_off = rel(h_k[1], h_s[0]), rel(h_s[1], -h_k[0])
    v = _directions(geom)[0].astype(plan.real)
    hv, jv2 = plan.gn_hvp_lossy(cu(v[0]), cu(v[1]))
    nd = plan.ncg_linesearch_lossy(cu(v[0]), cu(v[1])).cpu().numpy()
    vhv, jv2 = float(np.sum(v.astype(np.float64) * hv.double().cpu().numpy())), float(jv2[0])
    vg = float(np.sum(v.astype(np.float64) * g))
    print(f"{dtype}: |H_kk - H_ss| {e_diag:.2e}, |H_ks + H_sk| {e_off:.2e}; <v,Hv> {vhv:.12e} jv2 {jv2:.12e} den {nd[1]:.12e}; "
          f"num {nd[0]:.12e} -<v,g> {-vg:.12e}")
    tol = 1e-5 if dtype == "c64" else 1e-12
    assert e_diag < tol and e_off < tol
    assert abs(vhv - jv2) <= (1e-4 if dtype == "c64" else 1e-10) * jv2
    assert abs(nd[1] - jv2) <= 1e-12 * jv2  # the same perturbation solve
    assert abs(nd[0] + vg) <= (1e-4 if dtype == "c64" else 1e-10) * abs(vg)
    plan.close()


@pytest.mark.gpu
def test_four_frequencies_are_the_sum_and_launch_chains_are_bit_identical(torch_):
    geom, freqs, recs, slow, kappa = _multi()
    v = _directions(geom)[0]
    plan = _plan(geom, "c128", nfreq=4)
    st, kt, rt, vs, vk = (torch_.as_tensor(np.ascontiguousarray(a)).cuda() for a in (slow, kappa, recs, v[0], v[1]))
    plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
    hj, jj = (x.clone() for x in plan.gn_hvp_lossy(vs, vk))
    nj = plan.ncg_linesearch_lossy(vs, vk).cpu().numpy()
    hsum, jsum, nsum = 0.0, 0.0, 0.0
    for i, f in enumerate(freqs):
        plan.fwi_loss_grad_lossy(st, kt, rt[i:i + 1].contiguous(), [f])
        h1, j1 = plan.gn_hvp_lossy(vs, vk)
        hsum, jsum = hsum + h1.cpu().numpy(), jsum + float(j1)
        nsum = nsum + plan.ncg_linesearch_lossy(vs, vk).cpu().numpy()
    e_h, e_j, e_n = rel(hj.cpu().numpy(), hsum), abs(float(jj) - jsum) / jsum, rel(nj, nsum)
    print(f"4 frequencies vs the sum of single ones: hv {e_h:.2e}, jv2 {e_j:.2e}, line search {e_n:.2e}")
    assert e_h < 1e-10 and e_j < 1e-12 and e_n < 1e-10
    plan.close()
    # two launch chains need >= 8 frequencies (4 per chain): complex64, 8 frequencies
    geom, freqs, recs, slow, kappa = _multi(nf=8, dtype="c64")
    plan = _plan(geom, "c64", nfreq=8)
    st, kt, rt = (torch_.as_tensor(a).cuda() for a in (slow, kappa, recs.astype(np.complex64)))
    vs, vk = (torch_.as_tensor(a.astype(np.float32)).cuda() for a in v)
    res = {}
    for groups in (1, 2, 1):
        plan.set_groups(groups)
        plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
        hv, _, jv = plan.gn_hvp_lossy(vs, vk, jv=True)
        if groups in res:
            assert torch_.equal(hv, res[groups][0]) and torch_.equal(jv, res[groups][1])
        res[groups] = (hv.clone(), jv.clone())
    assert torch_.equal(res[1][0], res[2][0]) and torch_.equal(res[1][1], res[2][1])
    plan.close()


@pytest.mark.gpu
def test_guards_and_interleaved_replays(torch_):
    from waveforminversionust_b200 import _lib
    geom, freqs, recs, slow, kappa = _multi(nf=2, dtype="c64")
    rec = recs.astype(np.complex64)
    st, kt, rt = (torch_.as_tensor(a).cuda() for a in (slow, kappa, rec))
    v = _directions(geom)[0].astype(np.float32)
    vs, vk = torch_.as_tensor(v[0]).cuda(), torch_.as_tensor(v[1]).cuda()
    plan = _plan(geom, "c64", nfreq=2)
    # before any evaluation
    with pytest.raises(_lib.UstError, match="ust_fwi_loss_grad_lossy first"):
        plan.gn_hvp_lossy(vs, vk)
    with pytest.raises(_lib.UstError, match="ust_fwi_loss_grad_lossy first"):
        plan.ncg_linesearch_lossy(vs, vk)
    # after a lossless evaluation
    plan.fwi_loss_grad(st, rt, freqs)
    with pytest.raises(_lib.UstError, match="lossless"):
        plan.gn_hvp_lossy(vs, vk)
    with pytest.raises(_lib.UstError, match="lossless"):
        plan.ncg_linesearch_lossy(vs, vk)
    # after a factorisation (lossless or lossy) since the lossy evaluation; available again after the next one
    for factor in (lambda: plan.factor(1.0 / st, freqs), lambda: plan.factor(1.0 / st, freqs, kappa=kt)):
        plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
        plan.gn_hvp_lossy(vs, vk)
        factor()
        with pytest.raises(_lib.UstError, match="replaced"):
            plan.gn_hvp_lossy(vs, vk)
        with pytest.raises(_lib.UstError, match="replaced"):
            plan.ncg_linesearch_lossy(vs, vk)
    # after an acquisition change
    plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
    plan._acq_key = None
    plan.set_acquisition(geom.src_lin, (geom.y_idx * geom.Nx + geom.x_idx).astype(np.int32), geom.mask_indices)
    with pytest.raises(_lib.UstError, match="first"):
        plan.gn_hvp_lossy(vs, vk)
    # the lossless entry points still refuse after a lossy evaluation
    plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
    with pytest.raises(_lib.UstError, match="lossy"):
        plan.gn_hvp(vs)
    with pytest.raises(_lib.UstError, match="lossy"):
        plan.ncg_linesearch(vs)
    # interleaved graph replays: the second round replays every captured graph and gives the first round's results
    close = lambda x, y: bool(torch_.all(torch_.abs(x - y) <= 1e-13 * torch_.abs(y)))
    rounds = []
    for rep in range(2):
        plan.fwi_loss_grad(st, rt, freqs)
        n0 = plan.ncg_linesearch(vs).clone()
        h0, _, jv0 = (x.clone() for x in plan.gn_hvp(vs, jv=True))
        plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
        n1 = plan.ncg_linesearch_lossy(vs, vk).clone()
        h1, j1, jv1 = (x.clone() for x in plan.gn_hvp_lossy(vs, vk, jv=True))
        rounds.append((n0, h0, jv0, n1, h1, j1, jv1))
    a, b = rounds
    assert torch_.equal(a[1], b[1]) and torch_.equal(a[2], b[2]) and torch_.equal(a[4], b[4]) and torch_.equal(a[6], b[6])
    assert close(a[0], b[0]) and close(a[3], b[3]) and close(a[5], b[5])
    assert bool(torch_.isfinite(a[4]).all()) and not torch_.equal(a[4][0], a[1])
    # a null kappa direction is an error
    L = plan.L
    out = torch_.empty(2, dtype=torch_.float64, device="cuda")
    hv = torch_.empty((2,) + tuple(vs.shape), dtype=vs.dtype, device="cuda")
    assert L.ust_ncg_linesearch_lossy(plan.h, C.c_void_p(vs.data_ptr()), None, C.c_void_p(out.data_ptr()), None) != 0
    assert b"kappa" in L.ust_last_error()
    assert L.ust_fwi_gn_hvp_lossy(plan.h, C.c_void_p(vs.data_ptr()), None, C.c_void_p(hv[0].data_ptr()), C.c_void_p(hv[1].data_ptr()),
                                  C.c_void_p(out.data_ptr()), None, None) != 0
    assert b"kappa" in L.ust_last_error()
    plan.close()


@pytest.mark.gpu
def test_joint_product_surface_evaluates_only_when_inputs_change(torch_):
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import _lib
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    params = np.stack([1.0 / c0, k0])
    v = _directions(geom)[0]
    st = lossy_state(params[0], params[1], args, bde)
    hv_t, _ = lossy_gn_hvp_ref(st, args, v)
    L = _lib.lib()
    pt, vt, rt = (torch_.as_tensor(a).cuda() for a in (params, v, rec))
    targs = (geom.xi, geom.yi, rt) + args[3:]
    w.fwi_joint_loss_function(pt, *targs, dtype="c128", bde=bde)
    n0 = L.ust_launch_count()
    hv = w.fwi_joint_gauss_newton_product(pt, vt, *targs, dtype="c128", bde=bde)  # reuses the evaluation
    n_prod = L.ust_launch_count() - n0
    assert tuple(hv.shape) == (2, 48, 48) and rel(hv.cpu().numpy(), hv_t) < 1e-10
    n0 = L.ust_launch_count()
    hv2 = w.fwi_joint_gauss_newton_product(pt, vt, *targs, dtype="c128", bde=bde)
    assert L.ust_launch_count() - n0 == n_prod and torch_.equal(hv, hv2)
    # other inputs, or a lossless evaluation in between: the product evaluates first
    w.fwi_loss_function(pt[0].contiguous(), *targs, dtype="c128", bde=bde)
    n0 = L.ust_launch_count()
    hv3 = w.fwi_joint_gauss_newton_product(pt, vt, *targs, dtype="c128", bde=bde)
    n_eval = L.ust_launch_count() - n0
    print(f"launches: product {n_prod}, evaluation + product {n_eval}")
    assert n_eval > n_prod and torch_.equal(hv3, hv)
    p2 = pt.clone()
    p2[1] *= 1.5
    n0 = L.ust_launch_count()
    w.fwi_joint_gauss_newton_product(p2, vt, *targs, dtype="c128", bde=bde)
    assert L.ust_launch_count() - n0 == n_eval
    # NumPy in, NumPy out
    hv_np = w.fwi_joint_gauss_newton_product(params, v, *args, dtype="c128", bde=bde)
    assert isinstance(hv_np, np.ndarray) and rel(hv_np, hv.cpu().numpy()) < 1e-12
    with pytest.raises(ValueError, match="shape"):
        w.fwi_joint_gauss_newton_product(params, v[0], *args, dtype="c128", bde=bde)
    w.clear_plans()


@pytest.mark.gpu
def test_gpu_drivers_match_the_drivers_on_the_reference(torch_, monkeypatch):
    """Joint NCG (3 iterations) and joint Gauss-Newton (2 outer iterations, cg_iters=3), complex128: every evaluation point of
    the GPU run equals the reference run's."""
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import api
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    kw = dict(kappa_init=0.0, kappa_scale=float(G.db_cm_mhz_to_kappa(20.0)), dtype="c128")
    pts_g = []
    orig = api.fwi_joint_loss_function

    def recording(params, *a, **k):
        pts_g.append(params.detach().cpu().numpy().astype(np.float64).copy())
        return orig(params, *a, **k)

    monkeypatch.setattr(api, "fwi_joint_loss_function", recording)
    for name, drv, extra, niter in (("ncg", api.nonlinear_conjugate_gradient_joint, {}, 3),
                                    ("gn", api.gauss_newton_joint_fwi, dict(cg_iters=3), 2)):
        pts_o, ho, hg = [], [], []
        lg, ls, hvp = _ref_callables(args, bde, points=pts_o)
        inj = dict(loss_grad=lg, linesearch=ls) if name == "ncg" else dict(loss_grad=lg, hvp=hvp)
        ro = drv(*_driver_args(geom, f, None, niter), history=ho, **kw, **extra, **inj)
        pts_g.clear()
        rg = drv(*_driver_args(geom, f, rec, niter), bde=bde, history=hg, **kw, **extra)
        errs = [max(rel(a[0], b[0]), rel(a[1], b[1])) for a, b in zip(pts_g, pts_o)]
        print(name, "losses (CUDA):", [h["loss"] for h in hg], "\n   (reference):", [h["loss"] for h in ho], "\n   points rel:", errs)
        assert len(pts_g) == len(pts_o) >= niter and max(errs) < 1e-9
        assert rel(rg[0], ro[0]) < 1e-9 and rel(rg[1], ro[1]) < 1e-8
        assert len({float(np.sum(p[1])) for p in pts_g}) > 1  # the attenuation map moved
        w.clear_plans()


def _inversion_case():
    """The case of test_attenuation's short joint L-BFGS inversion: 64^2, 32 elements, 2 frequencies, blob truths."""
    n, nelem = 64, 32
    geom, f0, vel_true = small_case(n, nelem)
    kappa_true = G.attenuation_blob_model(geom, dalpha=20.0)
    freqs = np.array([0.8, 1.0]) * f0
    rec = np.stack([lossy_observed_data(geom, f, vel_true, kappa_true, bde=bde_for(geom, vel_true, f), seed=3 + i)
                    for i, f in enumerate(freqs)])
    return geom, freqs, vel_true, kappa_true, rec


def _errors(vel_true, kappa_true, c, kappa):
    inner = (slice(12, -12), slice(12, -12))
    ec0, ec1 = np.sqrt(np.mean((1480.0 - vel_true[inner]) ** 2)), np.sqrt(np.mean((c[inner] - vel_true[inner]) ** 2))
    ek0 = np.sqrt(np.mean(G.kappa_to_db_cm_mhz(kappa_true[inner]) ** 2))
    ek1 = np.sqrt(np.mean(G.kappa_to_db_cm_mhz(kappa[inner] - kappa_true[inner]) ** 2))
    return ec0, ec1, ek0, ek1


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["ncg", "gn"])
def test_short_joint_inversion_improves_both_maps(torch_, method):
    import waveforminversionust_b200 as w
    geom, freqs, vel_true, kappa_true, rec = _inversion_case()
    kw = dict(kappa_init=0.0, kappa_scale=float(G.db_cm_mhz_to_kappa(20.0)), dtype="c64")
    hist = []
    if method == "ncg":
        c, kappa = w.nonlinear_conjugate_gradient_joint(*_driver_args(geom, freqs, rec, 8), history=hist, **kw)
    else:
        c, kappa = w.gauss_newton_joint_fwi(*_driver_args(geom, freqs, rec, 4), cg_iters=4, history=hist, **kw)
    ec0, ec1, ek0, ek1 = _errors(vel_true, kappa_true, c, kappa)
    print(f"{method}: c RMS error {ec0:.3f} -> {ec1:.3f} m/s, attenuation RMS error {ek0:.3f} -> {ek1:.3f} dB/(cm MHz); "
          f"losses / first {[round(h['loss'] / hist[0]['loss'], 4) for h in hist]}")
    assert ec1 < ec0 and ek1 < ek0 and np.all(kappa >= 0)
    w.clear_plans()


@pytest.mark.gpu
@pytest.mark.parametrize("shard", ["freq", "source"])
def test_sharded_joint_products_sum_to_the_whole(torch_, shard):
    """ShardedFWI.gn_hvp_lossy_device with world = 3 emulated in one process (each rank's all-reduce returns its own part):
    the parts add up to the unsharded product."""
    from waveforminversionust_b200.distributed import ShardedFWI
    geom, freqs, recs, slow, kappa = _multi(n=60, nf=4)
    rec_all = torch_.as_tensor(np.ascontiguousarray(recs)).cuda()
    st, kt = torch_.as_tensor(slow).cuda(), torch_.as_tensor(kappa).cuda()
    v = _directions(geom)[0]
    vs, vk = torch_.as_tensor(v[0]).cuda(), torch_.as_tensor(v[1]).cuda()
    whole = ShardedFWI(geom, freqs, dtype="c128", rank=0, world=1)
    whole.loss_grad_lossy_device(st, kt, rec_all)
    h_all, j_all = whole.gn_hvp_lossy_device(vs, vk)
    h_all, j_all = h_all.clone(), float(j_all)
    whole.close()
    assert tuple(h_all.shape) == (2, 60, 60)
    h_sum, j_sum = torch_.zeros_like(h_all), 0.0
    for r in range(3):
        part = ShardedFWI(geom, freqs, dtype="c128", rank=r, world=3, shard=shard)
        part.loss_grad_lossy_device(st, kt, part.local_rec(rec_all).contiguous())
        h, j = part.gn_hvp_lossy_device(vs, vk)
        h_sum += h; j_sum += float(j)
        part.close()
    e = rel(h_sum.cpu().numpy(), h_all.cpu().numpy())
    print(f"{shard}: sharded joint product parts vs whole {e:.3e}, jv2 {abs(j_sum - j_all) / j_all:.3e}")
    assert e < 1e-12 and abs(j_sum - j_all) <= 1e-12 * j_all
    assert abs(j_all - float(torch_.sum(torch_.as_tensor(v).cuda() * h_all))) <= 1e-10 * j_all


@pytest.mark.gpu
def test_sharded_joint_gn_driver_matches_the_single_gpu_driver(torch_):
    import waveforminversionust_b200 as w
    from waveforminversionust_b200.distributed import ShardedFWI, run_gauss_newton_joint_sharded
    geom, freqs, recs, slow, kappa = _multi(n=56, nelem=16, nf=2)
    ks = float(G.db_cm_mhz_to_kappa(20.0))
    h1, h2 = [], []
    c1, k1 = w.gauss_newton_joint_fwi(*_driver_args(geom, freqs, recs, 2), kappa_scale=ks, cg_iters=3, dtype="c128", history=h1)
    w.clear_plans()
    eng = ShardedFWI(geom, freqs, dtype="c128", rank=0, world=1)
    c2, k2 = run_gauss_newton_joint_sharded(eng, torch_.as_tensor(recs).cuda(), 1480.0, 2, kappa_scale=ks, cg_iters=3, history=h2)
    eng.close()
    print([h["loss"] for h in h1], [h["loss"] for h in h2])
    assert len(h1) == len(h2) and all(abs(a["loss"] - b["loss"]) <= 1e-10 * a["loss"] for a, b in zip(h1, h2))
    assert [h["cg_iters"] for h in h1] == [h["cg_iters"] for h in h2]
    assert rel(c1, c2) < 1e-10 and np.max(np.abs(k1 - k2)) <= 1e-8 * max(float(np.max(k1)), 1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["ncg", "gn", "lbfgs"])
def test_joint_frequency_continuation(torch_, method):
    import waveforminversionust_b200 as w
    geom, freqs, vel_true, kappa_true, rec = _inversion_case()
    hist = []
    c, kappa = w.joint_frequency_continuation(geom.xi, geom.yi, geom.num_elements, rec, geom.dense_src(), geom.tx_include,
                                              geom.ind_matlab, 1480.0, freqs, [[0], [1]], 2, geom.a0, geom.L_PML, geom.mask_indices,
                                              dtype="c64", history=hist, method=method)
    print(method, [len(h) for h in hist], _errors(vel_true, kappa_true, c, kappa))
    assert len(hist) == 2 and all(len(h) > 0 for h in hist)
    assert c.shape == kappa.shape == (64, 64) and np.all(np.isfinite(c)) and np.all(np.isfinite(kappa)) and np.all(kappa >= 0)
    w.clear_plans()
