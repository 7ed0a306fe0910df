"""Joint sound-speed and attenuation inversion: complex slowness sigma = s - i kappa, k = w sigma (DESIGN.md section 7d).

The lossy reference (``lossy_setup``, ``LossyFactor``, ``lossy_loss_and_grad``) is built here from the oracle's pieces: the
oracle restates the reference, which has no attenuation, and stays as it is.

CPU: the lossy reference (kappa = 0 is the lossless matrix, the decay rate and its sign), the adjoint identities and finite
differences of the two gradients, and the joint L-BFGS driver on the reference objective.  GPU: the lossy assembly,
evaluation and gradients through the C ABI against the complex128 reference, kappa = 0 against the lossless path bit for
bit, the plan-state guards, the Python surfaces and the sharded joint evaluation."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse.linalg as spla

from common import bde_for, rel, small_case
from oracle import fwi as ofwi
from oracle import helmholtz as oh
from waveforminversionust_b200 import geometry as G

GRAD_TOL = 1e-4


def lossy_setup(x, y, vel, f, a0, L_PML, dtype, bde, stencil, kappa):
    """``oracle.helmholtz._setup`` for a lossy medium: complex slowness ``1/vel - i kappa``, so ``k = w/vel - i w kappa`` and the
    amplitude decays as ``exp(-w kappa r)`` under the ``exp(-ikr)`` outgoing convention (``sign_convention = -1``).  The stencil
    weights still come from min/max(vel).  ``oracle.helmholtz.assemble_planes`` forms the mass term as ``C * k.astype(R)**2``,
    so the complex ``C k^2`` goes in as its ``C`` with ``k = 1`` (multiplying by 1 is exact): kappa = 0 gives the lossless
    matrix bit for bit."""
    R, Cx = oh._REAL[dtype], oh._CPLX[dtype]
    x = np.asarray(x, dtype=R)
    y = np.asarray(y, dtype=R)
    vel = np.asarray(vel, dtype=R)
    f = R(f)
    h = np.mean(np.diff(x)).astype(R)
    g = R(np.mean(np.diff(y)).astype(R) / h)
    Nx, Ny = x.size, y.size
    k = (R(2 * np.pi) * f / vel).astype(R)
    k = (k - 1j * (R(2 * np.pi) * f * np.asarray(kappa, dtype=R))).astype(Cx)
    ex, ey = oh.pml_profiles(x, y, a0, L_PML, dtype)
    A, B, C = oh._abc(ex, ey)
    if bde is None:
        bde = oh.stencil_opt_params(vel.min(), vel.max(), f, h, g, dtype)
    b, d, e = bde
    Ck2 = (C.astype(Cx) * k ** 2).astype(Cx)
    H = oh.assemble_helmholtz(Nx, Ny, g, b, d, e, h, A.astype(Cx), B.astype(Cx), Ck2, np.ones((Ny, Nx), dtype=R), stencil)
    return H.astype(Cx), (Nx, Ny), bde


class LossyFactor(oh.HelmholtzFactor):
    """``oracle.helmholtz.HelmholtzFactor`` of the lossy operator (``lossy_setup``); ``solve`` is the oracle's."""

    def __init__(self, x, y, vel, f, a0, L_PML, kappa, dtype="c128", bde=None, stencil="python"):
        self.dtype = dtype
        self.H, (self.Nx, self.Ny), self.bde = lossy_setup(x, y, vel, f, a0, L_PML, dtype, bde, stencil, kappa)
        self.lu = spla.splu(self.H.T.tocsc())


def lossy_solve(x, y, vel, src, f, a0, L_PML, adjoint, kappa, dtype="c128", bde=None):
    return LossyFactor(x, y, vel, f, a0, L_PML, kappa, dtype, bde=bde).solve(src, adjoint)


def lossy_loss_and_grad(params, xi, yi, REC_DATA, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements,
                        kappa, dtype="c128", bde=None, return_fields=False, threads=1):
    """``oracle.fwi.fwi_loss_and_grad`` for the complex slowness ``sigma = s - i kappa``: ``(loss, grad_s, grad_kappa)`` from the
    virtual sources ``VIRT_s = 2 w^2 sigma alpha u`` (``d(w^2 sigma^2)/ds``) and ``VIRT_kappa = -2i w^2 sigma alpha u``
    (``d(w^2 sigma^2)/dkappa``), each as ``sum_t -Re(conj(VIRT) * ADJ_WV)`` with alpha held fixed (nonlinearcg.py:243-265)."""
    R, Cx = oh._REAL[dtype], oh._CPLX[dtype]
    Nyi, Nxi = np.asarray(yi).size, np.asarray(xi).size
    Nt = np.asarray(tx_include).size
    params = np.asarray(params, dtype=R)
    SLOW = params.reshape(Nyi, Nxi)
    KAPPA = np.asarray(kappa, dtype=R).reshape(Nyi, Nxi)
    REC_DATA = np.asarray(REC_DATA).astype(Cx)
    fac = LossyFactor(xi, yi, (R(1) / SLOW).astype(R), f, a0, L_PML, KAPPA, dtype, bde=bde)
    solve = lambda src, adjoint: fac.solve(src, adjoint, threads=threads)
    WV = solve(SRC, False)
    rec_sim, global_inds = ofwi.receiver_gather(WV, ind_matlab, mask_indices)
    rec = np.take_along_axis(REC_DATA, mask_indices, axis=1)
    SRC_EST = ofwi.estimate_src_strength_batched(rec_sim, rec)
    WV = (WV * SRC_EST[None, None, :]).astype(Cx)
    rec_sim, _ = ofwi.receiver_gather(WV, ind_matlab, mask_indices)
    diff = rec_sim - rec
    loss = R(0.5) * np.sum(np.abs(diff) ** 2)
    flat_adj = np.zeros((Nt, Nyi * Nxi), dtype=Cx)
    flat_adj[np.arange(Nt)[:, None], global_inds] = diff
    ADJ_SRC = np.transpose(flat_adj.reshape(Nt, Nxi, Nyi), (2, 1, 0))
    w = R(2 * np.pi) * R(f)
    SIGMA = (SLOW - 1j * KAPPA).astype(Cx)
    VIRT = (R(2) * w**2) * SIGMA[:, :, None] * WV
    VIRT_K = (-2j * w**2) * SIGMA[:, :, None] * WV
    ADJ_WV = solve(ADJ_SRC, True)
    grad = np.sum(-np.real(np.conj(VIRT) * ADJ_WV), axis=2)
    grad_k = np.sum(-np.real(np.conj(VIRT_K) * ADJ_WV), axis=2)
    out = (float(loss), grad.astype(R).reshape(params.shape), grad_k.astype(R).reshape(params.shape))
    if return_fields:
        return out + (dict(WV=WV, ADJ_WV=ADJ_WV, SRC_EST=SRC_EST, rec_sim=rec_sim, VIRT=VIRT, VIRT_K=VIRT_K),)
    return out


def lossy_observed_data(geom, f, vel_true, kappa_true, bde=None, seed=1234):
    """REC_DATA[t, e] = amplitude_t * u_t(element e) of the lossy medium (complex128 reference), like common.observed_data."""
    fac = LossyFactor(geom.xi, geom.yi, vel_true, f, geom.a0, geom.L_PML, kappa_true, "c128", bde=bde)
    WV = fac.solve(geom.dense_src(np.complex128))
    amp = G.source_amplitudes(geom.tx_include.size, seed)
    return np.ascontiguousarray(WV[geom.y_idx, geom.x_idx, :].T * amp[:, None])


def _case(n=48, nelem=32, dalpha=20.0):
    """Blob truths for both maps; the start is c = 1480 m/s and a uniform kappa of half the blobs' scale.  At 48^2 the
    frequency is ~55 kHz, so the attenuation is given in tens of dB/(cm MHz) to matter over the ring."""
    geom, f, vel_true = small_case(n, nelem)
    kappa_true = G.attenuation_blob_model(geom, dalpha=dalpha)
    c0 = np.full((n, n), 1480.0)
    k0 = np.full((n, n), float(G.db_cm_mhz_to_kappa(0.5 * dalpha)))
    bde = bde_for(geom, c0, f)
    rec = lossy_observed_data(geom, f, vel_true, kappa_true, bde=bde_for(geom, vel_true, f))
    args = (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab,
            geom.mask_indices, geom.num_elements)
    return geom, f, vel_true, kappa_true, c0, k0, bde, rec, args


def jv_ref(slow, kappa, w, direction, args, bde, return_all=False):
    """J w for the perturbation w of slowness (``direction="s"``) or attenuation slowness ("kappa"): the perturbation solve
    H^-1(-VIRT w) gathered at the kept receivers (nonlinearcg.py:279-293), with VIRT = VIRT_s or VIRT_kappa of
    ``lossy_loss_and_grad`` and the source estimates held fixed."""
    xi, yi, rec, SRC, f, a0, L_PML, tx_include, ind_matlab, mask_indices, num_elements = args
    loss, gs, gk, fl = lossy_loss_and_grad(slow, *args, dtype="c128", bde=bde, kappa=kappa, return_fields=True)
    VIRT = fl["VIRT"] if direction == "s" else fl["VIRT_K"]
    fac = LossyFactor(xi, yi, 1.0 / slow, f, a0, L_PML, kappa, "c128", bde=bde)
    jw = ofwi.receiver_gather(fac.solve((-VIRT * w[:, :, None]).astype(np.complex128), False), ind_matlab, mask_indices)[0]
    return (jw, loss, gs, gk, fl) if return_all else jw


# ---------------------------------------------------------------------------------------------------------------------
# lossy reference (CPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["c128", "c64"])
def test_reference_kappa_zero_is_the_lossless_matrix(dtype):
    geom, f, vel = small_case(40)
    bde = bde_for(geom, vel, f)
    H0, _, _ = oh._setup(geom.xi, geom.yi, vel, f, geom.a0, geom.L_PML, dtype, bde, "python")
    Hz, _, _ = lossy_setup(geom.xi, geom.yi, vel, f, geom.a0, geom.L_PML, dtype, bde, "python", np.zeros_like(vel))
    assert H0.dtype == Hz.dtype
    assert np.array_equal(H0.indptr, Hz.indptr) and np.array_equal(H0.indices, Hz.indices) and np.array_equal(H0.data, Hz.data)


def test_oracle_decay_sign_and_rate():
    """Homogeneous medium, uniform kappa, one source at the centre: ln(|u_kappa| / |u_0|) along a grid row, from 3 wavelengths
    off the source to the absorbing layer, is a line of slope -2 pi f kappa (geometrical spreading cancels in the ratio).  A
    positive slope would mean the sign of kappa is wrong.  6 points per wavelength put ~5 wavelengths into the fit; the
    measured slope is within 4e-5 of -2 pi f kappa (complex128)."""
    n = 161
    geom = G.ring_geometry(n, 32)
    f = G.frequency_for_grid(n, ppw=6.0)
    c = 1500.0
    vel = np.full((n, n), c)
    kappa = float(G.db_cm_mhz_to_kappa(3.0))
    h = float(np.mean(np.diff(geom.xi.astype(np.float64))))
    bde = oh.stencil_opt_params(c, c, f, h, 1.0, "c128")
    src = np.zeros((n, n, 1))
    src[n // 2, n // 2, 0] = 1.0
    u0 = oh.solve_helmholtz(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, False, dtype="c128", bde=bde)[n // 2, :, 0]
    uk = lossy_solve(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, False, np.full((n, n), kappa), bde=bde)[n // 2, :, 0]
    x = geom.xi.astype(np.float64)
    i = np.arange(n // 2, n - int(round(geom.L_PML / h)) - 2)
    r = x[i] - x[n // 2]
    sel = r > 3 * c / f
    slope = np.polyfit(r[sel], np.log(np.abs(uk[i][sel]) / np.abs(u0[i][sel])), 1)[0]
    expected = -2 * np.pi * f * kappa
    print(f"decay slope {slope:.6f} Np/m, -2 pi f kappa = {expected:.6f} (ratio {slope / expected:.6f}) over {sel.sum()} nodes")
    assert slope < 0
    assert abs(slope / expected - 1) < 1e-2


def test_oracle_adjoint_identities():
    """Re<J w, diff> = <w, grad> in the kappa direction, and in the s direction at kappa != 0 (complex128)."""
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    slow = 1.0 / c0
    loss, gs, gk, fl = lossy_loss_and_grad(slow, *args, dtype="c128", bde=bde, kappa=k0, return_fields=True)
    diff = fl["rec_sim"] - np.take_along_axis(rec, geom.mask_indices, axis=1)
    ws = 1.0 / G.blob_model(geom, c0=1480.0, dc=20.0, seed=5) - slow
    wk = G.attenuation_blob_model(geom, dalpha=5.0, seed=6)
    for direction, w, grad in (("kappa", wk, gk), ("s", ws, gs)):
        jw = jv_ref(slow, k0, w, direction, args, bde)
        lhs, rhs = float(np.real(np.vdot(jw, diff))), float(np.sum(w * grad))
        print(f"{direction}: Re<Jw, diff> = {lhs:.15e}, <w, grad> = {rhs:.15e}")
        assert abs(lhs - rhs) <= 1e-10 * abs(rhs)


def test_oracle_jv_against_finite_differences():
    """J v against the central difference of alpha P u(. +- eps v) (alpha fixed), v inside the PML-free interior, in both
    directions at a lossy point.  J leaves out the stencil's mass weights and the PML factor like the lossless J
    (DESIGN.md section 7c: one complex factor ~1.1233 + 0.0004i at 48^2, 6.4e-5 left after it).  dsigma^2/dkappa =
    -i dsigma^2/ds, so both directions meet the same stencil and show the same factor; asserted to 1e-3 of each other."""
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    slow = 1.0 / c0
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64))
    bump = np.exp(-(X ** 2 + Y ** 2) / (2 * 0.015 ** 2))
    _, _, _, _, fl = jv_ref(slow, k0, bump, "s", args, bde, return_all=True)
    alpha = fl["SRC_EST"]

    def apu(s, k):
        fac = LossyFactor(geom.xi, geom.yi, 1.0 / s, f, geom.a0, geom.L_PML, k, "c128", bde=bde)
        return ofwi.receiver_gather(fac.solve(geom.dense_src(np.complex128)) * alpha[None, None, :], geom.ind_matlab,
                                    geom.mask_indices)[0]

    eps = 1e-3
    out = {}
    for direction, v in (("s", bump * slow * 1e-2), ("kappa", bump * k0 * 0.5)):
        jv = jv_ref(slow, k0, v, direction, args, bde)
        if direction == "s":
            fd = (apu(slow + eps * v, k0) - apu(slow - eps * v, k0)) / (2 * eps)
        else:
            fd = (apu(slow, k0 + eps * v) - apu(slow, k0 - eps * v)) / (2 * eps)
        c = np.vdot(fd, jv) / np.vdot(fd, fd)
        out[direction] = (c, rel(jv, fd), rel(jv, c * fd))
        print(f"{direction}: J v vs central difference rel-L2 {out[direction][1]:.3e}; best complex scale {c:.6f}, "
              f"rel-L2 after it {out[direction][2]:.3e}")
    for direction in ("s", "kappa"):
        c, e_raw, e_scaled = out[direction]
        assert e_raw < 0.15 and abs(c - 1.1233) < 1e-2 and e_scaled < 1e-3
    assert abs(out["s"][0] - out["kappa"][0]) < 1e-3


def _oracle_joint_objective(args, bde, points=None):
    def loss_grad(params):
        if points is not None:
            points.append(np.array(params, dtype=np.float64))
        loss, gs, gk = lossy_loss_and_grad(params[0], *args, dtype="c128", bde=bde, kappa=params[1])
        return loss, np.stack([gs, gk])
    return loss_grad


def _driver_args(geom, f, rec):
    return (geom.xi, geom.yi, rec, geom.dense_src(), geom.tx_include, geom.ind_matlab, 1480.0, f, geom.a0, geom.L_PML,
            geom.mask_indices)


def test_joint_lbfgs_driver_on_the_oracle_objective():
    from waveforminversionust_b200 import api
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    hist = []
    shapes = []
    lg = _oracle_joint_objective(args, bde)

    def recording(params):
        loss, grad = lg(params)
        shapes.append((params.shape, grad.shape))
        return loss, grad

    c, kappa = api.run_lbfgs_joint_fwi(*_driver_args(geom, f, None), kappa_init=0.0, maxiter=4, dtype="c128", history=hist,
                                       loss_grad=recording)
    print("joint L-BFGS losses:", [round(l / hist[0][0], 6) for l, _ in hist])
    assert c.shape == kappa.shape == (48, 48)
    assert all(s == (2, 48, 48) and g == (2, 48, 48) for s, g in shapes)
    assert np.all(kappa >= 0) and all(np.all(p[1] >= 0) for _, p in hist)
    assert min(l for l, _ in hist) < 0.9 * hist[0][0]


def _gloo_worker(rank, world, port, tmp):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from waveforminversionust_b200 import distributed as D
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    geom, freqs, recs, slow, kappa, tail = _gloo_case()
    loss, grad = 0.0, np.zeros((2,) + slow.shape)
    for i in D.shard_frequencies(freqs.size, rank, world):
        l, gs, gk = lossy_loss_and_grad(slow, geom.xi, geom.yi, recs[i], geom.dense_src(), freqs[i], *tail, dtype="c128",
                                           kappa=kappa)
        loss += l
        grad += np.stack([gs, gk])
    L, Gr = D.allreduce_loss_grad(loss, torch.as_tensor(grad))
    if rank == 0:
        np.savez(tmp, loss=float(L), grad=Gr.numpy())
    dist.barrier()
    dist.destroy_process_group()


def _gloo_case():
    n, nelem = 36, 16
    geom, f0, vel_true = small_case(n, nelem, pml_cells=4.0)
    freqs = np.array([0.8, 0.9, 1.0]) * f0
    kt = G.attenuation_blob_model(geom, dalpha=20.0)
    recs = [lossy_observed_data(geom, f, vel_true, kt, seed=5 + i) for i, f in enumerate(freqs)]
    slow = np.full((n, n), 1 / 1480.0)
    kappa = np.full((n, n), float(G.db_cm_mhz_to_kappa(10.0)))
    tail = (geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab, geom.mask_indices, geom.num_elements)
    return geom, freqs, recs, slow, kappa, tail


def test_two_rank_joint_packed_allreduce_matches_single_process(tmp_path):
    """The packed [grad_s, grad_kappa, loss] all-reduce of ShardedFWI.loss_grad_lossy_device over gloo (world 2, the lossy reference
    as the per-rank evaluator) equals the single-process joint sum."""
    import torch.multiprocessing as mp
    out = str(tmp_path / "r0.npz")
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    got = np.load(out)
    geom, freqs, recs, slow, kappa, tail = _gloo_case()
    loss, grad = 0.0, 0.0
    for f, r in zip(freqs, recs):
        l, gs, gk = lossy_loss_and_grad(slow, geom.xi, geom.yi, r, geom.dense_src(), f, *tail, dtype="c128", kappa=kappa)
        loss += l
        grad = grad + np.stack([gs, gk])
    assert float(got["loss"]) == pytest.approx(loss, rel=1e-12)
    assert rel(got["grad"], grad) < 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_():
    import torch
    return torch


def _plan(geom, dtype, nfreq=1, engine="auto"):
    from waveforminversionust_b200 import HelmholtzPlan
    n = geom.Nx
    p = HelmholtzPlan(n, geom.Ny, dtype=dtype, max_freq=nfreq, max_nrhs=geom.tx_include.size, fwi_buffers=True, engine=engine)
    p.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
    p.set_acquisition(geom.src_lin, (geom.y_idx * n + geom.x_idx).astype(np.int32), geom.mask_indices)
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
@pytest.mark.parametrize("n,stencil", [(40, "python"), (70, "python"), (70, "matlab")])
def test_lossy_assembly_planes(torch_, dtype, n, stencil):
    from waveforminversionust_b200 import HelmholtzPlan
    geom, f, vel = small_case(n)
    bde = bde_for(geom, vel, f)
    kappa = G.attenuation_blob_model(geom, alpha0=5.0, dalpha=20.0)
    plan = HelmholtzPlan(n, n, dtype=dtype, max_freq=1, max_nrhs=8, stencil=stencil)
    plan.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
    vr, kr = vel.astype(plan.real), kappa.astype(plan.real)
    plan.factor(torch_.as_tensor(vr).cuda(), [f], bde=[bde], kappa=torch_.as_tensor(kr).cuda())
    got = plan.planes(0).cpu().numpy()
    ex, ey = oh.pml_profiles(geom.xi, geom.yi, geom.a0, geom.L_PML, "c128")
    A, B, C = oh._abc(ex, ey)
    h = float(np.mean(np.diff(geom.xi.astype(np.float64))))
    w = 2 * np.pi * f
    k = w / vr.astype(np.float64) - 1j * w * kr.astype(np.float64)
    P = oh.assemble_planes(n, n, 1.0, *bde, h, A, B, C * k ** 2, np.ones((n, n)), stencil)  # complex C k^2 as in lossy_setup
    tol = 2e-6 if dtype == "c64" else 1e-13
    for i, name in enumerate(oh.PLANE_ORDER):
        e = rel(got[i, 1:-1, 1:-1], P[name])
        assert e < tol, (name, e)
        assert np.all(got[i, 0, :] == 0) and np.all(got[i, :, 0] == 0)
    assert plan.status() == 0
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
def test_kappa_zero_is_the_lossless_evaluation(torch_, dtype):
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    plan = _plan(geom, dtype)
    slow = torch_.as_tensor((1.0 / c0).astype(plan.real)).cuda()
    rt = torch_.as_tensor(np.ascontiguousarray(rec.astype(plan.cplx)[None])).cuda()
    l0, g0 = plan.fwi_loss_grad(slow, rt, [f], bde=[bde])
    g0 = g0.clone()
    l1, gs, gk = plan.fwi_loss_grad_lossy(slow, torch_.zeros_like(slow), rt, [f], bde=[bde])
    print(f"{dtype}: loss {float(l0):.17e} vs {float(l1):.17e}")
    assert torch_.equal(gs, g0)
    assert abs(float(l1) - float(l0)) <= 1e-13 * abs(float(l0))
    assert bool(torch_.isfinite(gk).all()) and float(torch_.abs(gk).max()) > 0
    plan.close()


def _parity(torch_, geom, f, c0, k0, rec, dtype, engine="auto", threads=1):
    """Device lossy evaluation vs the complex128 oracle on identical float32 (complex64) inputs (DESIGN.md section 5)."""
    plan = _plan(geom, dtype, engine=engine)
    slow_r = (1.0 / c0).astype(plan.real)
    vel_r = (plan.real(1.0) / slow_r).astype(plan.real)
    kap_r = k0.astype(plan.real)
    bde = bde_for(geom, vel_r, f)
    args = (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab, geom.mask_indices,
            geom.num_elements)
    loss_t, gs_t, gk_t, fl = lossy_loss_and_grad(1.0 / vel_r.astype(np.float64), *args, dtype="c128", bde=bde,
                                                    kappa=kap_r.astype(np.float64), return_fields=True, threads=threads)
    loss, gs, gk = plan.fwi_loss_grad_lossy(torch_.as_tensor(slow_r).cuda(), torch_.as_tensor(kap_r).cuda(),
                                            torch_.as_tensor(np.ascontiguousarray(rec.astype(plan.cplx)[None])).cuda(), [f], bde=[bde])
    alpha_t = fl["SRC_EST"]
    U = plan.wavefield(0).cpu().numpy()
    ADJ = plan.adjoint_wavefield(0).cpu().numpy()
    e_u = rel(U, fl["WV"] / alpha_t[None, None, :])
    e_lam = rel(ADJ[1:-1, 1:-1], fl["ADJ_WV"][1:-1, 1:-1])
    # The adjoint field solves for the residual alpha P u - rec, whose cancellation amplifies the field and source-estimate
    # errors (DESIGN.md section 5).  The adjoint solve itself is judged on the device's own residual: the reference's adjoint
    # solve of alpha P u - rec formed in float64 from the device's u and alpha.
    Nt, ny, nx = geom.tx_include.size, geom.Ny, geom.Nx
    alpha = plan.src_est(0).astype(np.complex128)
    sim, inds = ofwi.receiver_gather(U.astype(np.complex128) * alpha[None, None, :], geom.ind_matlab, geom.mask_indices)
    flat = np.zeros((Nt, ny * nx), dtype=np.complex128)
    flat[np.arange(Nt)[:, None], inds] = sim - np.take_along_axis(np.asarray(rec, dtype=np.complex128), geom.mask_indices, axis=1)
    fac = LossyFactor(geom.xi, geom.yi, vel_r.astype(np.float64), f, geom.a0, geom.L_PML, kap_r.astype(np.float64), "c128", bde=bde)
    ADJ_own = fac.solve(np.transpose(flat.reshape(Nt, nx, ny), (2, 1, 0)), True, threads=threads)
    e_lam_solve = rel(ADJ[1:-1, 1:-1], ADJ_own[1:-1, 1:-1])
    e_l, e_gs, e_gk = abs(float(loss) - loss_t) / loss_t, rel(gs.cpu().numpy(), gs_t), rel(gk.cpu().numpy(), gk_t)
    print(f"{dtype} {engine} n={geom.Nx}: forward field {e_u:.2e}, adjoint field (interior) {e_lam:.2e} (adjoint solve of the "
          f"device's residual {e_lam_solve:.2e}), loss {e_l:.2e}, grad_s {e_gs:.2e}, grad_kappa {e_gk:.2e}")
    assert plan.status() == 0
    plan.close()
    return e_u, e_lam_solve, e_lam, e_l, e_gs, e_gk


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["c128", "c64"])
@pytest.mark.parametrize("n,nelem", [(48, 32), (90, 64)])
def test_lossy_parity_against_the_reference(torch_, dtype, n, nelem):
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case(n, nelem)
    e_u, e_lam_solve, e_lam, e_l, e_gs, e_gk = _parity(torch_, geom, f, c0, k0, rec, dtype)
    wv_tol = 1e-5 if dtype == "c64" else 1e-10
    tol = GRAD_TOL if dtype == "c64" else 1e-8
    assert e_u < wv_tol and e_lam_solve < wv_tol and e_lam < wv_tol
    assert e_l < tol and e_gs < tol and e_gk < tol


@pytest.mark.gpu
def test_lossy_parity_at_256_with_the_tcgen05_engine(torch_):
    """256 x 256, 32 transmitters of a 256-element ring, complex64 on the tcgen05 engine, ~0.5 dB/(cm MHz) blobs on a
    0.25 dB/(cm MHz) background, against the complex128 lossy reference."""
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
    e_u, e_lam_solve, e_lam, e_l, e_gs, e_gk = _parity(torch_, geom, f, c0, k0, rec, "c64", engine="tc2", threads=thr)
    # the end-to-end adjoint field inherits the residual's cancellation (3 x the bar, as for the lossless field at 512^2,
    # DESIGN.md section 5); the adjoint solve itself is held to the wavefield bar
    assert e_u < 1e-5 and e_lam_solve < 1e-5 and e_lam < 3e-5
    assert e_l < GRAD_TOL and e_gs < GRAD_TOL and e_gk < GRAD_TOL


def _multi(n=48, nelem=32, nf=4, dtype="c128"):
    geom, f0, vel_true = small_case(n, nelem)
    kt = G.attenuation_blob_model(geom, dalpha=20.0)
    freqs = list(np.linspace(0.8, 1.1, nf) * f0)
    recs = np.ascontiguousarray(np.stack([lossy_observed_data(geom, f, vel_true, kt, seed=11 + i) for i, f in enumerate(freqs)]))
    real = np.float32 if dtype == "c64" else np.float64
    slow = np.full((n, n), 1 / 1490.0, dtype=real)
    kappa = G.attenuation_blob_model(geom, alpha0=5.0, dalpha=10.0, seed=3).astype(real)
    return geom, freqs, recs, slow, kappa


@pytest.mark.gpu
def test_four_frequencies_are_the_sum_and_launch_chains_are_bit_identical(torch_):
    geom, freqs, recs, slow, kappa = _multi()
    plan = _plan(geom, "c128", nfreq=4)
    st, kt, rt = (torch_.as_tensor(a).cuda() for a in (slow, kappa, recs))
    lj, gsj, gkj = (x.clone() for x in plan.fwi_loss_grad_lossy(st, kt, rt, freqs))
    ls, gss, gks = 0.0, 0.0, 0.0
    for i, f in enumerate(freqs):
        l1, gs1, gk1 = plan.fwi_loss_grad_lossy(st, kt, rt[i:i + 1].contiguous(), [f])
        ls += float(l1); gss = gss + gs1.cpu().numpy(); gks = gks + gk1.cpu().numpy()
    print(f"4 frequencies vs the sum of single ones: loss {abs(float(lj) - ls) / ls:.2e}, grad_s {rel(gsj.cpu().numpy(), gss):.2e}, "
          f"grad_kappa {rel(gkj.cpu().numpy(), gks):.2e}")
    assert abs(float(lj) - ls) / ls < 1e-12 and rel(gsj.cpu().numpy(), gss) < 1e-10 and rel(gkj.cpu().numpy(), gks) < 1e-10
    plan.close()
    # two launch chains need >= 8 frequencies (4 per chain): complex64, 8 frequencies
    geom, freqs, recs, slow, kappa = _multi(nf=8, dtype="c64")
    plan = _plan(geom, "c64", nfreq=8)
    st, kt, rt = (torch_.as_tensor(a).cuda() for a in (slow, kappa, recs.astype(np.complex64)))
    res = {}
    for groups in (1, 2, 1):
        plan.set_groups(groups)
        _, gs, gk = plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
        if groups in res:
            assert torch_.equal(gs, res[groups][0]) and torch_.equal(gk, res[groups][1])
        res[groups] = (gs.clone(), gk.clone())
    assert torch_.equal(res[1][0], res[2][0]) and torch_.equal(res[1][1], res[2][1])
    plan.close()


@pytest.mark.gpu
def test_guards_interleaving_and_host_entry(torch_):
    from waveforminversionust_b200 import _lib
    geom, freqs, recs, slow, kappa = _multi(nf=2, dtype="c64")
    rec = recs.astype(np.complex64)
    st, kt, rt = (torch_.as_tensor(a).cuda() for a in (slow, kappa, rec))
    v = torch_.as_tensor((1.0 / G.blob_model(geom, c0=1490.0, dc=20.0, seed=5)).astype(np.float32) - slow).cuda()

    def fresh(lossy):
        p = _plan(geom, "c64", nfreq=2)
        out = p.fwi_loss_grad_lossy(st, kt, rt, freqs) if lossy else p.fwi_loss_grad(st, rt, freqs)
        out = tuple(x.clone() for x in out)
        p.close()
        return out

    ref_lossless, ref_lossy = fresh(False), fresh(True)
    plan = _plan(geom, "c64", nfreq=2)
    for rep in range(2):  # the second round replays both captured graphs
        a = plan.fwi_loss_grad(st, rt, freqs)
        assert torch_.equal(a[1], ref_lossless[1]) and abs(float(a[0]) - float(ref_lossless[0])) <= 1e-13 * float(ref_lossless[0])
        nd = plan.ncg_linesearch(v)  # available after a lossless evaluation
        hv, _ = plan.gn_hvp(v)
        assert bool(torch_.isfinite(nd).all()) and bool(torch_.isfinite(hv).all())
        b = plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
        assert torch_.equal(b[1], ref_lossy[1]) and torch_.equal(b[2], ref_lossy[2])
        assert abs(float(b[0]) - float(ref_lossy[0])) <= 1e-13 * float(ref_lossy[0])
        with pytest.raises(_lib.UstError, match="lossy"):
            plan.ncg_linesearch(v)
        with pytest.raises(_lib.UstError, match="lossy"):
            plan.gn_hvp(v)
    # a lossy factorisation refuses them too; the next lossless evaluation makes them available again
    plan.fwi_loss_grad(st, rt, freqs)
    plan.factor(1.0 / st, freqs, kappa=kt)
    with pytest.raises(_lib.UstError, match="lossy"):
        plan.ncg_linesearch(v)
    plan.fwi_loss_grad(st, rt, freqs)
    plan.ncg_linesearch(v)
    # the host entry equals the device entry bitwise
    lh, gsh, gkh = plan.fwi_loss_grad_lossy_host(slow, kappa, rec, freqs)
    assert np.array_equal(gsh, ref_lossy[1].cpu().numpy()) and np.array_equal(gkh, ref_lossy[2].cpu().numpy())
    assert abs(lh - float(ref_lossy[0])) <= 1e-13 * lh
    # kappa is required
    L = plan.L
    import ctypes as C
    fr = np.asarray(freqs, dtype=np.float64)
    assert L.ust_fwi_loss_grad_lossy(plan.h, C.c_void_p(st.data_ptr()), None, C.c_void_p(rt.data_ptr()), 2,
                                     fr.ctypes.data_as(C.POINTER(C.c_double)), None, C.c_void_p(st.data_ptr()),
                                     C.c_void_p(st.data_ptr()), C.c_void_p(st.data_ptr()), None) != 0
    assert b"kappa" in L.ust_last_error()
    assert L.ust_factor_lossy(plan.h, C.c_void_p(st.data_ptr()), None, 2, fr.ctypes.data_as(C.POINTER(C.c_double)), None, None) != 0
    plan.close()


@pytest.mark.gpu
def test_solve_helmholtz_and_time_domain_with_kappa(torch_):
    import waveforminversionust_b200 as w
    n = 52
    geom, f, vel = small_case(n, 16)
    bde = bde_for(geom, vel, f)
    kappa = G.attenuation_blob_model(geom, alpha0=5.0, dalpha=20.0)
    src = geom.dense_src(np.complex64)
    truth = lossy_solve(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, False, kappa, bde=bde)
    lossless = w.solve_helmholtz(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, False, dtype="c128", bde=bde)
    got = w.solve_helmholtz(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, False, dtype="c128", bde=bde, kappa=kappa)
    assert isinstance(got, np.ndarray) and rel(got, truth) < 1e-10 and rel(lossless, truth) > 1e-3
    # the factor cache keys on kappa: back to lossless, and device buffers
    again = w.solve_helmholtz(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, False, dtype="c128", bde=bde)
    assert np.array_equal(again, lossless)
    got_d = w.solve_helmholtz(geom.xi, geom.yi, torch_.as_tensor(vel).cuda(), torch_.as_tensor(src).cuda(), f, geom.a0, geom.L_PML,
                              True, dtype="c64", bde=bde, kappa=torch_.as_tensor(kappa).cuda())
    truth_a = lossy_solve(geom.xi, geom.yi, vel, src, f, geom.a0, geom.L_PML, True, kappa, bde=bde)
    assert rel(got_d.cpu().numpy(), truth_a) < 1e-5
    # time-domain synthesis of a lossy medium: each frequency's field is the lossy solve
    fr = np.array([0.8, 1.0]) * f
    t = np.linspace(0, 1e-4, 5)
    WF, WT = w.time_domain_simulation(geom.xi, geom.yi, vel, src[:, :, 0], fr, np.ones(2), t, geom.a0, geom.L_PML, dtype="c128",
                                      kappa=kappa)
    for i, fi in enumerate(fr):
        ti = lossy_solve(geom.xi, geom.yi, vel, src[:, :, :1], fi, geom.a0, geom.L_PML, False, kappa)[:, :, 0]
        assert rel(WF[:, :, i], ti) < 1e-9
    w.clear_plans()


@pytest.mark.gpu
def test_joint_loss_function_surfaces_and_driver_match_the_reference(torch_, monkeypatch):
    """fwi_joint_loss_function through torch and through NumPy; run_lbfgs_joint_fwi with the GPU objective visits the same
    evaluation points as the same driver on the lossy reference's objective (complex128)."""
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import api
    geom, f, vel_true, kappa_true, c0, k0, bde, rec, args = _case()
    params = np.stack([1.0 / c0, k0])
    l_np, g_np = w.fwi_joint_loss_function(params, *args, dtype="c128", bde=bde)
    l_t, g_t = w.fwi_joint_loss_function(torch_.as_tensor(params).cuda(), geom.xi, geom.yi, torch_.as_tensor(rec).cuda(), *args[3:],
                                         dtype="c128", bde=bde)
    assert g_np.shape == params.shape and tuple(g_t.shape) == params.shape
    assert abs(float(l_t) - l_np) <= 1e-12 * l_np and rel(g_t.cpu().numpy(), g_np) < 1e-12
    with pytest.raises(ValueError, match="shape"):
        w.fwi_joint_loss_function(params[0], *args, dtype="c128", bde=bde)
    h_o, h_g = [], []
    k_init = float(k0[0, 0])  # off the bound kappa >= 0, so that both blocks move
    vo = api.run_lbfgs_joint_fwi(*_driver_args(geom, f, None), kappa_init=k_init, maxiter=3, dtype="c128", history=h_o,
                                 loss_grad=_oracle_joint_objective(args, bde))
    vg = api.run_lbfgs_joint_fwi(*_driver_args(geom, f, rec), kappa_init=k_init, maxiter=3, dtype="c128", bde=bde, history=h_g)
    print("joint L-BFGS losses (CUDA):  ", [round(l / h_g[0][0], 6) for l, _ in h_g])
    print("joint L-BFGS losses (reference):", [round(l / h_o[0][0], 6) for l, _ in h_o])
    assert len(h_g) == len(h_o) >= 4
    for (lg, pg), (lo, po) in zip(h_g, h_o):
        assert abs(lg - lo) / lo < 1e-6 and rel(pg[0], po[0]) < 1e-9 and rel(pg[1], po[1]) < 1e-9
    assert len({float(np.sum(p[1])) for _, p in h_g}) > 1  # the attenuation map moved
    assert np.sqrt(np.mean((vg[0] - vo[0]) ** 2)) < 1e-4 and rel(vg[1], vo[1]) < 1e-6
    w.clear_plans()


@pytest.mark.gpu
def test_short_joint_inversion_improves_both_maps(torch_):
    """L-BFGS on synthetic lossy data (blob truths for c and kappa), complex64 on the GPU: both model errors go down."""
    import waveforminversionust_b200 as w
    n, nelem = 64, 32
    geom, f0, vel_true = small_case(n, nelem)
    kappa_true = G.attenuation_blob_model(geom, dalpha=20.0)
    freqs = np.array([0.8, 1.0]) * f0
    rec = np.stack([lossy_observed_data(geom, f, vel_true, kappa_true, bde=bde_for(geom, vel_true, f), seed=3 + i)
                    for i, f in enumerate(freqs)])
    c, kappa = w.run_lbfgs_joint_fwi(*_driver_args(geom, freqs, rec), kappa_init=0.0, kappa_scale=float(G.db_cm_mhz_to_kappa(20.0)),
                                     maxiter=8, dtype="c64")
    inner = (slice(12, -12), slice(12, -12))
    ec0, ec1 = np.sqrt(np.mean((1480.0 - vel_true[inner]) ** 2)), np.sqrt(np.mean((c[inner] - vel_true[inner]) ** 2))
    ek0 = np.sqrt(np.mean(G.kappa_to_db_cm_mhz(kappa_true[inner]) ** 2))
    ek1 = np.sqrt(np.mean(G.kappa_to_db_cm_mhz(kappa[inner] - kappa_true[inner]) ** 2))
    print(f"c RMS error {ec0:.3f} -> {ec1:.3f} m/s, attenuation RMS error {ek0:.3f} -> {ek1:.3f} dB/(cm MHz)")
    assert ec1 < ec0 and ek1 < ek0 and np.all(kappa >= 0)
    w.clear_plans()


@pytest.mark.gpu
@pytest.mark.parametrize("shard", ["freq", "source"])
def test_sharded_joint_evaluation_parts_sum_to_the_whole(torch_, shard):
    """ShardedFWI.loss_grad_lossy_device with world = 3 emulated in one process (each rank's all-reduce returns its own part,
    as in test_gpu_parity's sharding test): the parts add up to the unsharded joint evaluation."""
    from waveforminversionust_b200.distributed import ShardedFWI
    geom, freqs, recs, slow, kappa = _multi(n=60, nf=4)
    rec_all = torch_.as_tensor(np.ascontiguousarray(recs)).cuda()
    st, kt = torch_.as_tensor(slow).cuda(), torch_.as_tensor(kappa).cuda()
    whole = ShardedFWI(geom, freqs, dtype="c128", rank=0, world=1)
    l_all, g_all = whole.loss_grad_lossy_device(st, kt, rec_all)
    l_all, g_all = float(l_all), g_all.clone()
    whole.close()
    assert tuple(g_all.shape) == (2, 60, 60)
    l_sum, g_sum = 0.0, torch_.zeros_like(g_all)
    for r in range(3):
        part = ShardedFWI(geom, freqs, dtype="c128", rank=r, world=3, shard=shard)
        l, g = part.loss_grad_lossy_device(st, kt, part.local_rec(rec_all).contiguous())
        l_sum += float(l); g_sum += g
        part.close()
    assert abs(l_sum - l_all) / l_all < 1e-12 and rel(g_sum.cpu().numpy(), g_all.cpu().numpy()) < 1e-12


@pytest.mark.gpu
def test_sharded_joint_driver_matches_the_single_gpu_driver(torch_):
    import waveforminversionust_b200 as w
    from waveforminversionust_b200.distributed import ShardedFWI, run_lbfgs_joint_sharded
    geom, freqs, recs, slow, kappa = _multi(n=56, nelem=16, nf=2)
    h1, h2 = [], []
    c1, k1 = w.run_lbfgs_joint_fwi(*_driver_args(geom, freqs, recs), maxiter=2, dtype="c128", history=h1)
    w.clear_plans()
    eng = ShardedFWI(geom, freqs, dtype="c128", rank=0, world=1)
    c2, k2 = run_lbfgs_joint_sharded(eng, torch_.as_tensor(recs).cuda(), 1480.0, maxiter=2, history=h2)
    eng.close()
    assert len(h1) == len(h2) and all(abs(a[0] - b[0]) <= 1e-10 * a[0] for a, b in zip(h1, h2))
    assert np.sqrt(np.mean((c1 - c2) ** 2)) < 1e-6
    assert np.max(np.abs(k1 - k2)) <= 1e-6 * max(float(np.max(k1)), 1e-12)
