"""The discrete gradient mode (``gradient="discrete"``, ``ust_plan_set_gradient``, DESIGN.md section 7f): the exact derivative
of the discrete forward map at fixed stencil weights (b, d, e).

The reference's linearisation uses the virtual source ``2 w^2 sigma alpha u``.  The discrete forward map's interior row i holds
the mass term ``sum_j w_ij C_j w^2 sigma_j^2 u_j`` (w_ij = 1-d-e, d/4, e/4; C = e_x e_y), so its exact derivative applies the
mass matrix M (those weights times C, zero on the Dirichlet ring) to that source:

    J [v_s; v_kappa] = P H^-1( -M (2 w^2 sigma (v_s - i v_kappa) alpha u) ),   J^H r = -S^H M^H H^-H P^H r.

The discrete reference (``Discrete``) is built here from the oracle's pieces: M is ``oracle.helmholtz.assemble_helmholtz``
with A = B = 0, k = 1 and the true C, with the ring rows zeroed; the lossy operator is ``test_attenuation.LossyFactor``.  The
oracle restates the reference and stays as it is.

CPU: J v against central differences of alpha P u (alpha fixed), <v, g> against central differences of the loss (alpha
re-estimated), the adjoint and Gauss-Newton identities and the joint blocks.  GPU: parity of every quantity with the discrete
reference, finite differences of the device's own loss, launch chains, frequency sums, mode switching and its guards, shards,
and the Gauss-Newton driver on the discrete reference."""
import numpy as np
import pytest
import scipy.sparse as sp

from common import bde_for, observed_data, rel, small_case
from oracle import fwi as ofwi
from oracle import helmholtz as oh
from test_attenuation import LossyFactor, lossy_observed_data
from waveforminversionust_b200 import geometry as G

GRAD_TOL = 1e-4  # complex64 against the complex128 reference (the project's bar for the FWI kernels)
TOL128 = 1e-10


_M_CACHE = {}


def mass_matrix(xi, yi, a0, L_PML, bde, stencil="python"):
    """M: the mass part of the operator's interior rows (weights 1-d-e, d/4, e/4 times C = e_x e_y), zero on the ring."""
    key = (np.asarray(xi).tobytes(), np.asarray(yi).tobytes(), float(a0), float(L_PML), tuple(np.asarray(bde, np.float64)), stencil)
    if key in _M_CACHE:
        return _M_CACHE[key]
    x, y = np.asarray(xi, dtype=np.float64), np.asarray(yi, dtype=np.float64)
    Nx, Ny = x.size, y.size
    h = np.mean(np.diff(x))
    g = np.mean(np.diff(y)) / h
    ex, ey = oh.pml_profiles(x, y, a0, L_PML, "c128")
    A, B, C = oh._abc(ex, ey)
    b, d, e = bde
    M = oh.assemble_helmholtz(Nx, Ny, g, b, d, e, h, 0 * A, 0 * B, C.astype(np.complex128), np.ones((Ny, Nx)), stencil)
    interior = np.zeros((Ny, Nx))
    interior[1:-1, 1:-1] = 1.0
    _M_CACHE[key] = (sp.diags(interior.ravel()) @ M).tocsr()
    return _M_CACHE[key]


class Discrete:
    """Loss, gradient, J and J^H of the discrete forward map at fixed (b, d, e), complex128, one frequency, at the slowness
    ``slow`` and attenuation slowness ``kappa`` (0: lossless)."""

    def __init__(self, slow, kappa, args, bde, stencil="python"):
        xi, yi, rec, SRC, f, a0, L_PML, tx_include, ind_matlab, mask, _ = args
        self.ind, self.mask, self.geom_shape = ind_matlab, mask, slow.shape
        self.fac = LossyFactor(xi, yi, 1.0 / slow, f, a0, L_PML, kappa, "c128", bde=bde, stencil=stencil)
        WV = self.fac.solve(SRC)
        rec_sim, self.gi = ofwi.receiver_gather(WV, ind_matlab, mask)
        reck = np.take_along_axis(np.asarray(rec), mask, axis=1)
        self.alpha = ofwi.estimate_src_strength_batched(rec_sim, reck)
        self.U = WV * self.alpha[None, None, :]
        self.diff = ofwi.receiver_gather(self.U, ind_matlab, mask)[0] - reck
        self.loss = 0.5 * float(np.sum(np.abs(self.diff) ** 2))
        self.sigma = slow - 1j * np.asarray(kappa, dtype=np.float64) * np.ones_like(slow)
        self.w2 = (2 * np.pi * f) ** 2
        self.M = mass_matrix(xi, yi, a0, L_PML, bde, stencil)
        self.grad_s, self.grad_k = self.jh(self.diff)

    def jv(self, vs, vk=None):
        dsig = vs - 1j * (0.0 if vk is None else vk)
        src = (2 * self.w2) * (self.sigma * dsig)[:, :, None] * self.U
        N, nt = src.shape[0] * src.shape[1], src.shape[2]
        src = (self.M @ src.reshape(N, nt)).reshape(src.shape)
        return ofwi.receiver_gather(self.fac.solve(-src), self.ind, self.mask)[0]

    def jh(self, r):
        """J^H r as (grad_s, grad_kappa)."""
        Ny, Nx = self.geom_shape
        nt = r.shape[0]
        flat = np.zeros((nt, Ny * Nx), dtype=np.complex128)
        flat[np.arange(nt)[:, None], self.gi] = r
        lam = self.fac.solve(np.transpose(flat.reshape(nt, Nx, Ny), (2, 1, 0)), True)
        y = (self.M.conj().T @ lam.reshape(Ny * Nx, nt)).reshape(lam.shape)
        z = np.sum(np.conj(self.U) * y, axis=2)
        Gc = -2 * self.w2 * np.conj(self.sigma) * z
        return Gc.real, -Gc.imag

    def hv(self, vs, vk=None):
        jv = self.jv(vs, vk)
        return self.jh(jv), jv


def _case(n=48, nelem=32):
    geom, f, vel_true = small_case(n, nelem)
    c0 = np.full((n, n), 1480.0)
    bde = bde_for(geom, c0, f)
    rec = observed_data(geom, f, vel_true, bde=bde_for(geom, vel_true, f))
    args = (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab,
            geom.mask_indices, geom.num_elements)
    return geom, f, c0, bde, rec, args


def _directions(geom, slow):
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64))
    return {"interior blob": np.exp(-(X ** 2 + Y ** 2) / (2 * 0.015 ** 2)) * slow * 1e-2,
            "PML corner": np.exp(-((X - 0.11) ** 2 + (Y - 0.11) ** 2) / (2 * 0.006 ** 2)) * slow * 1e-2,
            "white noise": np.random.default_rng(3).standard_normal(slow.shape) * slow * 1e-2}


# ---------------------------------------------------------------------------------------------------------------------
# the discrete reference against finite differences (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def _apu(args, bde, s, kappa, alpha, stencil="python"):
    xi, yi, rec, SRC, f, a0, L_PML, tx_include, ind_matlab, mask, _ = args
    fac = LossyFactor(xi, yi, 1.0 / s, f, a0, L_PML, kappa, "c128", bde=bde, stencil=stencil)
    return ofwi.receiver_gather(fac.solve(SRC) * alpha[None, None, :], ind_matlab, mask)[0]


@pytest.mark.parametrize("name,bound", [("interior blob", 1e-7), ("PML corner", 2e-3), ("white noise", 1e-7)])
def test_exact_jv_against_finite_differences(name, bound):
    """J v against the central difference of alpha P u(s +- eps v), alpha fixed (measured 1.4e-9, 4.4e-4, 4.1e-9)."""
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    v = _directions(geom, slow)[name]
    ref = Discrete(slow, 0.0, args, bde)
    eps = 1e-3
    fd = (_apu(args, bde, slow + eps * v, 0.0, ref.alpha) - _apu(args, bde, slow - eps * v, 0.0, ref.alpha)) / (2 * eps)
    e = rel(ref.jv(v), fd)
    print(f"{name}: exact J v vs central difference rel-L2 {e:.3e}")
    assert e < bound


@pytest.mark.parametrize("stencil", ["python", "matlab"])
def test_exact_jv_kappa_direction_at_a_lossy_background(stencil):
    """A kappa direction and an s direction at 10 dB/(cm MHz), both stencil variants: the mass weights are the same in both."""
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    k0 = np.full_like(slow, float(G.db_cm_mhz_to_kappa(10.0)))
    ref = Discrete(slow, k0, args, bde, stencil)
    blob = _directions(geom, slow)["interior blob"] / (slow * 1e-2)
    eps = 1e-3
    for direction, v in (("kappa", blob * k0 * 0.5), ("s", blob * slow * 1e-2)):
        dk, ds = (v, 0 * v) if direction == "kappa" else (0 * v, v)
        fd = (_apu(args, bde, slow + eps * ds, k0 + eps * dk, ref.alpha, stencil)
              - _apu(args, bde, slow - eps * ds, k0 - eps * dk, ref.alpha, stencil)) / (2 * eps)
        jv = ref.jv(ds, dk)
        e = rel(jv, fd)
        print(f"{stencil}, {direction} direction: exact J v vs central difference rel-L2 {e:.3e}")
        assert e < 1e-7


@pytest.mark.parametrize("name", ["interior blob", "white noise"])
def test_exact_gradient_is_the_derivative_of_the_loss(name):
    """<v, g_exact> against the central difference of the loss with alpha re-estimated: alpha is the least-squares optimum,
    so holding it fixed is exact for the gradient.  On white noise the reference gradient has the wrong sign."""
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    v = _directions(geom, slow)[name]
    ref = Discrete(slow, 0.0, args, bde)
    eps = 1e-3
    lossf = lambda s: ofwi.fwi_loss_and_grad(s, *args, dtype="c128", bde=bde)[0]
    fd = (lossf(slow + eps * v) - lossf(slow - eps * v)) / (2 * eps)
    vg = float(np.sum(v * ref.grad_s))
    g_ref = ofwi.fwi_loss_and_grad(slow, *args, dtype="c128", bde=bde)[1]
    print(f"{name}: d loss FD {fd:.9e}, <v, g_exact> {vg:.9e}, <v, g_ref> {float(np.sum(v * g_ref)):.9e}")
    assert abs(vg - fd) <= 1e-6 * abs(fd)
    assert abs(ref.loss - lossf(slow)) <= 1e-12 * ref.loss


def test_adjoint_symmetry_and_gauss_newton_identities():
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    ref = Discrete(slow, 0.0, args, bde)
    d = _directions(geom, slow)
    v, w = d["interior blob"], d["white noise"]
    jw = ref.jv(w)
    lhs, rhs = float(np.real(np.vdot(jw, ref.diff))), float(np.sum(w * ref.grad_s))
    assert abs(lhs - rhs) <= 1e-10 * abs(rhs)
    (hv, _), jv = ref.hv(v)
    (hw, _), _ = ref.hv(w)
    a, b = float(np.sum(w * hv)), float(np.sum(v * hw))
    assert abs(a - b) <= 1e-10 * max(abs(a), abs(b))
    vhv, jv2 = float(np.sum(v * hv)), float(np.vdot(jv, jv).real)
    assert jv2 > 0 and abs(vhv - jv2) <= 1e-10 * jv2


def test_joint_blocks():
    """H_kk = H_ss and H_ks = -H_sk: J_kappa = -i J_s holds with the mass stencil, which multiplies both alike."""
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    k0 = np.full_like(slow, float(G.db_cm_mhz_to_kappa(10.0)))
    ref = Discrete(slow, k0, args, bde)
    v = _directions(geom, slow)["interior blob"]
    (h_ss, h_ks), _ = ref.hv(v, 0 * v)
    (h_sk, h_kk), _ = ref.hv(0 * v, v)
    assert rel(h_kk, h_ss) < 1e-12 and rel(h_sk, -h_ks) < 1e-12


def test_eval_key_separates_the_modes():
    """An evaluation in one mode is never reused for a product in the other (host inputs: no GPU needed)."""
    from waveforminversionust_b200 import api
    p, rec, fr = np.ones((4, 4)), np.ones((1, 2, 3), np.complex64), np.array([1.0])
    ref, disc = api._eval_key(p, rec, fr, None), api._eval_key(p, rec, fr, None, gradient="discrete")
    assert api._same_eval(ref, api._eval_key(p, rec, fr, None, gradient="reference"))
    assert not api._same_eval(ref, disc)
    assert not api._same_eval(api._eval_key(p, rec, fr, None, True, "discrete"), disc)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def torch_():
    import torch
    return torch


def _plan(geom, dtype, nfreq=1, engine="auto"):
    from waveforminversionust_b200 import HelmholtzPlan
    p = HelmholtzPlan(geom.Nx, geom.Ny, dtype=dtype, max_freq=nfreq, max_nrhs=geom.tx_include.size, fwi_buffers=True, engine=engine)
    p.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
    p.set_acquisition(geom.src_lin, (geom.y_idx * geom.Nx + geom.x_idx).astype(np.int32), geom.mask_indices)
    return p


def _dev(torch_, a):
    return torch_.as_tensor(np.ascontiguousarray(a)).cuda()


def _device_quantities(torch_, plan, slow, kappa, rec, f, bde, sd, v):
    """Every quantity of one evaluation, one line search and one product on the plan (lossy when kappa is not None; bde None:
    the weights the device computes from min/max(vel))."""
    cu = lambda a: _dev(torch_, np.asarray(a).astype(plan.real))
    rt = _dev(torch_, rec.astype(plan.cplx)[None])
    out = {}
    if kappa is None:
        loss, g = plan.fwi_loss_grad(cu(slow), rt, [f], bde=None if bde is None else [bde])
        out["grad_s"] = g
        out["linesearch"] = plan.ncg_linesearch(cu(sd))
        hv, jv2, jv = plan.gn_hvp(cu(v), jv=True)
        out["hv_s"] = hv
    else:
        loss, gs, gk = plan.fwi_loss_grad_lossy(cu(slow), cu(kappa), rt, [f], bde=None if bde is None else [bde])
        out["grad_s"], out["grad_k"] = gs, gk
        out["linesearch"] = plan.ncg_linesearch_lossy(cu(sd), cu(0.5 * sd * kappa / slow))
        hv, jv2, jv = plan.gn_hvp_lossy(cu(v), cu(0.5 * v * kappa / slow), jv=True)
        out["hv_s"], out["hv_k"] = hv[0], hv[1]
    out["loss"], out["jv2"], out["jv"] = loss, jv2, jv[0]
    return {k: t.cpu().numpy().astype(np.complex128 if t.is_complex() else np.float64) for k, t in out.items()}


def _reference_quantities(slow, kappa, args, bde, sd, v):
    ref = Discrete(slow, 0.0 if kappa is None else kappa, args, bde)
    out = {"loss": ref.loss, "grad_s": ref.grad_s}
    if kappa is None:
        jsd = ref.jv(sd)
        (hs, _), jv = ref.hv(v)
    else:
        out["grad_k"] = ref.grad_k
        jsd = ref.jv(sd, 0.5 * sd * kappa / slow)
        (hs, hk), jv = ref.hv(v, 0.5 * v * kappa / slow)
        out["hv_k"] = hk
    out["linesearch"] = np.array([float(np.real(np.vdot(jsd, -ref.diff))), float(np.vdot(jsd, jsd).real)])
    out["hv_s"], out["jv"], out["jv2"] = hs, jv, float(np.vdot(jv, jv).real)
    return out


def _compare(dev, ref, tol, label):
    errs = {k: rel(np.atleast_1d(dev[k]).ravel(), np.atleast_1d(ref[k]).ravel()) for k in ref}
    print(label, " ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    assert max(errs.values()) < tol, errs


@pytest.mark.gpu
@pytest.mark.parametrize("lossy", [False, True])
@pytest.mark.parametrize("dtype", ["c128", "c64"])
@pytest.mark.parametrize("n,nelem", [(48, 32), (90, 64)])
def test_parity_with_the_discrete_reference(torch_, dtype, n, nelem, lossy):
    geom, f, c0, bde, rec, args = _case(n, nelem)
    real = np.float32 if dtype == "c64" else np.float64
    slow = (1.0 / c0).astype(real).astype(np.float64)
    kappa = np.full_like(slow, float(G.db_cm_mhz_to_kappa(10.0))).astype(real).astype(np.float64) if lossy else None
    d = _directions(geom, slow)
    sd, v = d["interior blob"].astype(real).astype(np.float64), d["white noise"].astype(real).astype(np.float64)
    plan = _plan(geom, dtype)
    plan.set_gradient("discrete")
    dev = _device_quantities(torch_, plan, slow, kappa, rec, f, bde, sd, v)
    plan.close()
    _compare(dev, _reference_quantities(slow, kappa, args, bde, sd, v), GRAD_TOL if dtype == "c64" else TOL128,
             f"{dtype} n={n} lossy={lossy}:")


@pytest.mark.gpu
@pytest.mark.parametrize("lossy", [False, True])
@pytest.mark.parametrize("dtype", ["c128", "c64"])
def test_parity_on_a_non_square_grid_with_odd_nt_and_device_weights(torch_, dtype, lossy):
    """58 x 90 grid (a partial last row segment), 31 transmitters (complex64 lanes load one source, not two) and (b, d, e) left
    to the device (its min/max(vel) path): the discrete reference is built with the weights the device computed, after
    checking them against the oracle's."""
    from test_shapes_and_edges import H, bde_of, fwi_args, rect_case
    nx, ny = 58, 90
    geom, f, vel_true = rect_case(nx, ny, 31)
    assert geom.tx_include.size % 2 == 1
    rec = observed_data(geom, f, vel_true, bde=bde_of(vel_true, f))
    args = fwi_args(geom, rec, f)
    real = np.float32 if dtype == "c64" else np.float64
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64))
    c0 = 1480.0 + 20.0 * np.exp(-(X ** 2 + Y ** 2) / (2 * (8 * H) ** 2))
    slow = (1.0 / c0).astype(real).astype(np.float64)
    kappa = np.full_like(slow, float(G.db_cm_mhz_to_kappa(10.0))).astype(real).astype(np.float64) if lossy else None
    rng = np.random.default_rng(11)
    sd = (np.exp(-((X - 4 * H) ** 2 + Y ** 2) / (2 * (6 * H) ** 2)) * slow * 1e-2).astype(real).astype(np.float64)
    v = (rng.standard_normal(slow.shape) * slow * 1e-2).astype(real).astype(np.float64)
    plan = _plan(geom, dtype)
    plan.set_gradient("discrete")
    dev = _device_quantities(torch_, plan, slow, kappa, rec, f, None, sd, v)
    bde = plan.bde()[0]
    plan.close()
    vel = 1.0 / slow.astype(real)
    bde_o = np.asarray(oh.stencil_opt_params(float(vel.min()), float(vel.max()), f, H, 1.0, "c128"), dtype=np.float64)
    assert np.allclose(bde, bde_o, rtol=1e-5, atol=0)
    _compare(dev, _reference_quantities(slow, kappa, args, bde, sd, v), GRAD_TOL if dtype == "c64" else TOL128,
             f"{dtype} {nx}x{ny}, 31 transmitters, device (b, d, e), lossy={lossy}:")


@pytest.mark.gpu
def test_parity_at_256_with_the_tcgen05_engine(torch_):
    """256 x 256, 32 transmitters of a 256-element ring, complex64 on the tcgen05 engine, against the complex128 reference."""
    n = 256
    geom = G.ring_geometry(n, 256, dwnsmp=8)
    f = G.frequency_for_grid(n)
    vel_true = G.blob_model(geom)
    c0 = G.blob_model(geom, dc=15.0, seed=99)
    rec = observed_data(geom, f, vel_true, bde=bde_for(geom, vel_true, f))
    slow = (1.0 / c0).astype(np.float32).astype(np.float64)
    bde = bde_for(geom, (1.0 / slow.astype(np.float32)).astype(np.float32), f)
    args = (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab, geom.mask_indices,
            geom.num_elements)
    v = (1.0 / G.blob_model(geom, dc=20.0, seed=5) - 1.0 / c0).astype(np.float32).astype(np.float64)
    plan = _plan(geom, "c64", engine="tc2")
    plan.set_gradient("discrete")
    dev = _device_quantities(torch_, plan, slow, None, rec, f, bde, v, v)
    plan.close()
    _compare(dev, _reference_quantities(slow, None, args, bde, v, v), GRAD_TOL, "256^2 x 32 sources, c64 tcgen05:")


@pytest.mark.gpu
def test_device_gradient_is_the_derivative_of_the_device_loss(torch_):
    """complex128, white-noise direction: <v, grad> against the central difference of the device's own loss; and the line
    search's num = -<sd, grad>."""
    geom, f, c0, bde, rec, args = _case()
    slow = 1.0 / c0
    v = _directions(geom, slow)["white noise"]
    plan = _plan(geom, "c128")
    plan.set_gradient("discrete")
    rt = _dev(torch_, rec[None])
    loss = lambda s: float(plan.fwi_loss_grad(_dev(torch_, s), rt, [f], bde=[bde])[0][0])
    eps = 1e-3
    fd = (loss(slow + eps * v) - loss(slow - eps * v)) / (2 * eps)
    _, g = plan.fwi_loss_grad(_dev(torch_, slow), rt, [f], bde=[bde])
    vg = float(np.sum(v * g.cpu().numpy()))
    num = float(plan.ncg_linesearch(_dev(torch_, v))[0])
    print(f"device: d loss FD {fd:.9e}, <v, grad> {vg:.9e}, num {num:.9e}")
    assert abs(vg - fd) <= 1e-6 * abs(fd)
    assert abs(num + vg) <= 1e-10 * abs(vg)
    plan.close()


def _multi(n=48, nelem=32, nf=4, dtype="c128"):
    geom, f0, vel_true = small_case(n, nelem)
    kt = G.attenuation_blob_model(geom, dalpha=20.0)
    freqs = list(np.linspace(0.8, 1.1, nf) * f0)
    recs = np.ascontiguousarray(np.stack([lossy_observed_data(geom, f, vel_true, kt, seed=11 + i) for i, f in enumerate(freqs)]))
    real = np.float32 if dtype == "c64" else np.float64
    slow = np.full((n, n), 1 / 1490.0, dtype=real)
    kappa = G.attenuation_blob_model(geom, alpha0=5.0, dalpha=10.0, seed=3).astype(real)
    v = (np.random.default_rng(4).standard_normal((n, n)) * slow * 1e-2).astype(real)
    return geom, freqs, recs, slow, kappa, v


@pytest.mark.gpu
def test_four_frequencies_are_the_sum_and_launch_chains_are_bit_identical(torch_):
    geom, freqs, recs, slow, kappa, v = _multi()
    plan = _plan(geom, "c128", nfreq=4)
    plan.set_gradient("discrete")
    st, kt, rt, vt = (_dev(torch_, a) for a in (slow, kappa, recs, v))
    lj, gsj, gkj = (x.clone() for x in plan.fwi_loss_grad_lossy(st, kt, rt, freqs))
    hj, jj = (x.clone() for x in plan.gn_hvp_lossy(vt, vt))
    nj = plan.ncg_linesearch_lossy(vt, vt).cpu().numpy()
    sums = [0.0] * 6
    for i, f in enumerate(freqs):
        l1, gs1, gk1 = plan.fwi_loss_grad_lossy(st, kt, rt[i:i + 1].contiguous(), [f])
        h1, j1 = plan.gn_hvp_lossy(vt, vt)
        n1 = plan.ncg_linesearch_lossy(vt, vt)
        for k, x in enumerate((l1, gs1, gk1, h1, j1, n1)):
            sums[k] = sums[k] + x.cpu().numpy()
    whole = [t.cpu().numpy() if hasattr(t, "cpu") else t for t in (lj, gsj, gkj, hj, jj)] + [nj]
    errs = [rel(a, b) for a, b in zip(whole, sums)]
    print("4 frequencies vs the sum of single ones (loss, grad_s, grad_k, hv, jv2, line search):", [f"{e:.2e}" for e in errs])
    assert max(errs) < 1e-10
    plan.close()
    # two launch chains need >= 8 frequencies (4 per chain): complex64, 8 frequencies
    geom, freqs, recs, slow, kappa, v = _multi(nf=8, dtype="c64")
    plan = _plan(geom, "c64", nfreq=8)
    plan.set_gradient("discrete")
    st, kt, rt, vt = (_dev(torch_, a) for a in (slow, kappa, recs.astype(np.complex64), v))
    res = {}
    for groups in (1, 2, 1):
        plan.set_groups(groups)
        _, gs, gk = plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
        hv, _, jv = plan.gn_hvp_lossy(vt, vt, jv=True)
        cur = (gs.clone(), gk.clone(), hv.clone(), jv.clone())
        if groups in res:
            assert all(torch_.equal(a, b) for a, b in zip(cur, res[groups]))
        res[groups] = cur
    assert all(torch_.equal(a, b) for a, b in zip(res[1], res[2]))
    plan.close()


@pytest.mark.gpu
def test_mode_switching_guards_and_replays(torch_):
    """reference -> discrete -> reference on one plan, graph replays included: the reference results equal a fresh plan's bit
    for bit (the line-search scalars and jv2 are FP64 atomics over CTAs and agree to the last bits).  After a switch, the line
    search and the product refuse until the next evaluation; an invalid mode is rejected."""
    from waveforminversionust_b200 import _lib
    geom, freqs, recs, slow, kappa, v = _multi(nf=2, dtype="c64")
    rt = _dev(torch_, recs.astype(np.complex64))
    st, kt, vt = (_dev(torch_, a) for a in (slow, kappa, v))
    close = lambda x, y: bool(torch_.all(torch_.abs(x - y) <= 1e-12 * torch_.abs(y)))

    def run(plan, lossy):
        if lossy:
            _, gs, gk = plan.fwi_loss_grad_lossy(st, kt, rt, freqs)
            hv, jv2 = plan.gn_hvp_lossy(vt, vt)
            return (gs.clone(), gk.clone(), hv.clone()), (jv2.clone(), plan.ncg_linesearch_lossy(vt, vt).clone())
        _, g = plan.fwi_loss_grad(st, rt, freqs)
        hv, jv2 = plan.gn_hvp(vt)
        return (g.clone(), hv.clone()), (jv2.clone(), plan.ncg_linesearch(vt).clone())

    fresh = _plan(geom, "c64", nfreq=2)
    want = {lossy: run(fresh, lossy) for lossy in (False, True)}
    fresh.close()
    plan = _plan(geom, "c64", nfreq=2)
    for lossy in (False, True):
        first = run(plan, lossy)
        plan.set_gradient("discrete")
        with pytest.raises(_lib.UstError, match="gradient mode"):
            plan.gn_hvp_lossy(vt, vt) if lossy else plan.gn_hvp(vt)
        with pytest.raises(_lib.UstError, match="gradient mode"):
            plan.ncg_linesearch_lossy(vt, vt) if lossy else plan.ncg_linesearch(vt)
        disc = run(plan, lossy)
        run(plan, lossy)  # a replay of the discrete graphs
        plan.set_gradient("reference")
        with pytest.raises(_lib.UstError, match="gradient mode"):
            plan.gn_hvp_lossy(vt, vt) if lossy else plan.gn_hvp(vt)
        again = run(plan, lossy)
        for got in (first, again):
            assert all(torch_.equal(a, b) for a, b in zip(got[0], want[lossy][0]))
            assert all(close(a, b) for a, b in zip(got[1], want[lossy][1]))
        assert not torch_.equal(disc[0][0], want[lossy][0][0])
    with pytest.raises(ValueError):
        plan.set_gradient("exact")
    assert plan.L.ust_plan_set_gradient(plan.h, 2) != 0 and b"mode" in plan.L.ust_last_error()
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shard", ["freq", "source"])
def test_sharded_evaluation_and_products_sum_to_the_whole(torch_, shard):
    from waveforminversionust_b200.distributed import ShardedFWI
    n, nelem = 60, 32
    geom, f0, vel_true = small_case(n, nelem)
    freqs = np.array([0.8, 0.9, 1.0, 1.1]) * f0
    rec_all = _dev(torch_, np.stack([observed_data(geom, f, vel_true, seed=7 + i) for i, f in enumerate(freqs)]).astype(np.complex128))
    slow = _dev(torch_, np.full((n, n), 1.0 / 1485.0))
    v = _dev(torch_, np.random.default_rng(9).standard_normal((n, n)) / 1485.0 * 1e-2)
    whole = ShardedFWI(geom, freqs, dtype="c128", rank=0, world=1, gradient="discrete")
    l_all, g_all = whole.loss_grad_device(slow, rec_all)
    l_all, g_all = float(l_all), g_all.clone()
    h_all, j_all = whole.gn_hvp_device(v)
    h_all, j_all = h_all.clone(), float(j_all)
    whole.close()
    l_sum, g_sum, h_sum, j_sum = 0.0, torch_.zeros_like(g_all), torch_.zeros_like(h_all), 0.0
    for r in range(3):
        part = ShardedFWI(geom, freqs, dtype="c128", rank=r, world=3, shard=shard, gradient="discrete")
        l, g = part.loss_grad_device(slow, part.local_rec(rec_all).contiguous())
        h, j = part.gn_hvp_device(v)
        l_sum += float(l); g_sum += g; h_sum += h; j_sum += float(j)
        part.close()
    errs = (abs(l_sum - l_all) / l_all, rel(g_sum.cpu().numpy(), g_all.cpu().numpy()), rel(h_sum.cpu().numpy(), h_all.cpu().numpy()),
            abs(j_sum - j_all) / j_all)
    print(f"{shard}: shards vs whole (loss, grad, hv, jv2): {errs}")
    assert max(errs) < 1e-12
    assert abs(j_all - float(torch_.sum(v * h_all))) <= 1e-10 * j_all


@pytest.mark.gpu
def test_gauss_newton_driver_on_the_discrete_reference(torch_, monkeypatch):
    """Two outer iterations, cg_iters=4 (complex128): gauss_newton_fwi(gradient="discrete") visits the points of the same
    driver run on the discrete reference's callables."""
    import waveforminversionust_b200 as w
    from waveforminversionust_b200 import api
    geom, f, c0, bde, rec, args = _case()
    st = {}

    def loss_grad(slow):
        st["ref"] = Discrete(slow.cpu().numpy(), 0.0, args, bde)
        pts_o.append(slow.cpu().numpy().copy())
        return st["ref"].loss, st["ref"].grad_s

    def hvp(v):
        return st["ref"].hv(v.cpu().numpy())[0][0]

    dargs = (geom.xi, geom.yi, geom.num_elements, None, geom.dense_src(), geom.tx_include, geom.ind_matlab, 1480.0, f, 2,
             geom.a0, geom.L_PML, geom.mask_indices)
    pts_o, ho = [], []
    vel_o = api.gauss_newton_fwi(*dargs, cg_iters=4, dtype="c128", history=ho, loss_grad=loss_grad, hvp=hvp)
    pts_g, hg = [], []
    orig = api.fwi_loss_function

    def recording(params, *a, **k):
        assert k.get("gradient") == "discrete"
        pts_g.append(params.detach().cpu().numpy().astype(np.float64).copy())
        return orig(params, *a, **k)

    monkeypatch.setattr(api, "fwi_loss_function", recording)
    dargs = dargs[:3] + (rec,) + dargs[4:]
    vel_g = api.gauss_newton_fwi(*dargs, cg_iters=4, dtype="c128", bde=bde, history=hg, gradient="discrete")
    for a, b in zip(ho, hg):
        print(a, "\n", b)
    assert len(pts_g) == len(pts_o) and [h["cg_iters"] for h in hg] == [h["cg_iters"] for h in ho]
    errs = [rel(a, b) for a, b in zip(pts_g, pts_o)]
    print("evaluation points rel:", errs)
    assert max(errs) < 1e-9 and rel(vel_g, vel_o) < 1e-9
    w.clear_plans()
