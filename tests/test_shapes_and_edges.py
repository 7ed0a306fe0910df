"""Shapes and inputs the square ring-array cases never reach, against the complex128 oracle.

A. Non-square grids (CPU): a builder with Nx != Ny and the ``ind_matlab`` decoding of ``api._acquisition``.
B. Assembly planes and forward / adjoint solves on wide and tall grids, at block sizes around the tcgen05 engine's 128-row
   tile and one 64-wide Gauss-Jordan block, the smallest plans, and right-hand-side counts around the 128-column tile.
C. FWI on a non-square grid through the reference surface (lossless, Gauss-Newton, lossy, time domain).
D. The split-K sweep GEMM forced to 1, 2 and 4 CTAs per tile, and a stand-alone solve that must not depend on what the plan
   factorised before.
E. The one-hot row skip of the forward sweeps with hand-placed sources (one row, the chain junction, partial tiles, more
   than eight tiles).
F. Kept receivers of one transmitter that snap to the same node: the adjoint source there is the sum of their residuals.
   The oracle restates the reference's assignment (``.at[].set``, last write wins), which is not the adjoint of the gather,
   so the reference for these cases (``scatter_add_loss_grad``, ``scatter_add_gn_hvp``) lives here.

Every GPU case runs on three engines: complex64 on the tcgen05 engine, complex64 on the FMA engine and complex128."""
from types import SimpleNamespace

import numpy as np
import pytest

from common import observed_data, rel, small_case
from oracle import fwi as ofwi
from oracle import helmholtz as oh
from oracle import timedomain as otd
from waveforminversionust_b200 import api
from waveforminversionust_b200 import geometry as G

WV_TOL = {"c64": 1e-5, "c128": 1e-10}
GRAD_TOL = {"c64": 1e-4, "c128": 1e-8}
LOSS_TOL = {"c64": 1e-4, "c128": 1e-9}
ENGINES = [("c64", "tc2"), ("c64", "simt"), ("c128", "auto")]
ENGINE_IDS = ["c64-tc2", "c64-simt", "c128"]

H = 2.0 ** -8  # grid spacing (m): every node coordinate is exact in float32, so both spacings are exactly H
C_REF = 1480.0


# ---------------------------------------------------------------------------------------------------------------------
# builders
# ---------------------------------------------------------------------------------------------------------------------
def rect_grid(nx, ny, seed=0):
    """(xi, yi, a0, L_PML, f, vel) of an nx x ny grid with spacing H in both directions, centred on the origin, a PML of six
    cells (fewer on grids too small for that), ~5.3 points per wavelength at 1480 m/s and a smooth random blob model."""
    xi = ((np.arange(nx) - (nx - 1) / 2) * H).astype(np.float32)
    yi = ((np.arange(ny) - (ny - 1) / 2) * H).astype(np.float32)
    L_PML = min(6.0, (min(nx, ny) - 1) / 4) * H
    f = C_REF / (5.29 * H)
    vel = G.blob_model(SimpleNamespace(xi=xi, yi=yi), c0=C_REF, dc=60.0, seed=seed + 7, r_max=0.45 * (min(nx, ny) - 1) * H)
    return xi, yi, 10.0, L_PML, f, vel


def rect_case(nx, ny, nelem, seed=0):
    """Ring-array problem on an nx x ny grid (``rect_grid``): ``nelem`` elements on a circle inside the smaller extent that
    clears the PML by two cells, +-floor(31 E / 256) receivers excluded around each transmitter.  ``ind_matlab`` is the
    column-major index x_idx * Ny + y_idx of a (Ny, Nx) field.  Returns (geom, f, vel)."""
    xi, yi, a0, L_PML, f, vel = rect_grid(nx, ny, seed)
    radius = (min(nx, ny) - 1) / 2 * H - L_PML - 2 * H
    theta = -np.pi + 2 * np.pi * np.arange(nelem) / nelem
    x_idx, y_idx = G.snap_elements(xi.astype(np.float64), yi.astype(np.float64), radius * np.cos(theta), radius * np.sin(theta))
    tx = np.arange(nelem)
    geom = G.RingGeometry(xi=xi, yi=yi, x_idx=x_idx, y_idx=y_idx, ind_matlab=x_idx * ny + y_idx, tx_include=tx,
                          mask_indices=G.build_masks(nelem, tx, (31 * nelem) // 256), num_elements=nelem, a0=a0, L_PML=L_PML)
    return geom, f, vel


def bde_of(vel, f):
    return oh.stencil_opt_params(float(np.min(vel)), float(np.max(vel)), f, H, 1.0, "c128")


def fwi_args(geom, rec, f):
    """The arguments after ``params`` of ``fwi_loss_function`` and the oracle's ``fwi_loss_and_grad``."""
    return (geom.xi, geom.yi, rec, geom.dense_src(), f, geom.a0, geom.L_PML, geom.tx_include, geom.ind_matlab,
            geom.mask_indices, geom.num_elements)


def shared_nodes(geom):
    """Number of (transmitter, node) pairs holding more than one kept receiver."""
    nodes = np.take(geom.ind_matlab, geom.mask_indices)
    return sum(int(np.sum(np.unique(row, return_counts=True)[1] > 1)) for row in nodes)


def _adjoint_source(vals, inds, ny, nx):
    """(Ny, Nx, Nt) adjoint source of receiver values ``vals`` (Nt, Nm) at column-major nodes ``inds``: values of receivers that
    share a node are added (``np.add.at``), which makes it the adjoint of ``oracle.fwi.receiver_gather``."""
    nt = vals.shape[0]
    flat = np.zeros((nt, nx * ny), dtype=np.complex128)
    np.add.at(flat, (np.arange(nt)[:, None], inds), vals)
    return np.transpose(flat.reshape(nt, nx, ny), (2, 1, 0))


def scatter_add_loss_grad(slow, geom, rec, f, bde):
    """complex128 ``oracle.fwi.fwi_loss_and_grad`` with the adjoint source of ``_adjoint_source``: the gradient of the loss
    with the source estimates held fixed, also where kept receivers share a node.  Returns (loss, grad, fields)."""
    ny, nx = geom.Ny, geom.Nx
    slow = np.asarray(slow, dtype=np.float64).reshape(ny, nx)
    fac = oh.HelmholtzFactor(geom.xi, geom.yi, 1.0 / slow, f, geom.a0, geom.L_PML, "c128", bde=bde)
    U = fac.solve(geom.dense_src(np.complex128))
    sim, inds = ofwi.receiver_gather(U, geom.ind_matlab, geom.mask_indices)
    recm = np.take_along_axis(np.asarray(rec, dtype=np.complex128), geom.mask_indices, axis=1)
    alpha = ofwi.estimate_src_strength_batched(sim, recm)
    diff = sim * alpha[:, None] - recm
    w = 2 * np.pi * f
    VIRT = 2 * w ** 2 * slow[:, :, None] * U * alpha[None, None, :]
    ADJ = fac.solve(_adjoint_source(diff, inds, ny, nx), True)
    grad = np.sum(-np.real(np.conj(VIRT) * ADJ), axis=2)
    return 0.5 * float(np.sum(np.abs(diff) ** 2)), grad, dict(fac=fac, U=U, alpha=alpha, diff=diff, inds=inds, VIRT=VIRT)


def scatter_add_gn_hvp(v, geom, fields):
    """(H_GN v, J v) of ``scatter_add_loss_grad``'s linearisation: J v gathered at the kept receivers, J^H by ``_adjoint_source``."""
    fac, VIRT = fields["fac"], fields["VIRT"]
    P = fac.solve(-VIRT * np.asarray(v, dtype=np.float64).reshape(geom.Ny, geom.Nx)[:, :, None])
    jv, inds = ofwi.receiver_gather(P, geom.ind_matlab, geom.mask_indices)
    ADJ = fac.solve(_adjoint_source(jv, inds, geom.Ny, geom.Nx), True)
    return np.sum(-np.real(np.conj(VIRT) * ADJ), axis=2), jv


def _directions(geom, n, seed):
    """Smooth slowness perturbations of the size of an FWI update."""
    return [1.0 / G.blob_model(geom, c0=C_REF, dc=20.0, seed=seed + i) - 1.0 / C_REF for i in range(n)]


# ---------------------------------------------------------------------------------------------------------------------
# A. non-square builders (CPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nx,ny", [(90, 60), (60, 90)])
def test_rect_case_builder(nx, ny):
    geom, f, vel = rect_case(nx, ny, 64)
    assert (geom.Nx, geom.Ny) == (nx, ny) and vel.shape == (ny, nx)
    assert np.all(np.diff(geom.xi) == np.float32(H)) and np.all(np.diff(geom.yi) == np.float32(H))
    # every element clears the PML by at least one cell and sits on its own node
    px = np.abs(geom.xi[geom.x_idx].astype(np.float64)) + geom.L_PML + H
    py = np.abs(geom.yi[geom.y_idx].astype(np.float64)) + geom.L_PML + H
    assert np.all(px <= geom.xi[-1]) and np.all(py <= geom.yi[-1])
    assert np.unique(geom.ind_matlab).size == geom.num_elements and shared_nodes(geom) == 0


@pytest.mark.parametrize("nx,ny", [(90, 60), (60, 90)])
def test_acquisition_decodes_ind_matlab_on_a_non_square_grid(nx, ny):
    """``api._acquisition`` turns x_idx * Ny + y_idx back into the node ``snap_elements`` chose (row-major y * Nx + x), the
    oracle's gather reads the same node, and the reference's square-only x_idx * Nx + y_idx names other nodes."""
    geom, f, vel = rect_case(nx, ny, 64)
    src_lin, rx_lin, mask = api._acquisition(geom.dense_src(), geom.ind_matlab, geom.mask_indices, nx, ny)
    assert np.array_equal(rx_lin, geom.y_idx * nx + geom.x_idx)
    assert np.array_equal(src_lin, geom.src_lin) and np.array_equal(mask, geom.mask_indices)
    field = np.arange(ny * nx, dtype=np.float64).reshape(ny, nx)[:, :, None] + np.zeros(geom.tx_include.size)
    got, _ = ofwi.receiver_gather(field, geom.ind_matlab, geom.mask_indices)
    assert np.array_equal(got, np.take(rx_lin, geom.mask_indices).astype(np.float64))
    ref_ind = geom.x_idx * nx + geom.y_idx
    _, rx_ref, _ = api._acquisition(geom.dense_src(), ref_ind, geom.mask_indices, nx, ny)
    print(f"{nx}x{ny}: {int(np.sum(rx_ref != rx_lin))} of {rx_lin.size} receivers land elsewhere with x_idx * Nx + y_idx")
    assert np.sum(rx_ref != rx_lin) > rx_lin.size // 2


# ---------------------------------------------------------------------------------------------------------------------
# F. coinciding receivers: the scatter-add reference (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def _collision_case():
    geom = G.ring_geometry(48, 256)
    f = G.frequency_for_grid(48)
    vel_true = G.blob_model(geom)
    c0 = np.full((48, 48), C_REF)
    bde = oh.stencil_opt_params(C_REF, C_REF, f, float(np.mean(np.diff(geom.xi.astype(np.float64)))), 1.0, "c128")
    return geom, f, vel_true, c0, bde, observed_data(geom, f, vel_true)


def test_scatter_add_reference_is_the_adjoint_where_receivers_share_a_node():
    """On ring_geometry(48, 256) every transmitter has kept receivers on a shared node.  There Re<J w, diff> = <w, grad> and
    <J v, J w> = <v, H_GN w> hold for the scatter-add reference; the oracle's assignment breaks the first.  On a geometry without
    shared nodes the two references agree."""
    geom, f, vel_true, c0, bde, rec = _collision_case()
    assert shared_nodes(geom) > 0
    slow = 1.0 / c0
    loss, grad, fl = scatter_add_loss_grad(slow, geom, rec, f, bde)
    loss_o, grad_o = ofwi.fwi_loss_and_grad(slow, *fwi_args(geom, rec, f), dtype="c128", bde=bde)
    v, w = _directions(geom, 2, 11)
    hw, jw = scatter_add_gn_hvp(w, geom, fl)
    hv, jv = scatter_add_gn_hvp(v, geom, fl)
    lhs, rhs, rhs_o = float(np.real(np.vdot(jw, fl["diff"]))), float(np.sum(w * grad)), float(np.sum(w * grad_o))
    sym = [float(np.real(np.vdot(jv, jw))), float(np.sum(v * hw)), float(np.sum(w * hv))]
    print(f"shared (transmitter, node) pairs {shared_nodes(geom)}; loss {loss:.15e} vs oracle {loss_o:.15e}")
    print(f"Re<Jw, diff> {lhs:.15e}, <w, grad> scatter-add {rhs:.15e}, oracle {rhs_o:.15e}; <Jv,Jw>, <v,Hw>, <w,Hv> {sym}")
    assert abs(loss - loss_o) <= 1e-12 * loss
    assert abs(lhs - rhs) <= 1e-10 * abs(rhs) and abs(lhs - rhs_o) > 1e-3 * abs(rhs)
    assert max(abs(sym[1] - sym[0]), abs(sym[2] - sym[0])) <= 1e-10 * abs(sym[0])
    geom2, f2, vel2 = small_case(48, 32)
    assert shared_nodes(geom2) == 0
    rec2 = observed_data(geom2, f2, vel2)
    l2, g2, _ = scatter_add_loss_grad(slow, geom2, rec2, f2, bde)
    l2o, g2o = ofwi.fwi_loss_and_grad(slow, *fwi_args(geom2, rec2, f2), dtype="c128", bde=bde)
    assert abs(l2 - l2o) <= 1e-13 * l2o and rel(g2, g2o) < 1e-13


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_():
    import torch
    return torch


def _plan(nx, ny, dtype, engine, nrhs, fwi=False, nfreq=1):
    from waveforminversionust_b200 import HelmholtzPlan
    return HelmholtzPlan(nx, ny, dtype=dtype, max_freq=nfreq, max_nrhs=nrhs, fwi_buffers=fwi, engine=engine)


def _dense_rhs(nx, ny, nrhs, seed):
    """Random dense right-hand sides, non-zero (and smaller) on the Dirichlet ring too."""
    rng = np.random.default_rng(seed)
    src = rng.standard_normal((ny, nx, nrhs)) + 1j * rng.standard_normal((ny, nx, nrhs))
    src[0] *= 1e-3; src[-1] *= 1e-3; src[:, 0] *= 1e-3; src[:, -1] *= 1e-3
    return src


def _check_solves(torch_, plan, fac, src, dtype, label):
    ny, nx, nrhs = src.shape
    srcr = src.astype(plan.cplx)
    out = []
    for adjoint in (False, True):
        truth = fac.solve(srcr.astype(np.complex128), adjoint)
        x = torch_.as_tensor(srcr).cuda().reshape(ny * nx, nrhs).contiguous()
        plan.solve(x, 0, adjoint)
        got = x.cpu().numpy().reshape(ny, nx, nrhs)
        err = rel(got, truth)
        print(f"{label} adjoint={adjoint}: rel-L2 {err:.3e}")
        assert err < WV_TOL[dtype], (label, adjoint, err)
        # ring semantics: identity rows (forward) / coupled ring rows (adjoint)
        assert rel(got[0], truth[0]) < 1e-4 and rel(got[:, -1], truth[:, -1]) < 1e-4
        out.append(got)
    assert plan.status() == 0
    return out


SHAPES = [(70, 40), (40, 70), (130, 67), (67, 130), (129, 48), (131, 24), (65, 33), (5, 40), (40, 5), (6, 6), (7, 33), (5, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,engine", ENGINES, ids=ENGINE_IDS)
@pytest.mark.parametrize("nx,ny", SHAPES)
def test_rect_assembly_planes(torch_, dtype, engine, nx, ny):
    xi, yi, a0, L_PML, f, vel = rect_grid(nx, ny)
    bde = bde_of(vel, f)
    plan = _plan(nx, ny, dtype, engine, 4)
    plan.set_grid(xi, yi, a0, L_PML)
    velr = vel.astype(plan.real)
    plan.factor(torch_.as_tensor(velr).cuda(), [f], bde=[bde])
    got = plan.planes(0).cpu().numpy()
    ex, ey = oh.pml_profiles(xi, yi, a0, L_PML, "c128")
    A, B, C = oh._abc(ex, ey)
    P = oh.assemble_planes(nx, ny, 1.0, *bde, H, A, B, C, 2 * np.pi * f / velr.astype(np.float64), "python")
    errs = {name: rel(got[i, 1:-1, 1:-1], P[name]) for i, name in enumerate(oh.PLANE_ORDER)}
    print(f"{dtype} {engine} {nx}x{ny}: worst plane rel-L2 {max(errs.values()):.2e}")
    for i, name in enumerate(oh.PLANE_ORDER):
        assert errs[name] < (2e-6 if dtype == "c64" else 1e-12), (name, errs[name])
        assert np.all(got[i, [0, -1], :] == 0) and np.all(got[i, :, [0, -1]] == 0)
    assert plan.status() == 0
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,engine", ENGINES, ids=ENGINE_IDS)
@pytest.mark.parametrize("nx,ny", SHAPES)
def test_rect_solves(torch_, dtype, engine, nx, ny):
    """Forward and adjoint solves of dense right-hand sides; on (70, 40) and (131, 24) also for 1, 127, 128, 129 and 257
    right-hand sides, around the 128-column tile of the sweeps."""
    xi, yi, a0, L_PML, f, vel = rect_grid(nx, ny)
    bde = bde_of(vel, f)
    counts = [1, 127, 128, 129, 257] if (nx, ny) in ((70, 40), (131, 24)) else [8]
    plan = _plan(nx, ny, dtype, engine, max(counts))
    plan.set_grid(xi, yi, a0, L_PML)
    velr = vel.astype(plan.real)
    plan.factor(torch_.as_tensor(velr).cuda(), [f], bde=[bde])
    fac = oh.HelmholtzFactor(xi, yi, velr.astype(np.float64), f, a0, L_PML, "c128", bde=bde)
    for nrhs in counts:
        _check_solves(torch_, plan, fac, _dense_rhs(nx, ny, nrhs, nx * ny + nrhs), dtype, f"{dtype} {engine} {nx}x{ny} nrhs={nrhs}")
    plan.close()


# ---------------------------------------------------------------------------------------------------------------------
# C. FWI on a non-square grid, through the reference surface with host arrays
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype,engine", ENGINES, ids=ENGINE_IDS)
@pytest.mark.parametrize("nx,ny", [(90, 60), (60, 90)])
def test_rect_fwi_lossless(torch_, dtype, engine, nx, ny):
    import waveforminversionust_b200 as w
    from test_gauss_newton import gn_hvp_ref
    geom, f, vel_true = rect_case(nx, ny, 64)
    rec = observed_data(geom, f, vel_true, bde=bde_of(vel_true, f))
    real = np.float32 if dtype == "c64" else np.float64
    slow = np.full((ny, nx), 1.0 / C_REF).astype(real)
    bde = bde_of(1.0 / slow.astype(np.float64), f)
    args = fwi_args(geom, rec, f)
    loss_t, grad_t, fl = ofwi.fwi_loss_and_grad(slow.astype(np.float64), *args, dtype="c128", bde=bde, return_fields=True)
    loss, grad = w.fwi_loss_function(slow, *args, dtype=dtype, bde=bde, engine=engine)
    plan = w.api.get_plan(nx, ny, dtype, 0, 1, geom.tx_include.size, "python", True, engine)
    e_l, e_g = abs(loss - loss_t) / loss_t, rel(grad, grad_t)
    e_a = rel(plan.src_est(0), fl["SRC_EST"])
    e_u = rel(plan.wavefield(0).cpu().numpy(), fl["WV"] / fl["SRC_EST"][None, None, :])
    v = _directions(geom, 1, 5)[0].astype(real)
    hv = w.fwi_gauss_newton_product(slow, v, *args, dtype=dtype, bde=bde, engine=engine)
    hv_t = gn_hvp_ref(slow.astype(np.float64), v.astype(np.float64), *args, dtype="c128", bde=bde)
    e_h = rel(hv, hv_t)
    print(f"{dtype} {engine} {nx}x{ny}: loss {e_l:.2e}, grad {e_g:.2e}, src_est {e_a:.2e}, wavefield {e_u:.2e}, GN product {e_h:.2e}")
    assert grad.shape == (ny, nx) and hv.shape == (ny, nx)
    assert e_l < LOSS_TOL[dtype] and e_g < GRAD_TOL[dtype] and e_a < LOSS_TOL[dtype]
    assert e_u < WV_TOL[dtype] and e_h < GRAD_TOL[dtype]
    assert plan.status() == 0
    w.clear_plans()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,engine", ENGINES, ids=ENGINE_IDS)
@pytest.mark.parametrize("nx,ny", [(90, 60), (60, 90)])
def test_rect_fwi_lossy_and_time_domain(torch_, dtype, engine, nx, ny):
    import waveforminversionust_b200 as w
    from test_attenuation import lossy_loss_and_grad, lossy_observed_data
    geom, f, vel_true = rect_case(nx, ny, 64)
    kappa_true = G.attenuation_blob_model(geom, dalpha=20.0, r_max=0.07)
    rec = lossy_observed_data(geom, f, vel_true, kappa_true, bde=bde_of(vel_true, f))
    real = np.float32 if dtype == "c64" else np.float64
    slow = np.full((ny, nx), 1.0 / C_REF).astype(real)
    kap = np.full((ny, nx), float(G.db_cm_mhz_to_kappa(10.0))).astype(real)
    bde = bde_of(1.0 / slow.astype(np.float64), f)
    args = fwi_args(geom, rec, f)
    loss_t, gs_t, gk_t = lossy_loss_and_grad(slow.astype(np.float64), *args, kappa=kap.astype(np.float64), dtype="c128", bde=bde)
    loss, grad = w.fwi_joint_loss_function(np.stack([slow, kap]), *args, dtype=dtype, bde=bde, engine=engine)
    e_l, e_s, e_k = abs(loss - loss_t) / loss_t, rel(grad[0], gs_t), rel(grad[1], gk_t)
    # time domain: a few frequencies and time samples of one transmitter's field
    fs = np.linspace(0.6 * f, f, 4)
    resp = otd.hanning(fs.size)
    time = np.linspace(0.0, 2 * (max(nx, ny) - 1) * H / 1500.0, 9)
    src = geom.dense_src(np.complex128)[:, :, 5]
    velr = vel_true.astype(real)  # both sides get the sound speed the device holds, so the errors are the solver's
    WFo, WTo = otd.time_domain_simulation(geom.xi, geom.yi, velr.astype(np.float64), src, fs, resp, time, geom.a0, geom.L_PML,
                                          dtype="c128")
    WF, WT = w.time_domain_simulation(geom.xi, geom.yi, velr, src, fs, resp, time, geom.a0, geom.L_PML, dtype=dtype,
                                      engine=engine, batch=2)
    e_f, e_t = rel(WF, WFo), rel(WT, WTo)
    print(f"{dtype} {engine} {nx}x{ny}: lossy loss {e_l:.2e}, grad_s {e_s:.2e}, grad_kappa {e_k:.2e}; "
          f"frequency stack {e_f:.2e}, time samples {e_t:.2e}")
    assert grad.shape == (2, ny, nx) and WT.shape == (ny, nx, time.size)
    assert e_l < LOSS_TOL[dtype] and e_s < GRAD_TOL[dtype] and e_k < GRAD_TOL[dtype]
    td_tol = 1e-5 if dtype == "c64" else 1e-9
    assert e_f < td_tol and e_t < td_tol
    w.clear_plans()


# ---------------------------------------------------------------------------------------------------------------------
# D. split-K sweeps
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_split_k_settings_agree_with_the_reference_and_each_other(torch_, monkeypatch):
    """(258, 48): nI = 256 is 16 k-chunks and one frequency at 128 right-hand sides is 4 tiles, so the sweep GEMM may split
    each tile's k range over clusters of 2 or 4 CTAs.  UST_KSPLIT (read at plan creation) forces 1, 2 and 4.  The factors are
    the same bits under every setting, and each split adds the k range in its own order, so the three settings must differ
    in the last bits: the witness that each cluster path ran."""
    nx, ny, nrhs = 258, 48, 128
    xi, yi, a0, L_PML, f, vel = rect_grid(nx, ny)
    bde = bde_of(vel, f)
    velr = vel.astype(np.float32)
    fac = oh.HelmholtzFactor(xi, yi, velr.astype(np.float64), f, a0, L_PML, "c128", bde=bde)
    src = _dense_rhs(nx, ny, nrhs, 3)
    out = {}
    for ks in ("1", "2", "4"):
        monkeypatch.setenv("UST_KSPLIT", ks)
        plan = _plan(nx, ny, "c64", "tc2", nrhs)
        plan.set_grid(xi, yi, a0, L_PML)
        plan.factor(torch_.as_tensor(velr).cuda(), [f], bde=[bde])
        out[ks] = _check_solves(torch_, plan, fac, src, "c64", f"UST_KSPLIT={ks}")
        again = _check_solves(torch_, plan, fac, src, "c64", f"UST_KSPLIT={ks} again")
        assert all(np.array_equal(a, b) for a, b in zip(out[ks], again)), ks
        plan.close()
    monkeypatch.delenv("UST_KSPLIT")
    for ks, base in (("2", "1"), ("4", "1"), ("4", "2")):
        d = [rel(a, b) for a, b in zip(out[ks], out[base])]
        print(f"UST_KSPLIT={ks} vs {base}: forward {d[0]:.2e}, adjoint {d[1]:.2e}")
        assert max(d) < WV_TOL["c64"]
        assert not any(np.array_equal(a, b) for a, b in zip(out[ks], out[base])), (ks, base)


@pytest.mark.gpu
def test_stand_alone_solve_does_not_depend_on_the_last_factorisation_size(torch_, monkeypatch):
    """The split-K choice of a stand-alone solve is made from that solve: solving frequency 0 after factorising it alone and
    after factorising it with 39 others (enough tiles that an evaluation of all 40 would not split) gives the same bits."""
    monkeypatch.delenv("UST_KSPLIT", raising=False)
    nx, ny, nrhs, nf = 258, 48, 128, 40
    xi, yi, a0, L_PML, f, vel = rect_grid(nx, ny)
    velr = vel.astype(np.float32)
    freqs = [f] + list(np.linspace(0.6 * f, 0.99 * f, nf - 1))
    bdes = [bde_of(velr, fk) for fk in freqs]
    src = _dense_rhs(nx, ny, nrhs, 4).astype(np.complex64)
    plan = _plan(nx, ny, "c64", "tc2", nrhs, nfreq=nf)
    plan.set_grid(xi, yi, a0, L_PML)
    got = []
    for k in (1, nf):
        plan.factor(torch_.as_tensor(velr).cuda(), freqs[:k], bde=bdes[:k])
        for adjoint in (False, True):
            x = torch_.as_tensor(src).cuda().reshape(ny * nx, nrhs).contiguous()
            plan.solve(x, 0, adjoint)
            got.append(x.cpu().numpy())
    assert plan.status() == 0
    plan.close()
    d = [rel(got[2], got[0]), rel(got[3], got[1])]
    print(f"frequency 0 after factorising 1 vs {nf} frequencies: forward {d[0]:.2e}, adjoint {d[1]:.2e}")
    assert np.array_equal(got[0], got[2]) and np.array_equal(got[1], got[3])


# ---------------------------------------------------------------------------------------------------------------------
# E. one-hot row skip of the forward sweeps
# ---------------------------------------------------------------------------------------------------------------------
def _onehot_rows(case, M, rng):
    """Interior block rows (node row - 1) of the sources, 128 sources to a column tile."""
    mid = M // 2
    if case == "tile0_first_row_tile1_last_row":
        return [0] * 128 + [M - 1] * 128
    if case == "rows_around_mid":
        return [mid - 1, mid, mid + 1] * 64
    if case == "one_tile_both_ends":
        return [0, M - 1] * 64
    if case == "one_column_last_tile":
        return list(rng.integers(0, M, 128)) + [mid]
    return list(rng.integers(0, M, 1025))  # more than eight tiles: no row skip


ONEHOT_CASES = ["tile0_first_row_tile1_last_row", "rows_around_mid", "one_tile_both_ends", "one_column_last_tile", "nt_1025"]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,engine", ENGINES, ids=ENGINE_IDS)
@pytest.mark.parametrize("nx,ny", [(70, 40), (40, 70)])
@pytest.mark.parametrize("case", ONEHOT_CASES)
def test_onehot_row_skip(torch_, dtype, engine, nx, ny, case):
    rng = np.random.default_rng(len(case) + nx)
    rows = np.asarray(_onehot_rows(case, ny - 2, rng))
    nt = rows.size
    xs = 1 + (np.arange(nt) * 7) % (nx - 2)
    src_lin = ((rows + 1) * nx + xs).astype(np.int32)
    nelem = 24
    rx = rng.choice([y * nx + x for y in range(1, ny - 1) for x in range(1, nx - 1)], nelem, replace=False)
    rx_x, rx_y = rx % nx, rx // nx
    mask = np.tile(np.arange(nelem), (nt, 1))
    rec = rng.standard_normal((nt, nelem)) + 1j * rng.standard_normal((nt, nelem))
    xi, yi, a0, L_PML, f, vel = rect_grid(nx, ny)
    real = np.float32 if dtype == "c64" else np.float64
    slow = (1.0 / vel).astype(real)
    bde = bde_of(1.0 / slow.astype(np.float64), f)
    plan = _plan(nx, ny, dtype, engine, nt, fwi=True)
    plan.set_grid(xi, yi, a0, L_PML)
    plan.set_acquisition(src_lin, rx.astype(np.int32), mask)
    loss, grad = plan.fwi_loss_grad_host(slow, rec[None], [f], bde=[bde])
    U = plan.wavefield(0).cpu().numpy()
    SRC = np.zeros((ny, nx, nt), dtype=np.complex128)
    SRC[rows + 1, xs, np.arange(nt)] = 1.0
    vel64 = 1.0 / slow.astype(np.float64)
    truth = oh.HelmholtzFactor(xi, yi, vel64, f, a0, L_PML, "c128", bde=bde).solve(SRC.astype(np.complex128))
    loss_t, grad_t = ofwi.fwi_loss_and_grad(slow.astype(np.float64), xi, yi, rec, SRC, f, a0, L_PML, np.arange(nt),
                                            rx_x * ny + rx_y, mask, nelem, dtype="c128", bde=bde)
    e_u, e_l, e_g = rel(U, truth), abs(loss - loss_t) / loss_t, rel(grad, grad_t)
    worst = max(range(nt), key=lambda t: rel(U[:, :, t], truth[:, :, t]))
    print(f"{dtype} {engine} {nx}x{ny} {case} (nt={nt}): wavefield {e_u:.2e} (worst column {worst}: "
          f"{rel(U[:, :, worst], truth[:, :, worst]):.2e}), loss {e_l:.2e}, grad {e_g:.2e}")
    assert e_u < WV_TOL[dtype] and rel(U[:, :, worst], truth[:, :, worst]) < 10 * WV_TOL[dtype]
    assert e_l < LOSS_TOL[dtype] and e_g < GRAD_TOL[dtype]
    assert plan.status() == 0
    plan.close()


# ---------------------------------------------------------------------------------------------------------------------
# F. coinciding receivers on the GPU
# ---------------------------------------------------------------------------------------------------------------------
def _collision_plan(geom, dtype, engine):
    plan = _plan(geom.Nx, geom.Ny, dtype, engine, geom.tx_include.size, fwi=True)
    plan.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
    plan.set_acquisition(geom.src_lin, (geom.y_idx * geom.Nx + geom.x_idx).astype(np.int32), geom.mask_indices)
    return plan


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,engine", ENGINES, ids=ENGINE_IDS)
def test_coinciding_receivers_match_the_scatter_add_reference(torch_, dtype, engine):
    geom, f, vel_true, c0, bde, rec = _collision_case()
    real = np.float32 if dtype == "c64" else np.float64
    slow = (1.0 / c0).astype(real)
    loss_t, grad_t, fl = scatter_add_loss_grad(slow, geom, rec, f, bde)
    v = _directions(geom, 1, 11)[0].astype(real)
    hv_t, _ = scatter_add_gn_hvp(v.astype(np.float64), geom, fl)
    plan = _collision_plan(geom, dtype, engine)
    loss, grad = plan.fwi_loss_grad_host(slow, rec[None], [f], bde=[bde])
    hv, _ = plan.gn_hvp(torch_.as_tensor(v).cuda())
    e_l, e_g, e_h = abs(loss - loss_t) / loss_t, rel(grad, grad_t), rel(hv.cpu().numpy(), hv_t)
    print(f"{dtype} {engine}: loss {e_l:.2e}, grad {e_g:.2e}, GN product {e_h:.2e}")
    assert e_l < LOSS_TOL[dtype] and e_g < GRAD_TOL[dtype] and e_h < GRAD_TOL[dtype]
    assert plan.status() == 0
    plan.close()


@pytest.mark.gpu
def test_coinciding_receivers_adjoint_identities_and_determinism(torch_):
    """complex128 on ring_geometry(48, 256), on the device's own quantities:
    - the reported loss is 0.5 |alpha u - rec|^2 over every kept receiver;
    - the gradient is J^H of that residual: <w, grad> = Re<J w, diff> in several directions (J v from the Gauss-Newton
      product; J leaves out the stencil's mass weights, as the reference does, so a finite difference of the loss differs
      from it by ~12 % and cannot be the yardstick);
    - the Gauss-Newton product is symmetric: <J v, J w> = <v, H w> = <w, H v>;
    - two evaluations and two products give the same gradient and product bits."""
    geom, f, vel_true, c0, bde, rec = _collision_case()
    slow = 1.0 / c0
    plan = _collision_plan(geom, "c128", "auto")
    loss, grad = plan.fwi_loss_grad_host(slow, rec[None], [f], bde=[bde])
    grad = grad.copy()
    alpha = plan.src_est(0)
    sim, _ = ofwi.receiver_gather(plan.wavefield(0).cpu().numpy() * alpha[None, None, :], geom.ind_matlab, geom.mask_indices)
    diff = sim - np.take_along_axis(rec, geom.mask_indices, axis=1)
    e_loss = abs(0.5 * float(np.sum(np.abs(diff) ** 2)) - loss) / loss
    dirs = _directions(geom, 3, 21)
    prods = [plan.gn_hvp(torch_.as_tensor(d).cuda(), jv=True) for d in dirs]
    hs = [p[0].cpu().numpy() for p in prods]
    js = [p[2].cpu().numpy()[0] for p in prods]
    e_adj = [abs(float(np.real(np.vdot(j, diff))) - float(np.sum(d * grad))) / abs(float(np.sum(d * grad))) for d, j in zip(dirs, js)]
    jj = float(np.real(np.vdot(js[0], js[1])))
    e_sym = max(abs(float(np.sum(dirs[0] * hs[1])) - jj), abs(float(np.sum(dirs[1] * hs[0])) - jj)) / abs(jj)
    print(f"loss vs 0.5|diff|^2 {e_loss:.2e}; <w, grad> vs Re<Jw, diff> {[f'{e:.2e}' for e in e_adj]}; symmetry {e_sym:.2e}")
    assert e_loss < 1e-12 and max(e_adj) < 1e-10 and e_sym < 1e-10
    h_again = plan.gn_hvp(torch_.as_tensor(dirs[0]).cuda())[0].cpu().numpy()
    loss2, grad2 = plan.fwi_loss_grad_host(slow, rec[None], [f], bde=[bde])
    # (the loss is a sum of per-transmitter atomics, so only its last bits may move)
    assert abs(loss2 - loss) <= 1e-13 * loss and np.array_equal(grad2, grad) and np.array_equal(h_again, hs[0])
    assert plan.status() == 0
    plan.close()
