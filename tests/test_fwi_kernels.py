"""Per-entry parity of the FWI kernels that run after the sweeps, each held to its own arithmetic.

The end-to-end tests compare against the oracle, so for complex64 their bar is the solver's (1e-4 relative L2).  That hides a
kernel error below the solver's noise, and a relative L2 over the whole output hides an error in a few entries.  Here every
kernel is compared, entry by entry, with a float64 restatement of itself evaluated on the device's OWN inputs (fields, source
estimates, coefficient planes and stencil weights read back from the plan, promoted to float64):

    receiver_kernel        alpha, loss, adjoint source            gradient_kernel / gradient_mass_kernel     grad_s, grad_kappa
    pert_rhs_kernel / pert_rhs_mass_kernel   perturbation RHS     linesearch_kernel                          num, den
    gn_receiver_kernel / gn_scatter_kernel   J v, sum |J v|^2 and J v as the adjoint source of the product

A direct output must satisfy |dev - ref| <= (gamma u_R + depth u_64) S entry by entry, where S is the entry's magnitude sum,
u_R the unit roundoff of the field type, gamma the number of roundings in type R on the way to one entry and depth the number
of FP64 roundings (``kernel_tol`` derives both from the kernel's operations).  The adjoint source and the perturbation RHS
are consumed by a solve, so they are recovered through the operator: H P (H^H Lambda) from the device's nine coefficient
planes against the restated RHS, with the solve's share bounded by 4 beta |H||P|, beta the backward error of the plan's own
forward solves.  The CPU tests validate the restatements against the oracle and show that the bars catch subtle bugs: numpy
float32 emulations of the kernels pass them, and each mutated emulation fails them by at least 10x."""
import math

import numpy as np
import pytest

from common import observed_data, rel
from oracle import fwi as ofwi
from oracle import helmholtz as oh
from test_discrete_gradient import Discrete
from test_shapes_and_edges import C_REF, _adjoint_source, _collision_case, bde_of, fwi_args, rect_case, scatter_add_gn_hvp, \
    scatter_add_loss_grad
from waveforminversionust_b200 import geometry as G

U32, U64 = 2.0 ** -24, 2.0 ** -53
UNIT = {"c64": U32, "c128": U64}
# Gradual underflow: below the smallest normal number an operation's error is absolute, at most half the spacing of the
# subnormals.  The gradient kernels multiply two fields that both decay in the PML, so at a 256^2 grid's PML corners the float32
# products of alpha u and lambda fall below 1e-38 and keep few or no significant bits.
ETA = {U32: 2.0 ** -150, U64: 2.0 ** -1075}
OFFS = tuple(oh._OFFS[name] for name in oh.PLANE_ORDER)  # (dy, dx) of the planes c, l, r, d, u, dl, dr, ul, ur


# ---------------------------------------------------------------------------------------------------------------------
# float64 restatements (fields are (nf, Ny, Nx, nt), source estimates (nf, nt), data (nf, nt, nelem))
# ---------------------------------------------------------------------------------------------------------------------
def shift(X, dy, dx):
    """Y[y, x] = X[y + dy, x + dx] over the first two axes, zero off the grid."""
    Y = np.zeros_like(X)
    ny, nx = X.shape[:2]
    Y[max(0, -dy):ny - max(0, dy), max(0, -dx):nx - max(0, dx)] = X[max(0, dy):ny - max(0, -dy), max(0, dx):nx - max(0, -dx)]
    return Y


def interior(ny, nx):
    m = np.zeros((ny, nx), dtype=bool)
    m[1:-1, 1:-1] = True
    return m


def apply_H(planes, X, absolute=False):
    """H X (absolute: |H||X|) from the nine coefficient planes (9, Ny, Nx) of one frequency; ring rows are identity rows."""
    P, X = (np.abs(planes), np.abs(X)) if absolute else (planes, X)
    out = X.copy()
    inner = sum(P[p][:, :, None] * shift(X, dy, dx) for p, (dy, dx) in enumerate(OFFS))
    out[1:-1, 1:-1] = inner[1:-1, 1:-1]
    return out


def apply_HH(planes, X, absolute=False):
    """H^H X (absolute: |H|^T |X|): interior row i adds conj(H_ij) X_i to entry j, ring rows add X_i to entry i.  So the ring of
    H^H X is X_ring plus the interior rows next to it, the coupling the adjoint solve's ring_fix solves for (DESIGN.md section 5)."""
    P, X = (np.abs(planes), np.abs(X)) if absolute else (np.conj(planes), X)
    inside = interior(*X.shape[:2])[:, :, None]
    out = np.where(inside, 0, X)
    for p, (dy, dx) in enumerate(OFFS):
        out = out + shift(np.where(inside, P[p][:, :, None] * X, 0), -dy, -dx)
    return out


def mass_weights(bde, dtype=np.float64):
    """Stencil mass weights of the nine offsets: 1-d-e at the centre, d/4 at the edges, e/4 at the corners."""
    _, d, e = (float(x) for x in bde)
    return np.array([1 - d - e] + [d / 4] * 4 + [e / 4] * 4).astype(dtype)


def mass_W(X, bde, ring=False, absolute=False):
    """(W X)_j = sum_{i in N9(j)} w_ij X_i over interior rows i (ring: over every row i)."""
    w = mass_weights(bde, X.real.dtype)
    if absolute:
        X, w = np.abs(X), np.abs(w)
    if not ring:
        X = np.where(interior(*X.shape[:2])[:, :, None], X, 0)
    return sum(w[p] * shift(X, dy, dx) for p, (dy, dx) in enumerate(OFFS))


def pml_factor(geom):
    """C = e_x e_y at the nodes (oracle.helmholtz.pml_profiles)."""
    ex, ey = oh.pml_profiles(geom.xi, geom.yi, geom.a0, geom.L_PML, "c128")
    return ey[::2][:, None] * ex[::2][None, :]


def gather(F, rx_lin, mask):
    """F at the kept receivers of every transmitter, mask order: (nf, nt, nm)."""
    nf, ny, nx, nt = F.shape
    return F.reshape(nf, ny * nx, nt)[:, rx_lin[mask], np.arange(nt)[:, None]]


def scatter_add(vals, rx_lin, mask, shape, last_write_wins=False):
    """Receiver values (nf, nt, nm) added into (nf, Ny, Nx, nt) per node (last_write_wins: assigned instead)."""
    nf, ny, nx, nt = shape
    out = np.zeros((nf, ny * nx, nt), dtype=vals.dtype)
    idx = (np.arange(nf)[:, None, None], rx_lin[mask][None], np.arange(nt)[None, :, None])
    if last_write_wins:
        out[idx] = vals
    else:
        np.add.at(out, idx, vals)
    return out.reshape(shape)


def receiver_ref(U, rec, rx_lin, mask, alpha):
    """receiver_kernel with the device's alpha for the residual: alpha_ref and its magnitude sum, the loss and its magnitude sum,
    the adjoint source (residuals added per node) and its magnitude sum."""
    sim = gather(U, rx_lin, mask)
    ob = np.take_along_axis(rec, np.broadcast_to(mask, (rec.shape[0],) + mask.shape), axis=2)
    den = np.sum(np.abs(sim) ** 2, axis=2)
    out = dict(alpha=np.sum(np.conj(sim) * ob, axis=2) / den, S_alpha=np.sum(np.abs(sim) * np.abs(ob), axis=2) / den)
    d = alpha[:, :, None] * sim - ob
    mag = np.abs(alpha)[:, :, None] * np.abs(sim) + np.abs(ob)
    out.update(loss=0.5 * float(np.sum(np.abs(d) ** 2)), S_loss=float(np.sum(np.abs(d) * mag)), diff=d,
               adj=scatter_add(d, rx_lin, mask, U.shape), S_adj=scatter_add(mag, rx_lin, mask, U.shape))
    return out


def z_reference(U, lam, alpha):
    """z_f = sum_t conj(alpha_t u_t) lambda_t of gradient_kernel, its magnitude sum and its underflow sum (nf, Ny, Nx): per
    source, the two products of alpha u (one absolute error each) and their sum reach z times |lambda|, the products with lambda
    and the sums reach it directly."""
    au = alpha[:, None, None, :] * U
    return np.sum(np.conj(au) * lam, axis=3), np.sum(np.abs(au) * np.abs(lam), axis=3), np.sum(3 * np.abs(lam) + 3, axis=3)


def z_mass(U, lam, alpha, C, bde, Wl=None):
    """z_f = conj(C) sum_t conj(alpha_t u_t) (W lambda_t) of gradient_mass_kernel (W skips ring rows), its magnitude sum and its
    underflow sum (alpha u as in z_reference, times |W lambda|; the nine weight products and eight sums of W lambda, times
    |alpha u|; the products and sums of z).  ``Wl`` replaces W lambda."""
    au = alpha[:, None, None, :] * U
    if Wl is None:
        Wl = np.stack([mass_W(lam[f], bde[f]) for f in range(U.shape[0])])
    Wa = np.stack([mass_W(lam[f], bde[f], absolute=True) for f in range(U.shape[0])])
    z = np.conj(C) * np.sum(np.conj(au) * Wl, axis=3)
    return z, np.abs(C) * np.sum(np.abs(au) * Wa, axis=3), np.abs(C) * np.sum(3 * Wa + 17 * np.abs(au) + 3, axis=3)


def gradient_from_z(z, Sz, Sz_abs, freqs, slow, kappa):
    """A = sum_f -2 w^2 Re z, B = sum_f -2 w^2 Im z, grad_s = s A - kappa B, grad_kappa = -s B - kappa A, and the magnitude
    sum (|s| + |kappa|) sum_f 2 w^2 S_z of both (S_abs: the same of the underflow sum)."""
    q = 2.0 * (2.0 * np.pi * np.asarray(freqs, dtype=np.float64)) ** 2
    A = -np.tensordot(q, z.real.astype(np.float64), 1)
    B = -np.tensordot(q, z.imag.astype(np.float64), 1)
    k = np.zeros_like(slow) if kappa is None else kappa
    m = np.abs(slow) + np.abs(k)
    return dict(grad_s=slow * A - k * B, grad_k=-slow * B - k * A, A=A, S=m * np.tensordot(q, Sz, 1),
                S_abs=m * np.tensordot(q, Sz_abs, 1))


def rhs_coefficient(freqs, slow, kappa, ds, dk):
    """c = -2 w^2 sigma dsigma, sigma = s - i kappa, dsigma = ds - i dk: (nf, Ny, Nx)."""
    q = 2.0 * (2.0 * np.pi * np.asarray(freqs, dtype=np.float64)) ** 2
    sig = slow - 1j * (0.0 if kappa is None else kappa)
    dsig = ds - 1j * (0.0 if dk is None else dk)
    return -q[:, None, None] * (sig * dsig)[None]


def rhs_reference(U, alpha, c):
    """pert_rhs_kernel: c alpha_t u_t, and its magnitude sum."""
    v = alpha[:, None, None, :] * U
    return c[..., None] * v, np.abs(c)[..., None] * np.abs(v)


def rhs_mass(U, alpha, cC, bde, keep_ring_rows=False):
    """pert_rhs_mass_kernel: alpha_t sum_{j in N9(i)} w_ij (C c)_j u_tj on interior rows i, 0 on the ring; and its magnitude sum.
    ``cC`` = C c."""
    nf = U.shape[0]
    cu = cC[..., None] * U
    out = np.stack([alpha[f] * mass_W(cu[f], bde[f], ring=True) for f in range(nf)])
    S = np.stack([np.abs(alpha[f]) * mass_W(cu[f], bde[f], ring=True, absolute=True) for f in range(nf)])
    if not keep_ring_rows:
        ring = ~interior(*U.shape[1:3])[None, :, :, None]
        out, S = np.where(ring, 0, out), np.where(ring, 0, S)
    return out, S


def linesearch_ref(U, P, alpha, rec, rx_lin, mask):
    """linesearch_kernel: num = sum Re(conj(P)(rec - alpha U)), den = sum |P|^2 over the kept receivers, with magnitude sums."""
    sim, p = gather(U, rx_lin, mask), gather(P, rx_lin, mask)
    ob = np.take_along_axis(rec, np.broadcast_to(mask, (rec.shape[0],) + mask.shape), axis=2)
    r = ob - alpha[:, :, None] * sim
    return dict(num=float(np.sum((np.conj(p) * r).real)), den=float(np.sum(np.abs(p) ** 2)),
                S_num=float(np.sum(np.abs(p) * (np.abs(alpha)[:, :, None] * np.abs(sim) + np.abs(ob)))),
                S_den=float(np.sum(np.abs(p) ** 2)))


def nodes_shared(rx_lin, mask):
    """Largest number of kept receivers of one transmitter on one node."""
    return max(int(np.max(np.unique(row, return_counts=True)[1])) for row in rx_lin[mask])


# ---------------------------------------------------------------------------------------------------------------------
# bars
# ---------------------------------------------------------------------------------------------------------------------
def kernel_tol(kernel, dtype, nt, nm=1, nf=1, nshare=1):
    """(gamma, depth) of a kernel: |dev - ref| <= (gamma u_R + depth u_64) S.  gamma counts the roundings in the field type R
    (float32 for complex64, float64 for complex128) on the way to one entry, relative to that entry's magnitude sum S; depth
    counts the FP64 roundings (sums of FP64 partials, warp and block trees, atomics over CTAs, products of FP64 values).  A
    complex product rounds each part twice (two products, one sum): 2 u |a||b|."""
    lanes_serial = math.ceil(nt / 32)  # sources (or units of two) a lane accumulates one after the other
    blk = math.ceil(nm / 256) + 8      # a block_sum over 256 threads: per-thread serial sum, 5 warp and 3 CTA levels
    vec = dtype == "c64" and nt % 2 == 0
    if kernel == "gradient":
        # alpha u (2), the cast of the gradient (1); the complex64 vector path sums Re / Im into four FP32 partials of
        # ceil(nt/64) terms each; every other path sums products in FP64 per lane (nt/32), then a warp tree (5), the
        # frequency sum, -2 w^2 (3), the products with s and kappa and their difference (3), two roundings per product (2)
        return 3 + (math.ceil(nt / 64) if vec else 0), lanes_serial + nf + 13
    if kernel == "gradient_mass":
        # alpha u (2); W lambda in R: two sums of pairs and their sum for the edges and the corners (2), three weight casts and
        # products and two sums (4); Re / Im of conj(alpha u) W lambda (2); z accumulated in R over ceil(nt/32) + 1 terms per
        # lane; e_x, e_y held in R on the device, C here from float64 profiles (2); the cast of the gradient (1)
        return 14 + lanes_serial, nf + 13
    if kernel == "rhs":
        # the FP64 coefficient's cast (1, complex: 2 parts), alpha u (2), c (alpha u) (2)
        return 6, 6
    if kernel == "rhs_mass":
        # the coefficient's cast (1), c u (2), W in R (6), alpha (W c u) (2), e_x, e_y in R (2)
        return 14, 8
    if kernel == "alpha":
        # FP64 sums of products of R values, the division, the cast (relative to |alpha|: gamma applies to |alpha|, depth to S)
        return 2, blk + 4
    if kernel == "loss":
        # d = alpha sim - rec in R: 2 (product) + 1 (difference) + 1 (alpha's cast); |d|^2 doubles the relative error, the
        # 1/2 halves it back; FP64: products, the block sum and the atomics over nt * nf CTAs
        return 5, blk + nt * nf + 3
    if kernel == "adjoint":
        # d (4) plus one addition per further receiver on the node
        return 4 + nshare, 0
    if kernel == "num":
        # rec - alpha U in R (3) plus alpha's own rounding (1); FP64 products, block sum, atomics
        return 4, blk + nt * nf + 3
    if kernel == "den":
        # products of R values are exact in FP64 for complex64; FP64 products, block sum, atomics
        return 0, blk + nt * nf + 3
    if kernel == "jv_scatter":
        # J v copied, or added over the receivers of one node
        return nshare - 1, 0
    raise ValueError(kernel)


def _ratio(err, bound):
    err, bound = np.broadcast_arrays(np.asarray(err, dtype=np.float64), np.asarray(bound, dtype=np.float64))
    out = np.zeros(err.shape)
    np.divide(err, bound, out=out, where=bound > 0)
    out[(bound <= 0) & (err > 0)] = np.inf
    return out


def report(label, ratio, axes):
    """Worst err / bound, printed with its location; axes names the dimensions of ``ratio``."""
    ratio = np.atleast_1d(ratio)
    i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    loc = dict(zip(axes, (int(k) for k in i)))
    if "x" in loc:
        loc["x mod 4"] = loc["x"] % 4
    where = ", ".join(f"{k} {v}" for k, v in loc.items())
    print(f"  {label:28s} worst err/bound {float(ratio[i]):9.3e}" + (f"  at {where}" if where else ""))
    return float(ratio[i])


def direct(label, dev, ref, S, tol, u, axes=("f", "y", "x"), S_depth=None, S_abs=None):
    """|dev - ref| <= (gamma u_R) S + (depth u_64) S_depth + eta_R S_abs entry by entry."""
    gamma, depth = tol
    bound = gamma * u * np.asarray(S) + depth * U64 * np.asarray(S if S_depth is None else S_depth)
    if S_abs is not None:
        bound = bound + ETA[u] * np.asarray(S_abs)
    return report(label, _ratio(np.abs(np.asarray(dev) - np.asarray(ref)), bound), axes)


def backward_error(planes, U, src_lin):
    """Backward error of the plan's forward solves H u_t = e_src(t), from its own fields: normwise, the largest over the columns
    of ||H u_t - e_src|| / || |H||u_t| || (what ust_residual_onehot computes); per entry, the largest |H u - e| over the largest
    |H||u| of the same grid row, column and frequency."""
    nf, ny, nx, nt = U.shape
    norm = row = 0.0
    for f in range(nf):
        r = apply_H(planes[f], U[f]).reshape(ny * nx, nt)
        r[src_lin, np.arange(nt)] -= 1.0
        r = r.reshape(ny, nx, nt)
        M = apply_H(planes[f], U[f], absolute=True)
        norm = max(norm, float(np.max(np.linalg.norm(r, axis=(0, 1)) / np.linalg.norm(M, axis=(0, 1)))))
        row = max(row, float(np.max(_ratio(np.abs(r), np.max(M, axis=1, keepdims=True)))))
    return norm, row


def behind_solve(label, planes, X, rhs, S, tol, u, beta, adjoint):
    """The RHS a solve consumed, recovered through the operator: with r = H X - rhs (adjoint: H^H X - rhs) and M = |H||X|,
    ||r|| <= 4 beta_norm ||M|| + (gamma u_R + depth u_64) ||S||, and for every entry |r| <= 4 beta_row max_row(M) + (...) S."""
    gamma, depth = tol
    t = gamma * u + depth * U64
    op = apply_HH if adjoint else apply_H
    r = np.stack([op(planes[f], X[f]) - rhs[f] for f in range(X.shape[0])])
    M = np.stack([op(planes[f], X[f], absolute=True) for f in range(X.shape[0])])
    a = report(label + " (norm)", _ratio(np.linalg.norm(r), 4 * beta[0] * np.linalg.norm(M) + t * np.linalg.norm(S)), ())
    b = report(label + " (entry)", _ratio(np.abs(r), 4 * beta[1] * np.max(M, axis=2, keepdims=True) + t * S), ("f", "y", "x", "t"))
    return max(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# one evaluation, one line search and one product checked against the restatements
# ---------------------------------------------------------------------------------------------------------------------
def check_state(st, dtype, mode):
    """Every kernel of one evaluation, line search and product (``st``: the device's inputs and outputs, promoted) against its
    restatement.  Returns {quantity: worst err / bound}."""
    u = UNIT[dtype]
    U, lam, alpha, planes, bde = st["U"], st["lam"], st["alpha"], st["planes"], st["bde"]
    rx_lin, mask, freqs, slow, kappa = st["rx_lin"], st["mask"], st["freqs"], st["slow"], st["kappa"]
    nf, ny, nx, nt = U.shape
    nm = mask.shape[1]
    nshare = nodes_shared(rx_lin, mask)
    beta = backward_error(planes, U, st["src_lin"])
    print(f"  backward error of the forward solves: normwise {beta[0]:.2e}, per entry (row scale) {beta[1]:.2e}")
    out = {}
    rc = receiver_ref(U, st["rec"], rx_lin, mask, alpha)
    out["src_est"] = direct("src_est", alpha, rc["alpha"], np.abs(rc["alpha"]), kernel_tol("alpha", dtype, nt, nm, nf), u,
                            ("f", "t"), S_depth=rc["S_alpha"])
    out["loss"] = direct("loss", st["loss"], rc["loss"], rc["S_loss"], kernel_tol("loss", dtype, nt, nm, nf), u, ())
    out["adjoint source"] = behind_solve("adjoint source", planes, lam, rc["adj"], rc["S_adj"],
                                         kernel_tol("adjoint", dtype, nt, nshare=nshare), u, beta, True)
    C = st["C"]

    def grad(L):
        z = z_mass(U, L, alpha, C, bde) if mode == "discrete" else z_reference(U, L, alpha)
        return gradient_from_z(*z, freqs, slow, kappa)

    gt = kernel_tol("gradient_mass" if mode == "discrete" else "gradient", dtype, nt, nf=nf)
    g = grad(lam)
    out["grad_s"] = direct("grad_s", st["grad_s"], g["grad_s"], g["S"], gt, u, ("y", "x"), S_abs=g["S_abs"])
    if kappa is not None:
        out["grad_kappa"] = direct("grad_kappa", st["grad_k"], g["grad_k"], g["S"], gt, u, ("y", "x"), S_abs=g["S_abs"])
    c = rhs_coefficient(freqs, slow, kappa, st["v"], st["vk"])
    if mode == "discrete":
        rhs, S = rhs_mass(U, alpha, C[None] * c, bde)
        rt = kernel_tol("rhs_mass", dtype, nt)
    else:
        rhs, S = rhs_reference(U, alpha, c)
        rt = kernel_tol("rhs", dtype, nt)
    P = st["P"]
    out["perturbation RHS"] = behind_solve("perturbation RHS", planes, P, rhs, S, rt, u, beta, False)
    ls = linesearch_ref(U, P, alpha, st["rec"], rx_lin, mask)
    out["num"] = direct("line search num", st["linesearch"][0], ls["num"], ls["S_num"], kernel_tol("num", dtype, nt, nm, nf), u, ())
    out["den"] = direct("line search den", st["linesearch"][1], ls["den"], ls["S_den"], kernel_tol("den", dtype, nt, nm, nf), u, ())
    # J v of the product is P at the kept receivers: the line search ran on the same direction, and the solves are deterministic
    jv = gather(P, rx_lin, mask)
    assert np.array_equal(st["jv"], jv), "J v is not the perturbation field at the kept receivers"
    jv2 = float(np.sum(np.abs(jv) ** 2))
    out["jv2"] = direct("jv2", st["jv2"], jv2, jv2, kernel_tol("den", dtype, nt, nm, nf), u, ())
    out["J v adjoint source"] = behind_solve("J v adjoint source", planes, st["lam_gn"], scatter_add(jv, rx_lin, mask, U.shape),
                                             scatter_add(np.abs(jv), rx_lin, mask, U.shape),
                                             kernel_tol("jv_scatter", dtype, nt, nshare=nshare), u, beta, True)
    h = grad(st["lam_gn"])
    out["hv_s"] = direct("hv_s", st["hv_s"], h["grad_s"], h["S"], gt, u, ("y", "x"), S_abs=h["S_abs"])
    if kappa is not None:
        out["hv_kappa"] = direct("hv_kappa", st["hv_k"], h["grad_k"], h["S"], gt, u, ("y", "x"), S_abs=h["S_abs"])
    return out


# ---------------------------------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------------------------------
def model(geom, seed=0):
    """(slow, kappa, v, vk) on a geometry: a smooth starting model, a non-constant attenuation slowness and white-noise
    directions (white noise: every pixel's entry differs from its neighbours', so a window or a ring row off by one shows)."""
    X, Y = np.meshgrid(geom.xi.astype(np.float64), geom.yi.astype(np.float64))
    r = 0.2 * min(X.max(), Y.max())
    slow = 1.0 / (C_REF + 20.0 * np.exp(-(X ** 2 + Y ** 2) / (2 * r ** 2)))
    rng = np.random.default_rng(seed + 17)
    k0 = float(G.db_cm_mhz_to_kappa(10.0))
    kappa = k0 * (1.0 + 0.5 * rng.random(slow.shape))
    v = rng.standard_normal(slow.shape) * slow * 1e-2
    vk = rng.standard_normal(slow.shape) * k0 * 0.5
    return slow, kappa, v, vk


def acquisition(geom):
    return (geom.y_idx * geom.Nx + geom.x_idx).astype(np.int64), np.asarray(geom.mask_indices, dtype=np.int64), geom.src_lin


def planes_of(Hm, nx, ny):
    """The nine coefficient planes (9, Ny, Nx) of a sparse operator with interior stencil rows (zero on the ring)."""
    ys, xs = np.meshgrid(np.arange(1, ny - 1), np.arange(1, nx - 1), indexing="ij")
    ctr = (ys * nx + xs).ravel()
    P = np.zeros((9, ny, nx), dtype=Hm.dtype)
    for p, (dy, dx) in enumerate(OFFS):
        P[p, 1:-1, 1:-1] = np.asarray(Hm[ctr, ctr + dy * nx + dx]).reshape(ny - 2, nx - 2)
    return P


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the restatements against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def test_apply_H_and_its_adjoint_match_the_oracle_matrix():
    geom, f, vel = rect_case(58, 44, 32)
    fac = oh.HelmholtzFactor(geom.xi, geom.yi, vel, f, geom.a0, geom.L_PML, "c128", bde=bde_of(vel, f))
    Hm = fac.H.tocsr()
    planes = planes_of(Hm, geom.Nx, geom.Ny)
    rng = np.random.default_rng(5)
    X = rng.standard_normal((geom.Ny, geom.Nx, 3)) + 1j * rng.standard_normal((geom.Ny, geom.Nx, 3))
    N = geom.Nx * geom.Ny
    hx = (Hm @ X.reshape(N, 3)).reshape(X.shape)
    hhx = (Hm.conj().T @ X.reshape(N, 3)).reshape(X.shape)
    habs = (abs(Hm) @ np.abs(X).reshape(N, 3)).reshape(X.shape)
    errs = rel(apply_H(planes, X), hx), rel(apply_HH(planes, X), hhx), rel(apply_H(planes, X, True), habs)
    print(f"H X {errs[0]:.2e}, H^H X {errs[1]:.2e}, |H||X| {errs[2]:.2e}")
    assert max(errs) <= 1e-14
    # the ring of H^H X carries the interior rows next to it
    assert rel(apply_HH(planes, X)[0], hhx[0]) <= 1e-14 and np.abs(hhx[0] - X[0]).max() > 0


def _oracle_state(geom, f, rec, slow, kappa, bde):
    """complex128 oracle fields of one frequency on the discrete reference's operator: unscaled U, alpha, lambda, residuals."""
    ref = Discrete(slow, 0.0 if kappa is None else kappa, fwi_args(geom, rec, f), bde)
    U = ref.fac.solve(geom.dense_src(np.complex128))
    lam = ref.fac.solve(_adjoint_source(ref.diff, ref.gi, geom.Ny, geom.Nx), True)
    return ref, U, lam


def test_restatements_match_the_oracle_reference_mode():
    """Reference linearisation: alpha, loss, adjoint source, gradient, line search and product restated from oracle fields
    against oracle.fwi and the scatter-add reference of test_shapes_and_edges."""
    geom, f, vel_true = rect_case(58, 44, 32)
    slow, _, v, _ = model(geom)
    bde = bde_of(1.0 / slow, f)
    rec = observed_data(geom, f, vel_true, bde=bde_of(vel_true, f))
    rx_lin, mask, _ = acquisition(geom)
    loss_o, grad_o, fl = scatter_add_loss_grad(slow, geom, rec, f, bde)
    loss_oo, grad_oo = ofwi.fwi_loss_and_grad(slow, *fwi_args(geom, rec, f), dtype="c128", bde=bde)
    fac, U, alpha = fl["fac"], fl["U"][None], fl["alpha"][None]
    rc = receiver_ref(U, rec[None], rx_lin, mask, alpha)
    adj_o = _adjoint_source(fl["diff"], fl["inds"], geom.Ny, geom.Nx)
    lam = fac.solve(rc["adj"][0], True)[None]
    g = gradient_from_z(*z_reference(U, lam, alpha), [f], slow, None)
    c = rhs_coefficient([f], slow, None, v, None)
    P = fac.solve(rhs_reference(U, alpha, c)[0][0])[None]
    ls = linesearch_ref(U, P, alpha, rec[None], rx_lin, mask)
    jv = gather(P, rx_lin, mask)
    lam_gn = fac.solve(scatter_add(jv, rx_lin, mask, U.shape)[0], True)[None]
    hv = gradient_from_z(*z_reference(U, lam_gn, alpha), [f], slow, None)["grad_s"]
    hv_o, jv_o = scatter_add_gn_hvp(v, geom, fl)
    errs = dict(alpha=rel(rc["alpha"][0], fl["alpha"]), loss=abs(rc["loss"] - loss_o) / loss_o, adj=rel(rc["adj"][0], adj_o),
                grad=rel(g["grad_s"], grad_o), grad_oracle=rel(g["grad_s"], grad_oo), jv=rel(jv[0], jv_o),
                num=abs(ls["num"] - float(np.real(np.vdot(jv_o, -fl["diff"])))) / abs(ls["num"]),
                den=abs(ls["den"] - float(np.vdot(jv_o, jv_o).real)) / ls["den"], hv=rel(hv, hv_o))
    print(" ".join(f"{k} {e:.1e}" for k, e in errs.items()))
    assert max(errs.values()) <= 1e-13 and abs(loss_oo - loss_o) <= 1e-13 * loss_o


@pytest.mark.parametrize("lossy", [False, True])
def test_restatements_match_the_discrete_reference(lossy):
    """Discrete linearisation (mass stencil and C): gradient, line search, J v and product restated from oracle fields against
    test_discrete_gradient.Discrete, lossless and lossy."""
    geom, f, vel_true = rect_case(63, 40, 31)
    slow, kappa, v, vk = model(geom)
    kappa, vk = (kappa, vk) if lossy else (None, None)
    bde = np.asarray(bde_of(1.0 / slow, f))
    rec = observed_data(geom, f, vel_true, bde=bde_of(vel_true, f))
    rx_lin, mask, _ = acquisition(geom)
    ref, U, lam = _oracle_state(geom, f, rec, slow, kappa, bde)
    U, lam, alpha, C = U[None], lam[None], ref.alpha[None], pml_factor(geom)
    g = gradient_from_z(*z_mass(U, lam, alpha, C, bde[None]), [f], slow, kappa)
    c = rhs_coefficient([f], slow, kappa, v, vk)
    P = ref.fac.solve(rhs_mass(U, alpha, C[None] * c, bde[None])[0][0])[None]
    ls = linesearch_ref(U, P, alpha, rec[None], rx_lin, mask)
    jv = gather(P, rx_lin, mask)
    lam_gn = ref.fac.solve(scatter_add(jv, rx_lin, mask, U.shape)[0], True)[None]
    h = gradient_from_z(*z_mass(U, lam_gn, alpha, C, bde[None]), [f], slow, kappa)
    (hs_o, hk_o), jv_o = ref.hv(v, vk)
    errs = dict(grad_s=rel(g["grad_s"], ref.grad_s), jv=rel(jv[0], jv_o),
                num=abs(ls["num"] - float(np.real(np.vdot(jv_o, -ref.diff)))) / abs(ls["num"]),
                den=abs(ls["den"] - float(np.vdot(jv_o, jv_o).real)) / ls["den"], hv_s=rel(h["grad_s"], hs_o))
    if lossy:
        errs.update(grad_k=rel(g["grad_k"], ref.grad_k), hv_k=rel(h["grad_k"], hk_o))
    print(" ".join(f"{k} {e:.1e}" for k, e in errs.items()))
    assert max(errs.values()) <= 1e-13


# ---------------------------------------------------------------------------------------------------------------------
# CPU: numpy float32 emulations pass the bars, mutated emulations fail them by >= 10x
# ---------------------------------------------------------------------------------------------------------------------
EMULATION_CASES = {
    "odd": (63, 40, 31, 1),     # Nx % 4 = 3: a three-pixel last segment; odd nt: one-source units
    "even": (58, 44, 32, 1),    # Nx % 4 = 2; even nt: two-source units and gradient_kernel's vector path
    "freqs": (49, 36, 32, 3),   # Nx % 4 = 1, three frequencies with their own (b, d, e)
}
_EMU = {}


def emulation_case(name):
    """complex128 oracle fields of a case, cast to complex64 as a complex64 plan would hold them, and the backward error of a
    complex64 direct solver (SuperLU) on the same operator, which stands in for the device's in the bars of the solves."""
    if name in _EMU:
        return _EMU[name]
    if name == "shared":
        geom, f, vel_true, c0, _, _ = _collision_case()
        freqs = [f]
    else:
        nx, ny, nt, nf = EMULATION_CASES[name]
        geom, f, vel_true = rect_case(nx, ny, nt)
        freqs = list(f * np.linspace(0.85, 1.15, nf)) if nf > 1 else [f]
    slow, kappa, v, vk = (a.astype(np.float32) for a in model(geom))
    vel = 1.0 / slow.astype(np.float64)
    rx_lin, mask, src_lin = acquisition(geom)
    SRC = geom.dense_src(np.complex128)
    st = dict(U=[], lam=[], alpha=[], planes=[], rec=[], bde=[], fac=[])
    beta = [0.0, 0.0]
    for i, fi in enumerate(freqs):
        bde = np.asarray(bde_of(vel, fi))
        rec = observed_data(geom, fi, vel_true, bde=bde_of(vel_true, fi), seed=1234 + i)
        fac = oh.HelmholtzFactor(geom.xi, geom.yi, vel, fi, geom.a0, geom.L_PML, "c128", bde=bde)
        U = fac.solve(SRC)
        sim = gather(U[None], rx_lin, mask)[0]
        ob = np.take_along_axis(rec, mask, axis=1)
        alpha = ofwi.estimate_src_strength_batched(sim, ob)
        lam = fac.solve(scatter_add((alpha[:, None] * sim - ob)[None], rx_lin, mask, (1,) + U.shape)[0], True)
        planes = planes_of(fac.H.tocsr(), geom.Nx, geom.Ny)
        fac64 = oh.HelmholtzFactor(geom.xi, geom.yi, vel, fi, geom.a0, geom.L_PML, "c64", bde=bde)
        b = backward_error(planes.astype(np.complex64).astype(np.complex128)[None],
                           fac64.solve(SRC.astype(np.complex64)).astype(np.complex128)[None], src_lin)
        beta = [max(beta[0], b[0]), max(beta[1], b[1])]
        for k, a in (("U", U), ("lam", lam), ("alpha", alpha), ("planes", planes), ("rec", rec), ("bde", bde), ("fac", fac)):
            st[k].append(a)
    for k in ("U", "lam", "alpha", "planes", "rec"):
        st[k] = np.stack(st[k]).astype(np.complex64)
    ex, ey = oh.pml_profiles(geom.xi, geom.yi, geom.a0, geom.L_PML, "c128")
    st.update(geom=geom, freqs=np.asarray(freqs), bde=np.stack(st["bde"]), slow=slow, kappa=kappa, v=v, vk=vk, rx_lin=rx_lin,
              mask=mask, src_lin=src_lin, beta=tuple(beta), C=pml_factor(geom),
              C32=ey[::2].astype(np.complex64).astype(np.complex128)[:, None] * ex[::2].astype(np.complex64)[None, :])
    print(f"{name}: complex64 SuperLU backward error normwise {beta[0]:.2e}, per entry {beta[1]:.2e}")
    _EMU[name] = st
    return st


def _p(st, *keys):
    """float64 promotions of the complex64 / float32 inputs."""
    return [None if st[k] is None else np.asarray(st[k]).astype(np.complex128 if np.iscomplexobj(st[k]) else np.float64)
            for k in keys]


def _lane_terms(au, L):
    """sum_t conj(au_t) L_t as the gradient kernels form it: Re and Im of each term in float32 (au.re L.re + au.im L.im and
    au.re L.im - au.im L.re), the terms summed in FP64."""
    re = au.real * L.real + au.imag * L.imag
    im = au.real * L.imag - au.imag * L.real
    return np.sum(re.astype(np.float64), axis=3) + 1j * np.sum(im.astype(np.float64), axis=3)


def _emulate_gradient(st, mode, lossy, mutation):
    """gradient_kernel / gradient_mass_kernel in float32 (FP64 after z), with one mutation or none: (emulated, restated) dicts."""
    U, lam, alpha = st["U"], st["lam"].copy(), st["alpha"].copy()
    bde, C = st["bde"].copy(), st["C32"]
    kappa = st["kappa"].astype(np.float64) if lossy else None
    slow = st["slow"].astype(np.float64)
    Up, lamp, alphap = _p(st, "U", "lam", "alpha")
    if mutation in ("drop the last source", "drop the last unit of an odd-nt lane"):
        lam[..., -1] = 0
    if mutation == "swap alpha inside a two-source unit":
        alpha = alpha.reshape(alpha.shape[0], -1, 2)[..., ::-1].reshape(alpha.shape)
    if mutation == "frequency 0's (b, d, e) for every frequency":
        bde[:] = bde[0]
    if mutation == "C instead of conj(C)":
        C = np.conj(C)
    if mode == "discrete":
        Wl = np.stack([mass_W(lam[f], bde[f], ring=mutation == "include ring rows of lambda") for f in range(U.shape[0])])
        if mutation == "shift the window of the partial last segment":
            x0 = (U.shape[2] // 4) * 4
            Wl[:, :, x0:] = np.concatenate([Wl[:, :, x0 + 1:], np.zeros_like(Wl[:, :, :1])], axis=2)
        z = np.conj(C) * _lane_terms(alpha[:, None, None, :] * U, Wl)
        emu = gradient_from_z(z, np.abs(z), np.abs(z), st["freqs"], slow, kappa)
        ref = gradient_from_z(*z_mass(Up, lamp, alphap, st["C"], st["bde"]), st["freqs"], slow, kappa)
    else:
        z = _lane_terms(alpha[:, None, None, :] * U, lam)
        emu = gradient_from_z(z, np.abs(z), np.abs(z), st["freqs"], slow, kappa)
        ref = gradient_from_z(*z_reference(Up, lamp, alphap), st["freqs"], slow, kappa)
    if mutation == "flip the sign of kappa A in grad_kappa":
        emu["grad_k"] = emu["grad_k"] + 2 * kappa * emu["A"]
    for k in ("grad_s", "grad_k"):
        emu[k] = emu[k].astype(np.float32)
    return emu, ref


def _gradient_ratio(st, mode, lossy, mutation):
    emu, ref = _emulate_gradient(st, mode, lossy, mutation)
    nt = st["U"].shape[3]
    tol = kernel_tol("gradient_mass" if mode == "discrete" else "gradient", "c64", nt, nf=st["U"].shape[0])
    r = direct("grad_s", emu["grad_s"], ref["grad_s"], ref["S"], tol, U32, ("y", "x"), S_abs=ref["S_abs"])
    if lossy:
        r = max(r, direct("grad_kappa", emu["grad_k"], ref["grad_k"], ref["S"], tol, U32, ("y", "x"), S_abs=ref["S_abs"]))
    return r


def _rhs_ratio(st, mutation):
    """pert_rhs_mass_kernel in float32 on the lossy coefficient, solved exactly (complex128, then cast to complex64), checked
    through the operator like the device's perturbation field."""
    U, alpha, bde = st["U"], st["alpha"], st["bde"].copy()
    slow, kappa, v, vk = (st[k].astype(np.float64) for k in ("slow", "kappa", "v", "vk"))
    c = rhs_coefficient(st["freqs"], slow, kappa, v, vk)
    if mutation == "frequency 0's (b, d, e) for every frequency":
        bde[:] = bde[0]
    coef = (st["C32"][None] * c).astype(np.complex64)
    emu, _ = rhs_mass(U, alpha, coef, bde, keep_ring_rows=mutation == "leave the ring nonzero in the RHS")
    if mutation == "skip the partial segment":
        emu[:, :, (U.shape[2] // 4) * 4:] = 0
    P = np.stack([st["fac"][f].solve(emu[f].astype(np.complex128)) for f in range(U.shape[0])]).astype(np.complex64)
    Up, alphap, planes, Pp = _p(dict(st, P=P), "U", "alpha", "planes", "P")
    rhs, S = rhs_mass(Up, alphap, st["C"][None] * c, st["bde"])
    return behind_solve("perturbation RHS", planes, Pp, rhs, S, kernel_tol("rhs_mass", "c64", U.shape[3]), U32, st["beta"], False)


def _jv2_ratio(st, mutation):
    """gn_receiver_kernel's sum |J v|^2 (FP64 squares of complex64 values) over every kept receiver."""
    U, rx_lin, mask = st["U"], st["rx_lin"], st["mask"]
    jv = gather(U, rx_lin, mask).astype(np.complex128)  # any receiver values: jv2 is their sum of squares
    kept = scatter_add(jv, rx_lin, mask, U.shape, last_write_wins=True) if mutation else jv
    ref = float(np.sum(np.abs(jv) ** 2))
    return direct("jv2", float(np.sum(np.abs(kept) ** 2)), ref, ref, kernel_tol("den", "c64", U.shape[3], mask.shape[1]), U32, ())


def _receiver_ratio(st, mutation):
    """receiver_kernel's adjoint source (float32 residuals) solved exactly and checked through the operator."""
    U, alpha, rec, rx_lin, mask = st["U"], st["alpha"], st["rec"], st["rx_lin"], st["mask"]
    nshare = nodes_shared(rx_lin, mask)
    Up, alphap, recp = _p(st, "U", "alpha", "rec")
    ob = np.take_along_axis(rec, np.broadcast_to(mask, (rec.shape[0],) + mask.shape), axis=2)
    d = alpha[:, :, None] * gather(U, rx_lin, mask) - ob
    adj = scatter_add(d, rx_lin, mask, U.shape, last_write_wins=mutation == "last write wins on a shared node")
    lam = np.stack([st["fac"][f].solve(adj[f].astype(np.complex128), True) for f in range(U.shape[0])]).astype(np.complex64)
    planes, lamp = _p(dict(st, L=lam), "planes", "L")
    rc = receiver_ref(Up, recp, rx_lin, mask, alphap)
    return behind_solve("adjoint source", planes, lamp, rc["adj"], rc["S_adj"], kernel_tol("adjoint", "c64", U.shape[3], nshare=nshare),
                        U32, st["beta"], True)


MUTATIONS = [  # (mutation, case, kernel, mode, lossy)
    ("drop the last source", "even", "gradient", "reference", False),
    ("drop the last unit of an odd-nt lane", "odd", "gradient", "discrete", False),
    ("swap alpha inside a two-source unit", "even", "gradient", "discrete", False),
    ("shift the window of the partial last segment", "odd", "gradient", "discrete", False),
    ("skip the partial segment", "even", "rhs", "discrete", True),
    ("include ring rows of lambda", "odd", "gradient", "discrete", False),
    ("leave the ring nonzero in the RHS", "odd", "rhs", "discrete", True),
    ("C instead of conj(C)", "even", "gradient", "discrete", True),
    ("frequency 0's (b, d, e) for every frequency", "freqs", "gradient", "discrete", False),
    ("frequency 0's (b, d, e) for every frequency", "freqs", "rhs", "discrete", True),
    ("flip the sign of kappa A in grad_kappa", "even", "gradient", "reference", True),
    ("flip the sign of kappa A in grad_kappa", "odd", "gradient", "discrete", True),
    ("last write wins on a shared node", "shared", "receiver", "reference", False),
    ("count a shared-node receiver once in jv2", "shared", "jv2", "reference", False),
]


def _emulated_ratio(case, kernel, mode, lossy, mutation):
    st = emulation_case(case)
    if kernel == "gradient":
        return _gradient_ratio(st, mode, lossy, mutation)
    if kernel == "rhs":
        return _rhs_ratio(st, mutation)
    if kernel == "jv2":
        return _jv2_ratio(st, mutation)
    return _receiver_ratio(st, mutation)


@pytest.mark.parametrize("mutation,case,kernel,mode,lossy", MUTATIONS, ids=[f"{m[0]}-{m[1]}-{m[2]}" for m in MUTATIONS])
def test_bars_catch_mutated_kernels(mutation, case, kernel, mode, lossy):
    print(f"{case}, {kernel}, {mode}, lossy={lossy}: unmutated emulation")
    ok = _emulated_ratio(case, kernel, mode, lossy, None)
    print(f"mutation: {mutation}")
    bad = _emulated_ratio(case, kernel, mode, lossy, mutation)
    assert ok < 1.0, f"the float32 emulation fails its own bar ({ok:.3g})"
    assert bad >= 10.0, f"the bar misses '{mutation}' ({bad:.3g} x the bar)"


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_():
    import torch
    return torch


def _device_state(torch_, plan, geom, freqs, rec, slow, kappa, v, vk, mode):
    """One evaluation, one line search and one product on the plan (same direction for both), with every input and output read
    back and promoted to float64."""
    cplx = np.complex128
    dev = lambda a: torch_.as_tensor(np.ascontiguousarray(np.asarray(a).astype(plan.real))).cuda()
    nf = len(freqs)
    rt = torch_.as_tensor(np.ascontiguousarray(rec.astype(plan.cplx))).cuda()
    plan.set_gradient(mode)
    fields = lambda fn: np.stack([fn(f).cpu().numpy() for f in range(nf)]).astype(cplx)
    st = {}
    if kappa is None:
        loss, g = plan.fwi_loss_grad(dev(slow), rt, freqs)
        st["grad_s"] = g.cpu().numpy().astype(np.float64)
    else:
        loss, gs, gk = plan.fwi_loss_grad_lossy(dev(slow), dev(kappa), rt, freqs)
        st["grad_s"], st["grad_k"] = gs.cpu().numpy().astype(np.float64), gk.cpu().numpy().astype(np.float64)
    st.update(loss=float(loss.cpu().numpy()[0]), U=fields(plan.wavefield), lam=fields(plan.adjoint_wavefield),
              alpha=np.stack([plan.src_est(f) for f in range(nf)]).astype(cplx),
              planes=np.stack([plan.planes(f).cpu().numpy() for f in range(nf)]).astype(cplx), bde=plan.bde()[:nf])
    ls = plan.ncg_linesearch(dev(v)) if kappa is None else plan.ncg_linesearch_lossy(dev(v), dev(vk))
    st["linesearch"] = ls.cpu().numpy()
    st["P"] = fields(plan.adjoint_wavefield)
    if kappa is None:
        hv, jv2, jv = plan.gn_hvp(dev(v), jv=True)
        st["hv_s"] = hv.cpu().numpy().astype(np.float64)
    else:
        hv, jv2, jv = plan.gn_hvp_lossy(dev(v), dev(vk), jv=True)
        st["hv_s"], st["hv_k"] = (h.cpu().numpy().astype(np.float64) for h in hv)
    st.update(jv2=float(jv2.cpu().numpy()[0]), jv=jv.cpu().numpy().astype(cplx), lam_gn=fields(plan.adjoint_wavefield))
    assert plan.status() == 0
    rx_lin, mask, src_lin = acquisition(geom)
    promote = lambda a: None if a is None else np.asarray(a).astype(plan.real).astype(np.float64)
    st.update(rec=rec.astype(plan.cplx).astype(cplx), rx_lin=rx_lin, mask=mask, src_lin=src_lin, freqs=np.asarray(freqs, np.float64),
              slow=promote(slow), kappa=promote(kappa), v=promote(v), vk=promote(vk), C=pml_factor(geom))
    return st


def _run_case(torch_, geom, freqs, rec, dtype, label, groups=(1,)):
    """Both gradient modes, lossless and lossy, on one plan; every ratio must be under 1."""
    from waveforminversionust_b200 import HelmholtzPlan
    engine = "tc2" if dtype == "c64" else "auto"
    plan = HelmholtzPlan(geom.Nx, geom.Ny, dtype=dtype, max_freq=len(freqs), max_nrhs=geom.tx_include.size, fwi_buffers=True,
                         engine=engine)
    plan.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
    plan.set_acquisition(geom.src_lin, (geom.y_idx * geom.Nx + geom.x_idx).astype(np.int32), geom.mask_indices)
    slow, kappa, v, vk = model(geom)
    worst = {}
    try:
        for ngroups in groups:
            plan.set_groups(ngroups)
            for mode in ("reference", "discrete"):
                for lossy in (False, True):
                    tag = f"{label} groups={ngroups} {mode} lossy={lossy}"
                    print(tag)
                    st = _device_state(torch_, plan, geom, freqs, rec, slow, kappa if lossy else None, v, vk if lossy else None, mode)
                    for k, r in check_state(st, dtype, mode).items():
                        worst[(tag, k)] = r
    finally:
        plan.close()
    top = max(worst, key=worst.get)
    print(f"{label}: worst ratio {worst[top]:.3e} ({top[1]}, {top[0]})")
    bad = {k: r for k, r in worst.items() if not r < 1.0}
    assert not bad, bad


DTYPES = ["c64", "c128"]
GRIDS = [(48, 40), (49, 36), (58, 44), (63, 40)]  # Nx % 4 = 0, 1, 2, 3


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("nt", [31, 32])
@pytest.mark.parametrize("nx,ny", GRIDS)
def test_kernels_on_rect_grids(torch_, nx, ny, nt, dtype):
    geom, f, vel_true = rect_case(nx, ny, nt)
    rec = observed_data(geom, f, vel_true, bde=bde_of(vel_true, f))[None]
    _run_case(torch_, geom, [f], rec, dtype, f"{dtype} {nx}x{ny} nt={nt}")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("nt", [67, 96])
def test_kernels_with_lanes_looping_over_units(torch_, nt, dtype):
    """More than 32 units per pixel: every lane of gradient_kernel and of the mass kernels runs several iterations."""
    geom, f, vel_true = rect_case(90, 72, nt)
    rec = observed_data(geom, f, vel_true, bde=bde_of(vel_true, f))[None]
    _run_case(torch_, geom, [f], rec, dtype, f"{dtype} 90x72 nt={nt}")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_kernels_with_receivers_sharing_nodes(torch_, dtype):
    geom, f, vel_true, _, _, rec = _collision_case()
    _run_case(torch_, geom, [f], rec[None], dtype, f"{dtype} shared nodes (48^2, 256 transmitters)")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_kernels_with_two_launch_chains(torch_, dtype):
    """Eight frequencies, one and two launch chains: the second chain's kernels start at frequency q.f0 = 4 and must read that
    frequency's (b, d, e) and w (a group needs four frequencies or more)."""
    geom, f, vel_true = rect_case(58, 44, 32)
    freqs = list(f * np.linspace(0.8, 1.15, 8))
    rec = np.stack([observed_data(geom, fi, vel_true, bde=bde_of(vel_true, fi), seed=1234 + i) for i, fi in enumerate(freqs)])
    _run_case(torch_, geom, freqs, rec, dtype, f"{dtype} 58x44 8 frequencies", groups=(1, 2))


@pytest.mark.gpu
def test_kernels_at_256_with_the_tcgen05_engine(torch_):
    n = 256
    geom = G.ring_geometry(n, 256, dwnsmp=8)
    f = G.frequency_for_grid(n)
    vel_true = G.blob_model(geom)
    h = float(np.mean(np.diff(geom.xi.astype(np.float64))))
    rec = observed_data(geom, f, vel_true, bde=oh.stencil_opt_params(float(vel_true.min()), float(vel_true.max()), f, h, 1.0))
    _run_case(torch_, geom, [f], rec[None], "c64", "c64 256^2 32 transmitters")
