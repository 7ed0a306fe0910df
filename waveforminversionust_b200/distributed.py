"""Frequency and source-block sharding over the GPUs of one box (SURVEY.md section 8(e)).

``shard="freq"``: the joint multi-frequency objective sum_f loss_f shards naturally: rank r owns a contiguous block of
frequencies -- its own assembly, factorisation, all-source sweeps, source estimates and partial gradient.
``shard="source"`` (BASELINE configs[3]: one large grid, many sources): the right-hand-side columns are independent
(``solve_helmholtz.py:78``) and loss and gradient are sums over sources (``nonlinearcg.py:264-265``,
``fwi_loss_function.py:102``), so rank r owns a contiguous block of transmitters -- its rows of REC_DATA / mask_indices, its
one-hot columns -- while the factorisation of every frequency is REPLICATED on every rank (the sweeps shrink by 1/world, the
factorisation does not: the speed-up is capped at (F + S) / (F + S / world)).
Either way the only exchange is ONE all-reduce (sum) per evaluation of a packed buffer
[grad (Ny*Nx reals), loss_hi, loss_lo] over NCCL/NVLink (gloo on CPU for the host-logic tests).
torch.distributed is plumbing only; all numerics are in libustfwi.so.
"""
from __future__ import annotations

import numpy as np


def shard_frequencies(nfreq, rank, world):
    """Contiguous balanced partition of range(nfreq) (frequencies, or transmitters for source-block sharding): the first
    nfreq % world ranks get one extra item."""
    base, extra = divmod(int(nfreq), int(world))
    lo = rank * base + min(rank, extra)
    return list(range(lo, lo + base + (1 if rank < extra else 0)))


def pack_loss_grad(loss, grad):
    """One flat buffer [grad..., loss_hi, loss_lo]; the loss is split so that a float32 gradient buffer
    still carries it to ~1e-14 relative."""
    import torch
    flat = grad.reshape(-1)
    loss = torch.as_tensor(loss, dtype=torch.float64, device=flat.device).reshape(1)
    hi = loss.to(flat.dtype)
    lo = (loss - hi.to(torch.float64)).to(flat.dtype)
    return torch.cat([flat, hi, lo])


def unpack_loss_grad(buf, shape):
    import torch
    loss = buf[-2].to(torch.float64) + buf[-1].to(torch.float64)
    return loss, buf[:-2].reshape(shape)


def allreduce_loss_grad(loss, grad, group=None):
    """Sum (loss, grad) over the ranks of ``group`` with a single all-reduce."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        import torch
        return torch.as_tensor(loss, dtype=torch.float64, device=grad.device).reshape(()), grad
    buf = pack_loss_grad(loss, grad)
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return unpack_loss_grad(buf, grad.shape)


class ShardedFWI:
    """(loss, grad) of the joint objective over ``freqs`` with the frequencies sharded over the ranks of
    the default process group.  One instance per rank / GPU.  ``gradient`` (``"reference"`` or ``"discrete"``,
    ``HelmholtzPlan.set_gradient``) is the linearisation of its gradients and Gauss-Newton products."""

    def __init__(self, geom, freqs, dtype="c64", device=0, stencil="python", rank=None, world=None, group=None,
                 engine="auto", shard="freq", *, gradient="reference"):
        import torch
        import torch.distributed as dist
        from .plan import HelmholtzPlan
        self.torch = torch
        self.group = group
        if rank is None:
            rank = dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0
        if world is None:
            world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank, self.world = rank, world
        self.freqs = np.asarray(freqs, dtype=np.float64)
        if shard not in ("freq", "source"):
            raise ValueError("shard must be 'freq' or 'source'")
        self.shard = shard
        nt_all = geom.tx_include.size
        if shard == "freq":
            self.local = shard_frequencies(self.freqs.size, rank, world)  # plan frequency slots = these frequencies
            self.local_tx = list(range(nt_all))
        else:
            self.local = list(range(self.freqs.size))                      # every rank factorises every frequency
            self.local_tx = shard_frequencies(nt_all, rank, world)         # ... and sweeps its own block of transmitters
        self.local_freqs = self.freqs[self.local]
        self.geom, self.device = geom, device
        self.plan = HelmholtzPlan(geom.Nx, geom.Ny, dtype=dtype, max_freq=max(len(self.local), 1),
                                  max_nrhs=max(len(self.local_tx), 1), device=device, stencil=stencil, fwi_buffers=True,
                                  engine=engine)
        self.plan.set_grid(geom.xi, geom.yi, geom.a0, geom.L_PML)
        self.plan.set_gradient(gradient)
        rx_lin = (geom.y_idx * geom.Nx + geom.x_idx).astype(np.int32)
        if len(self.local_tx):
            self.plan.set_acquisition(geom.src_lin[self.local_tx], rx_lin, geom.mask_indices[self.local_tx])
        dv = torch.device(f"cuda:{device}")
        self._slow_dev = torch.empty((geom.Ny, geom.Nx), dtype=self.plan.treal, device=dv)
        self._rec_dev = torch.empty((max(len(self.local), 1), max(len(self.local_tx), 1), geom.num_elements),
                                    dtype=self.plan.tcplx, device=dv)

    def _allreduced(self, evaluate, like, blocks):
        """``evaluate() -> (scalar (1-element float64 tensor), result)`` on a rank that owns frequencies and transmitters,
        zeros of ``like``'s shape (``blocks`` > 1: ``(blocks,) + like.shape``) on one that does not, then one all-reduce of
        the packed ``[result, scalar]``.  Returns ``(scalar (0-d float64 tensor), result)``."""
        torch = self.torch
        if len(self.local) and len(self.local_tx):
            scalar, result = evaluate()
            scalar = scalar[0]
        else:
            scalar = torch.zeros((), dtype=torch.float64, device=like.device)
            result = torch.zeros(((blocks,) if blocks > 1 else ()) + tuple(like.shape), dtype=like.dtype, device=like.device)
        return allreduce_loss_grad(scalar, result, self.group)

    def loss_grad_device(self, slow_dev, rec_local_dev, bde=None):
        """Inputs already resident in HBM.  Returns all-reduced (loss (0-d float64 tensor), grad)."""
        return self._allreduced(lambda: self.plan.fwi_loss_grad(slow_dev, rec_local_dev, self.local_freqs, bde=bde), slow_dev, 1)

    def gn_hvp_device(self, v_dev):
        """Gauss-Newton product of the joint objective at the point of the last ``loss_grad_device``: this rank's part
        (``HelmholtzPlan.gn_hvp``: its frequencies or its transmitters) and one all-reduce of the packed ``[hv, jv2]``.
        Returns ``(hv, jv2)`` with ``jv2 = sum |J v|^2`` (0-d float64 tensor)."""
        jv2, hv = self._allreduced(lambda: self.plan.gn_hvp(v_dev)[::-1], v_dev, 1)
        return hv, jv2

    def loss_grad_lossy_device(self, slow_dev, kappa_dev, rec_local_dev, bde=None):
        """Joint sound-speed and attenuation evaluation (``HelmholtzPlan.fwi_loss_grad_lossy``) of this rank's frequencies or
        transmitters, and one all-reduce of the packed ``[grad_s, grad_kappa, loss]``.  Returns (loss (0-d float64 tensor),
        grad (2, Ny, Nx) = [grad_s, grad_kappa])."""
        def evaluate():
            loss, gs, gk = self.plan.fwi_loss_grad_lossy(slow_dev, kappa_dev, rec_local_dev, self.local_freqs, bde=bde)
            return loss, self.torch.stack([gs, gk])
        return self._allreduced(evaluate, slow_dev, 2)

    def gn_hvp_lossy_device(self, v_s_dev, v_k_dev):
        """Joint Gauss-Newton product at the point of the last ``loss_grad_lossy_device``: this rank's part
        (``HelmholtzPlan.gn_hvp_lossy``: its frequencies or its transmitters) and one all-reduce of the packed
        ``[hv_s, hv_kappa, jv2]``.  Returns ``(hv (2, Ny, Nx), jv2 (0-d float64 tensor))``."""
        jv2, hv = self._allreduced(lambda: self.plan.gn_hvp_lossy(v_s_dev, v_k_dev)[::-1], v_s_dev, 2)
        return hv, jv2

    def local_rec(self, rec_all):
        """This rank's part of the full observed data ``rec_all`` (nfreq, Nt, E): its frequencies (all transmitters) or its
        transmitters (all frequencies)."""
        r = rec_all[self.local] if self.shard == "freq" else rec_all[:, self.local_tx]
        return r

    def loss_grad_host(self, slow_host, rec_local_host, bde=None):
        """HOST buffers in (pinned torch tensors or NumPy arrays), host results out: host->device copies,
        the evaluation, the all-reduce and the device->host read are all inside this call."""
        torch = self.torch
        s = slow_host if torch.is_tensor(slow_host) else torch.as_tensor(np.asarray(slow_host))
        r = rec_local_host if torch.is_tensor(rec_local_host) else torch.as_tensor(np.asarray(rec_local_host))
        self._slow_dev.copy_(s.reshape(self._slow_dev.shape), non_blocking=True)
        nl = len(self.local)
        if nl:
            self._rec_dev[:nl].copy_(r.reshape(self._rec_dev[:nl].shape), non_blocking=True)
        loss, grad = self.loss_grad_device(self._slow_dev, self._rec_dev[:max(nl, 1)], bde=bde)
        out = pack_loss_grad(loss, grad).cpu()  # device->host read of the step's result (synchronises)
        l, g = unpack_loss_grad(out, grad.shape)
        return float(l), g.numpy()

    @property
    def h2d_bytes(self):
        nl = len(self.local)
        return int(self._slow_dev.numel() * self._slow_dev.element_size()
                   + nl * self._rec_dev[0].numel() * self._rec_dev.element_size())

    @property
    def d2h_bytes(self):
        return int((self._slow_dev.numel() + 2) * self._slow_dev.element_size())

    def close(self):
        self.plan.close()


def _engine_callables(eng, rec_local_dev, lossy):
    """The objective of the ``api`` drivers on a sharded engine, on (Ny, Nx) slowness maps or, ``lossy``, (2, Ny, Nx) =
    [s, kappa] models: ``loss_grad(x)`` and ``hvp(v)`` (at the point of the last ``loss_grad``) on float64 torch tensors, and
    ``loss_grad_np(x)`` on NumPy arrays for the L-BFGS drivers."""
    import torch
    plan = eng.plan
    dv = torch.device(f"cuda:{eng.device}")

    def split(x):
        x = x.to(dv, plan.treal)
        return (x[0].contiguous(), x[1].contiguous()) if lossy else (x.contiguous(),)

    def loss_grad(x):
        loss, grad = (eng.loss_grad_lossy_device if lossy else eng.loss_grad_device)(*split(x), rec_local_dev)
        return float(loss), grad

    def hvp(v):
        return (eng.gn_hvp_lossy_device if lossy else eng.gn_hvp_device)(*split(v))[0]

    def loss_grad_np(x):
        loss, grad = loss_grad(torch.as_tensor(np.ascontiguousarray(x.astype(plan.real))))
        return loss, grad.to(torch.float64).cpu().numpy()

    return loss_grad, hvp, loss_grad_np


def _use_gradient(eng, gradient):
    """``gradient`` None keeps the engine's mode; a mode name sets it on the engine's plan for this and later calls."""
    if gradient is not None:
        eng.plan.set_gradient(gradient)


def run_lbfgs_sharded(eng, rec_local_dev, c_init, maxiter=1, tol=1e-5, history_size=10, history=None, pert_scale=1e-2, *,
                      gradient=None):
    """``run_lbfgs_fwi`` (``fwi_loss_function.py:106-132``) on a sharded engine -- BASELINE configs[4]: multi-frequency L-BFGS on
    several GPUs.  Every rank runs the same L-BFGS driver (``api.run_lbfgs_fwi``) on the all-reduced joint (loss, grad), which
    NCCL delivers bit-identically to all ranks, so the ranks take identical steps without any further exchange.
    ``rec_local_dev``: this rank's observed data on its device (``eng.local_rec`` of the full set).  Returns the final sound
    speed (Ny, Nx) as a NumPy array (identical on every rank).  ``gradient``: the gradient mode (None: the engine's)."""
    from . import api
    _use_gradient(eng, gradient)
    geom, plan = eng.geom, eng.plan
    loss_grad = _engine_callables(eng, rec_local_dev, False)[2]
    return api.run_lbfgs_fwi(geom.xi, geom.yi, None, None, geom.tx_include, geom.ind_matlab, c_init, eng.freqs, geom.a0, geom.L_PML,
                             geom.mask_indices, maxiter=maxiter, tol=tol, history_size=history_size, dtype=plan.dtype,
                             history=history, loss_grad=loss_grad, pert_scale=pert_scale)


def run_gauss_newton_sharded(eng, rec_local_dev, c_init, Niter, cg_iters=8, cg_tol=1e-2, damping=0.0, max_backtracks=4, history=None,
                             *, gradient=None):
    """``api.gauss_newton_fwi`` on a sharded engine: every rank runs the same driver on the all-reduced (loss, grad) and
    products, which NCCL delivers bit-identically to all ranks, so the ranks take identical steps.  ``rec_local_dev``: this
    rank's observed data on its device (``eng.local_rec`` of the full set).  Returns the final sound speed (Ny, Nx).
    ``gradient``: the linearisation of the gradient and the products (None: the engine's)."""
    from . import api
    _use_gradient(eng, gradient)
    geom, plan = eng.geom, eng.plan
    loss_grad, hvp, _ = _engine_callables(eng, rec_local_dev, False)
    return api.gauss_newton_fwi(geom.xi, geom.yi, geom.num_elements, None, None, geom.tx_include, geom.ind_matlab, c_init, eng.freqs,
                                Niter, geom.a0, geom.L_PML, geom.mask_indices, cg_iters=cg_iters, cg_tol=cg_tol, damping=damping,
                                max_backtracks=max_backtracks, dtype=plan.dtype, device=eng.device, history=history,
                                loss_grad=loss_grad, hvp=hvp)


def run_lbfgs_joint_sharded(eng, rec_local_dev, c_init, kappa_init=0.0, kappa_scale=None, maxiter=1, tol=1e-5, history_size=10,
                            history=None, pert_scale=1e-2, *, gradient=None):
    """``api.run_lbfgs_joint_fwi`` on a sharded engine: every rank runs the same joint L-BFGS driver on the all-reduced
    ``(loss, [grad_s, grad_kappa])`` of ``ShardedFWI.loss_grad_lossy_device``, so the ranks take identical steps.  Returns
    ``(c, kappa)`` (Ny, Nx) NumPy arrays (identical on every rank).  ``gradient``: the gradient mode (None: the engine's)."""
    from . import api
    _use_gradient(eng, gradient)
    geom, plan = eng.geom, eng.plan
    loss_grad = _engine_callables(eng, rec_local_dev, True)[2]
    return api.run_lbfgs_joint_fwi(geom.xi, geom.yi, None, None, geom.tx_include, geom.ind_matlab, c_init, eng.freqs, geom.a0,
                                   geom.L_PML, geom.mask_indices, kappa_init=kappa_init, kappa_scale=kappa_scale, maxiter=maxiter,
                                   tol=tol, history_size=history_size, dtype=plan.dtype, history=history, loss_grad=loss_grad,
                                   pert_scale=pert_scale)


def run_gauss_newton_joint_sharded(eng, rec_local_dev, c_init, Niter, kappa_init=0.0, kappa_scale=None, pert_scale=1e-2, cg_iters=8,
                                   cg_tol=1e-2, damping=0.0, max_backtracks=4, history=None, *, gradient=None):
    """``api.gauss_newton_joint_fwi`` on a sharded engine: every rank runs the same joint driver on the all-reduced
    ``loss_grad_lossy_device`` and ``gn_hvp_lossy_device``, so the ranks take identical steps.  Returns ``(c, kappa)`` (Ny, Nx)
    NumPy arrays (identical on every rank).  ``gradient``: the linearisation of the gradient and the products (None: the
    engine's)."""
    from . import api
    _use_gradient(eng, gradient)
    geom, plan = eng.geom, eng.plan
    loss_grad, hvp, _ = _engine_callables(eng, rec_local_dev, True)
    return api.gauss_newton_joint_fwi(geom.xi, geom.yi, geom.num_elements, None, None, geom.tx_include, geom.ind_matlab, c_init,
                                      eng.freqs, Niter, geom.a0, geom.L_PML, geom.mask_indices, kappa_init=kappa_init,
                                      kappa_scale=kappa_scale, pert_scale=pert_scale, cg_iters=cg_iters, cg_tol=cg_tol,
                                      damping=damping, max_backtracks=max_backtracks, dtype=plan.dtype, device=eng.device,
                                      history=history, loss_grad=loss_grad, hvp=hvp)
