"""Python handle on a ``ust_plan`` (include/ustfwi.h).  torch is used only for device memory,
streams and (in ``distributed.py``) the NCCL all-reduce -- every numerical step is a call into
libustfwi.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

DTYPES = {"c64": 0, "c128": 1}
STENCILS = {"python": 0, "matlab": 1}
ENGINES = {"auto": 0, "simt": 1, "tc2": 3}
GRADIENTS = {"reference": 0, "discrete": 1}
_NP_REAL = {"c64": np.float32, "c128": np.float64}
_NP_CPLX = {"c64": np.complex64, "c128": np.complex128}


def _pd(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _pi(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _torch():
    import torch
    return torch


def _stream_ptr(device):
    torch = _torch()
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class HelmholtzPlan:
    """Owns factor storage and workspaces for one grid size / precision on one GPU."""

    def __init__(self, nx, ny, dtype="c64", max_freq=1, max_nrhs=256, device=0, stencil="python",
                 fwi_buffers=False, engine="auto"):
        self.L = _lib.lib()
        self.nx, self.ny, self.dtype = int(nx), int(ny), dtype
        self.max_freq, self.max_nrhs, self.device = int(max_freq), int(max_nrhs), int(device)
        self.real, self.cplx = _NP_REAL[dtype], _NP_CPLX[dtype]
        desc = _lib.PlanDesc(self.nx, self.ny, DTYPES[dtype], self.max_freq, self.max_nrhs, self.device,
                             STENCILS[stencil], ENGINES[engine], int(bool(fwi_buffers)))
        self.engine = engine
        h = C.c_void_p()
        _lib.check(self.L.ust_plan_create(C.byref(desc), C.byref(h)), "ust_plan_create")
        self.h = h
        self.nt = 0
        self._grid_key = None
        self._acq_key = None
        self._factor_key = None
        self._eval_key = None  # inputs of the last fwi_loss_function on this plan (api.fwi_gauss_newton_product)
        self.gradient = "reference"  # ust_plan_set_gradient's mode (set_gradient)

    def close(self):
        if getattr(self, "h", None):
            self.L.ust_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_bytes(self):
        return int(self.L.ust_plan_device_bytes(self.h))

    def set_groups(self, ngroups):
        """Number of independent launch chains (streams) the frequencies of one call are split into."""
        _lib.check(self.L.ust_plan_set_groups(self.h, int(ngroups)), "ust_plan_set_groups")

    def set_gradient(self, mode):
        """Linearisation behind the gradient, the line search and the Gauss-Newton product (``ust_plan_set_gradient``):
        ``"reference"`` (the default) is the reference's virtual source ``2 w^2 sigma alpha u``; ``"discrete"`` adds the
        stencil's 9-point mass weights and the PML factor, so that the gradient is the exact derivative of the discrete loss at
        fixed stencil weights (DESIGN.md section 7f).  A line search or product refuses when the mode differs from the one the
        last evaluation ran with."""
        if mode not in GRADIENTS:
            raise ValueError(f"gradient must be one of {sorted(GRADIENTS)}, got {mode!r}")
        _lib.check(self.L.ust_plan_set_gradient(self.h, GRADIENTS[mode]), "ust_plan_set_gradient")
        self.gradient = mode

    # -- setup ------------------------------------------------------------------------------
    def set_grid(self, x, y, a0, L_PML):
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float64))
        if x.size != self.nx or y.size != self.ny:
            raise ValueError("grid size does not match the plan")
        key = (x.tobytes(), y.tobytes(), float(a0), float(L_PML))
        if key == self._grid_key:
            return
        _lib.check(self.L.ust_plan_set_grid(self.h, _pd(x), _pd(y), float(a0), float(L_PML)), "ust_plan_set_grid")
        self._grid_key = key
        self._factor_key = None

    def set_acquisition(self, src_lin, rx_lin, mask_indices):
        src_lin = np.ascontiguousarray(np.asarray(src_lin, dtype=np.int32))
        rx_lin = np.ascontiguousarray(np.asarray(rx_lin, dtype=np.int32))
        mask = np.ascontiguousarray(np.asarray(mask_indices, dtype=np.int32))
        key = (src_lin.tobytes(), rx_lin.tobytes(), mask.tobytes())
        if key == self._acq_key:
            return
        nt, nm = mask.shape
        if src_lin.size != nt:
            raise ValueError("mask_indices must have one row per transmitter")
        _lib.check(self.L.ust_plan_set_acquisition(self.h, nt, _pi(src_lin), rx_lin.size, _pi(rx_lin), nm, _pi(mask)),
                   "ust_plan_set_acquisition")
        self.nt, self.nelem, self.nm = nt, rx_lin.size, nm
        self._acq_key = key

    # -- device-pointer entry points (torch CUDA tensors) -------------------------------------
    def _check_tensor(self, t, dtype, numel=None):
        torch = _torch()
        if not (t.is_cuda and t.is_contiguous() and t.device.index == self.device):
            raise ValueError("expected a contiguous CUDA tensor on the plan's device")
        if t.dtype != dtype:
            raise ValueError(f"expected dtype {dtype}, got {t.dtype}")
        if numel is not None and t.numel() != numel:
            raise ValueError("tensor has the wrong number of elements")

    @property
    def treal(self):
        torch = _torch()
        return torch.float32 if self.dtype == "c64" else torch.float64

    @property
    def tcplx(self):
        torch = _torch()
        return torch.complex64 if self.dtype == "c64" else torch.complex128

    def factor(self, vel, freqs, bde=None, kappa=None):
        """Assemble + factorise for ``freqs`` (list) from a (ny, nx) CUDA tensor of sound speed.  ``kappa`` (a (ny, nx) CUDA
        tensor of attenuation slowness, s/m) factorises the lossy operator of the complex slowness ``1/vel - i kappa``
        (``ust_factor_lossy``)."""
        self._check_tensor(vel, self.treal, self.nx * self.ny)
        fr = np.ascontiguousarray(np.atleast_1d(np.asarray(freqs, dtype=np.float64)))
        b = None if bde is None else np.ascontiguousarray(np.asarray(bde, dtype=np.float64).reshape(fr.size, 3))
        if kappa is None:
            _lib.check(self.L.ust_factor(self.h, C.c_void_p(vel.data_ptr()), fr.size, _pd(fr), _pd(b), _stream_ptr(self.device)),
                       "ust_factor")
        else:
            self._check_tensor(kappa, self.treal, self.nx * self.ny)
            _lib.check(self.L.ust_factor_lossy(self.h, C.c_void_p(vel.data_ptr()), C.c_void_p(kappa.data_ptr()), fr.size, _pd(fr),
                                               _pd(b), _stream_ptr(self.device)), "ust_factor_lossy")
        self.nfreq = fr.size
        self._factor_key = None  # api.solve_helmholtz's cached factorisation is gone (it re-sets the key itself)
        self._eval_key = None  # the factors of the last fwi_loss_grad are gone too (api.fwi_gauss_newton_product)

    def solve(self, rhs, ifreq=0, adjoint=False):
        """In-place solve; ``rhs`` is an (ny*nx, nrhs) (or (ny, nx, nrhs)) complex CUDA tensor."""
        nrhs = rhs.numel() // (self.nx * self.ny)
        self._check_tensor(rhs, self.tcplx, self.nx * self.ny * nrhs)
        _lib.check(self.L.ust_solve(self.h, int(ifreq), C.c_void_p(rhs.data_ptr()), nrhs, int(bool(adjoint)),
                                    _stream_ptr(self.device)), "ust_solve")
        return rhs

    def _evaluated(self, nfreq):
        self.nfreq = nfreq
        self._factor_key = None  # the plan now holds the factors of this evaluation, not api.solve_helmholtz's
        self._eval_key = None  # api.fwi_loss_function records its inputs after this call

    def _freqs_bde(self, freqs, bde):
        fr = np.ascontiguousarray(np.atleast_1d(np.asarray(freqs, dtype=np.float64)))
        b = None if bde is None else np.ascontiguousarray(np.asarray(bde, dtype=np.float64).reshape(fr.size, 3))
        return fr, b

    def _loss_grad(self, slow, kappa, rec, freqs, bde):
        """(loss, grad) on device tensors, or (loss, grad_s, grad_kappa) of the lossy medium when ``kappa`` is given."""
        torch = _torch()
        fr, b = self._freqs_bde(freqs, bde)
        maps = [slow] if kappa is None else [slow, kappa]
        for t in maps:
            self._check_tensor(t, self.treal, self.nx * self.ny)
        self._check_tensor(rec, self.tcplx, fr.size * self.nt * self.nelem)
        loss = torch.empty(1, dtype=torch.float64, device=slow.device)
        grads = [torch.empty((self.ny, self.nx), dtype=self.treal, device=slow.device) for _ in maps]
        name = "ust_fwi_loss_grad" if kappa is None else "ust_fwi_loss_grad_lossy"
        _lib.check(getattr(self.L, name)(self.h, *map(_ptr, maps), _ptr(rec), fr.size, _pd(fr), _pd(b), _ptr(loss),
                                         *map(_ptr, grads), _stream_ptr(self.device)), name)
        self._evaluated(fr.size)
        return (loss, *grads)

    def fwi_loss_grad(self, slow, rec, freqs, bde=None):
        """Fused (loss, grad) on device tensors.  slow (ny,nx) real; rec (nfreq, nt, nelem) complex."""
        return self._loss_grad(slow, None, rec, freqs, bde)

    def fwi_loss_grad_lossy(self, slow, kappa, rec, freqs, bde=None):
        """Fused (loss, grad_s, grad_kappa) of a lossy medium on device tensors (``ust_fwi_loss_grad_lossy``): slow and kappa
        (ny, nx) real, rec (nfreq, nt, nelem) complex.  Afterwards ``ncg_linesearch`` and ``gn_hvp`` refuse until the next
        ``fwi_loss_grad``."""
        return self._loss_grad(slow, kappa, rec, freqs, bde)

    def _linesearch(self, sd, sd_k):
        """Line-search scalars [num, den] of ``sd`` (lossy: of the joint direction [sd, sd_k])."""
        torch = _torch()
        dirs = [sd] if sd_k is None else [sd, sd_k]
        for t in dirs:
            self._check_tensor(t, self.treal, self.nx * self.ny)
        out = torch.empty(2, dtype=torch.float64, device=sd.device)
        name = "ust_ncg_linesearch" if sd_k is None else "ust_ncg_linesearch_lossy"
        _lib.check(getattr(self.L, name)(self.h, *map(_ptr, dirs), _ptr(out), _stream_ptr(self.device)), name)
        return out

    def ncg_linesearch(self, sd):
        return self._linesearch(sd, None)

    def ncg_linesearch_lossy(self, sd_s, sd_k):
        """Line-search scalars ``[num, den]`` (2-element float64 tensor) of the joint direction ``[sd_s, sd_k]`` on the state of
        the last ``fwi_loss_grad_lossy`` (``ust_ncg_linesearch_lossy``)."""
        return self._linesearch(sd_s, sd_k)

    def _gn_hvp(self, v, v_k, jv):
        """Gauss-Newton product of ``v`` (lossy: of the joint direction [v, v_k], hv of shape (2, ny, nx))."""
        torch = _torch()
        dirs = [v] if v_k is None else [v, v_k]
        for t in dirs:
            self._check_tensor(t, self.treal, self.nx * self.ny)
        hv = torch.empty((self.ny, self.nx) if v_k is None else (2, self.ny, self.nx), dtype=self.treal, device=v.device)
        jv2 = torch.empty(1, dtype=torch.float64, device=v.device)
        jvt = torch.empty((getattr(self, "nfreq", 1), self.nt, getattr(self, "nm", 0)), dtype=self.tcplx, device=v.device) if jv else None
        name = "ust_fwi_gn_hvp" if v_k is None else "ust_fwi_gn_hvp_lossy"
        hvs = [hv] if v_k is None else [hv[0], hv[1]]
        _lib.check(getattr(self.L, name)(self.h, *map(_ptr, dirs), *map(_ptr, hvs), _ptr(jv2), _ptr(jvt) if jv else None,
                                         _stream_ptr(self.device)), name)
        return (hv, jv2, jvt) if jv else (hv, jv2)

    def gn_hvp(self, v, jv=False):
        """Gauss-Newton product on the state of the last ``fwi_loss_grad`` (no factorisation): ``v`` (ny, nx) real CUDA
        tensor -> ``(hv, jv2[, jv])`` with ``hv = Re(J^H J v)`` (ny, nx), ``jv2 = sum |J v|^2`` (1-element float64 tensor)
        and, when ``jv``, ``J v`` at the kept receivers (nfreq, nt, nm) complex (``ust_fwi_gn_hvp``)."""
        return self._gn_hvp(v, None, jv)

    def gn_hvp_lossy(self, v_s, v_k, jv=False):
        """Joint Gauss-Newton product on the state of the last ``fwi_loss_grad_lossy``: ``v_s``, ``v_k`` (ny, nx) real CUDA
        tensors -> ``(hv, jv2[, jv])`` with ``hv = Re(J^H J v)`` (2, ny, nx) = [s, kappa] blocks, ``jv2 = sum |J v|^2``
        (1-element float64 tensor) and, when ``jv``, ``J v`` at the kept receivers (nfreq, nt, nm) complex
        (``ust_fwi_gn_hvp_lossy``)."""
        return self._gn_hvp(v_s, v_k, jv)

    # -- host-buffer entry points (NumPy; no torch needed) ------------------------------------
    def solve_helmholtz_host(self, vel, src, f, adjoint=False, bde=None, refactor=True):
        vel = None if vel is None else np.ascontiguousarray(np.asarray(vel, dtype=self.real))
        src = np.ascontiguousarray(np.asarray(src).astype(self.cplx, copy=False))
        nrhs = src.size // (self.nx * self.ny)
        out = np.empty((self.ny, self.nx, nrhs), dtype=self.cplx)
        b = None if bde is None else np.ascontiguousarray(np.asarray(bde, dtype=np.float64).reshape(3))
        if refactor:
            self._eval_key = None
        _lib.check(self.L.ust_solve_helmholtz_host(
            self.h, None if vel is None else vel.ctypes.data_as(C.c_void_p), src.ctypes.data_as(C.c_void_p),
            out.ctypes.data_as(C.c_void_p), nrhs, float(f), _pd(b), int(bool(adjoint)), int(bool(refactor))),
            "ust_solve_helmholtz_host")
        return out

    def _loss_grad_host(self, slow, kappa, rec, freqs, bde, out_grad):
        """(loss, grad) on host arrays, or (loss, grad_s, grad_kappa) of the lossy medium when ``kappa`` is given.
        ``out_grad``: the gradient array to fill, (ny, nx) or, lossy, (2, ny, nx); None allocates."""
        fr, b = self._freqs_bde(freqs, bde)
        maps = [np.ascontiguousarray(np.asarray(m, dtype=self.real)) for m in ([slow] if kappa is None else [slow, kappa])]
        rec = np.ascontiguousarray(np.asarray(rec).astype(self.cplx, copy=False))
        if rec.size != fr.size * self.nt * self.nelem:
            raise ValueError("REC_DATA has the wrong shape for (nfreq, nt, nelem)")
        if any(m.size != self.nx * self.ny for m in maps):
            raise ValueError("slowness and kappa must have ny * nx entries" if kappa is not None else "slowness must have ny * nx entries")
        if out_grad is None:
            grads = [np.empty((self.ny, self.nx), dtype=self.real) for _ in maps]
        elif out_grad.dtype != self.real or out_grad.size != len(maps) * self.nx * self.ny or not out_grad.flags.c_contiguous:
            raise ValueError(f"out_grad must be a C-contiguous {np.dtype(self.real)} array of {len(maps)} * ny * nx entries")
        else:
            grads = [out_grad] if kappa is None else list(out_grad.reshape(2, self.ny, self.nx))
        loss = C.c_double(0.0)
        name = "ust_fwi_loss_grad_host" if kappa is None else "ust_fwi_loss_grad_lossy_host"
        _lib.check(getattr(self.L, name)(self.h, *(m.ctypes.data_as(C.c_void_p) for m in maps), rec.ctypes.data_as(C.c_void_p),
                                         fr.size, _pd(fr), _pd(b), C.byref(loss), *(g.ctypes.data_as(C.c_void_p) for g in grads)),
                   name)
        self._evaluated(fr.size)
        return (loss.value, *grads)

    def fwi_loss_grad_host(self, slow, rec, freqs, bde=None, out_grad=None):
        """slow (ny,nx) real host array, rec (nfreq, nt, nelem) complex host array (pinned or pageable)."""
        return self._loss_grad_host(slow, None, rec, freqs, bde, out_grad)

    def fwi_loss_grad_lossy_host(self, slow, kappa, rec, freqs, bde=None):
        """Host twin of ``fwi_loss_grad_lossy`` (``ust_fwi_loss_grad_lossy_host``): NumPy in, ``(loss, grad_s, grad_kappa)`` out."""
        return self._loss_grad_host(slow, kappa, rec, freqs, bde, None)

    # -- introspection ---------------------------------------------------------------------
    def bde(self):
        out = np.zeros((self.max_freq, 3), dtype=np.float64)
        _lib.check(self.L.ust_get_bde(self.h, _pd(out)), "ust_get_bde")
        return out

    def planes(self, ifreq=0):
        torch = _torch()
        out = torch.empty((9, self.ny, self.nx), dtype=self.tcplx, device=f"cuda:{self.device}")
        _lib.check(self.L.ust_get_planes(self.h, int(ifreq), C.c_void_p(out.data_ptr()), _stream_ptr(self.device)),
                   "ust_get_planes")
        return out

    def src_est(self, ifreq=0):
        out = np.zeros(self.nt, dtype=self.cplx)
        _lib.check(self.L.ust_get_src_est(self.h, int(ifreq), out.ctypes.data_as(C.c_void_p)), "ust_get_src_est")
        return out

    def residual_onehot(self, ifreq=0, t=0):
        """(||H u_t - e_src||, || |H||u| ||) of forward column t after fwi_loss_grad: a correct solve has a ratio at the
        rounding level of the precision, whatever the grid size."""
        out = np.zeros(2, dtype=np.float64)
        _lib.check(self.L.ust_residual_onehot(self.h, int(ifreq), int(t), _pd(out)), "ust_residual_onehot")
        return float(out[0]), float(out[1])

    def _field(self, fn, ifreq):
        torch = _torch()
        ptr = fn(self.h, int(ifreq))
        if not ptr:
            raise _lib.UstError("wavefield buffers are not allocated (fwi_buffers=False)")
        n = self.nx * self.ny * self.nt
        out = torch.empty((self.ny, self.nx, self.nt), dtype=self.tcplx, device=f"cuda:{self.device}")
        torch.cuda.current_stream(self.device).synchronize()
        # view the plan-owned buffer through __cuda_array_interface__ and copy it device-to-device
        itemsize = np.dtype(self.cplx).itemsize
        src = _from_dev_ptr(ptr, n * itemsize, self.device)
        out.view(torch.uint8).reshape(-1).copy_(src)
        return out

    def wavefield(self, ifreq=0):
        """Forward field of the last fwi_loss_grad (UNSCALED by the source estimate), (ny, nx, nt)."""
        return self._field(self.L.ust_get_wavefield, ifreq)

    def adjoint_wavefield(self, ifreq=0):
        return self._field(self.L.ust_get_adjoint_wavefield, ifreq)

    PROFILE_CLASSES = ("assemble", "schur", "gj_panel", "gj_update", "tri_apply", "sweep_gemm", "receiver", "gradient", "t_split", "gj_pivot", "gj_rowpanel", "gj_k0")

    def profile(self, enable=True):
        _lib.check(self.L.ust_profile(self.h, int(bool(enable))), "ust_profile")

    def get_profile(self):
        """{class: (total_ms, launches)} of the kernels launched since profiling was enabled / last read."""
        ms = np.zeros(16, dtype=np.float64)
        cnt = np.zeros(16, dtype=np.int64)
        _lib.check(self.L.ust_get_profile(self.h, _pd(ms), cnt.ctypes.data_as(C.POINTER(C.c_longlong))), "ust_get_profile")
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.PROFILE_CLASSES)}

    def status(self):
        s = C.c_int(0)
        _lib.check(self.L.ust_get_status(self.h, C.byref(s)), "ust_get_status")
        return s.value


class _DevMem:
    """Minimal __cuda_array_interface__ wrapper so torch can view a raw device pointer."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def _from_dev_ptr(ptr, nbytes, device):
    torch = _torch()
    return torch.as_tensor(_DevMem(ptr, nbytes), device=f"cuda:{device}")
