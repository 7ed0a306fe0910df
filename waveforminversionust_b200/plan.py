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
_NP_REAL = {"c64": np.float32, "c128": np.float64}
_NP_CPLX = {"c64": np.complex64, "c128": np.complex128}


def _pd(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _pi(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


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

    def fwi_loss_grad(self, slow, rec, freqs, bde=None):
        """Fused (loss, grad) on device tensors.  slow (ny,nx) real; rec (nfreq, nt, nelem) complex."""
        torch = _torch()
        fr = np.ascontiguousarray(np.atleast_1d(np.asarray(freqs, dtype=np.float64)))
        self._check_tensor(slow, self.treal, self.nx * self.ny)
        self._check_tensor(rec, self.tcplx, fr.size * self.nt * self.nelem)
        b = None if bde is None else np.ascontiguousarray(np.asarray(bde, dtype=np.float64).reshape(fr.size, 3))
        loss = torch.empty(1, dtype=torch.float64, device=slow.device)
        grad = torch.empty((self.ny, self.nx), dtype=self.treal, device=slow.device)
        _lib.check(self.L.ust_fwi_loss_grad(self.h, C.c_void_p(slow.data_ptr()), C.c_void_p(rec.data_ptr()), fr.size,
                                            _pd(fr), _pd(b), C.c_void_p(loss.data_ptr()), C.c_void_p(grad.data_ptr()),
                                            _stream_ptr(self.device)), "ust_fwi_loss_grad")
        self.nfreq = fr.size
        self._factor_key = None  # the plan now holds the factors of (slow, freqs), not api.solve_helmholtz's
        self._eval_key = None  # api.fwi_loss_function records its inputs after this call
        self._keep = (slow, rec)  # ust_ncg_linesearch reads them again
        return loss, grad

    def fwi_loss_grad_lossy(self, slow, kappa, rec, freqs, bde=None):
        """Fused (loss, grad_s, grad_kappa) of a lossy medium on device tensors (``ust_fwi_loss_grad_lossy``): slow and kappa
        (ny, nx) real, rec (nfreq, nt, nelem) complex.  Afterwards ``ncg_linesearch`` and ``gn_hvp`` refuse until the next
        ``fwi_loss_grad``."""
        torch = _torch()
        fr = np.ascontiguousarray(np.atleast_1d(np.asarray(freqs, dtype=np.float64)))
        self._check_tensor(slow, self.treal, self.nx * self.ny)
        self._check_tensor(kappa, self.treal, self.nx * self.ny)
        self._check_tensor(rec, self.tcplx, fr.size * self.nt * self.nelem)
        b = None if bde is None else np.ascontiguousarray(np.asarray(bde, dtype=np.float64).reshape(fr.size, 3))
        loss = torch.empty(1, dtype=torch.float64, device=slow.device)
        grad_s = torch.empty((self.ny, self.nx), dtype=self.treal, device=slow.device)
        grad_k = torch.empty((self.ny, self.nx), dtype=self.treal, device=slow.device)
        _lib.check(self.L.ust_fwi_loss_grad_lossy(self.h, C.c_void_p(slow.data_ptr()), C.c_void_p(kappa.data_ptr()),
                                                  C.c_void_p(rec.data_ptr()), fr.size, _pd(fr), _pd(b), C.c_void_p(loss.data_ptr()),
                                                  C.c_void_p(grad_s.data_ptr()), C.c_void_p(grad_k.data_ptr()),
                                                  _stream_ptr(self.device)), "ust_fwi_loss_grad_lossy")
        self.nfreq = fr.size
        self._factor_key = None
        self._eval_key = None
        return loss, grad_s, grad_k

    def ncg_linesearch(self, sd):
        torch = _torch()
        self._check_tensor(sd, self.treal, self.nx * self.ny)
        out = torch.empty(2, dtype=torch.float64, device=sd.device)
        _lib.check(self.L.ust_ncg_linesearch(self.h, C.c_void_p(sd.data_ptr()), C.c_void_p(out.data_ptr()),
                                             _stream_ptr(self.device)), "ust_ncg_linesearch")
        return out

    def gn_hvp(self, v, jv=False):
        """Gauss-Newton product on the state of the last ``fwi_loss_grad`` (no factorisation): ``v`` (ny, nx) real CUDA
        tensor -> ``(hv, jv2[, jv])`` with ``hv = Re(J^H J v)`` (ny, nx), ``jv2 = sum |J v|^2`` (1-element float64 tensor)
        and, when ``jv``, ``J v`` at the kept receivers (nfreq, nt, nm) complex (``ust_fwi_gn_hvp``)."""
        torch = _torch()
        self._check_tensor(v, self.treal, self.nx * self.ny)
        hv = torch.empty((self.ny, self.nx), dtype=self.treal, device=v.device)
        jv2 = torch.empty(1, dtype=torch.float64, device=v.device)
        jvt = torch.empty((getattr(self, "nfreq", 1), self.nt, getattr(self, "nm", 0)), dtype=self.tcplx, device=v.device) if jv else None
        _lib.check(self.L.ust_fwi_gn_hvp(self.h, C.c_void_p(v.data_ptr()), C.c_void_p(hv.data_ptr()), C.c_void_p(jv2.data_ptr()),
                                         C.c_void_p(jvt.data_ptr()) if jv else None, _stream_ptr(self.device)), "ust_fwi_gn_hvp")
        return (hv, jv2, jvt) if jv else (hv, jv2)

    def ncg_linesearch_lossy(self, sd_s, sd_k):
        """Line-search scalars ``[num, den]`` (2-element float64 tensor) of the joint direction ``[sd_s, sd_k]`` on the state of
        the last ``fwi_loss_grad_lossy`` (``ust_ncg_linesearch_lossy``)."""
        torch = _torch()
        self._check_tensor(sd_s, self.treal, self.nx * self.ny)
        self._check_tensor(sd_k, self.treal, self.nx * self.ny)
        out = torch.empty(2, dtype=torch.float64, device=sd_s.device)
        _lib.check(self.L.ust_ncg_linesearch_lossy(self.h, C.c_void_p(sd_s.data_ptr()), C.c_void_p(sd_k.data_ptr()),
                                                   C.c_void_p(out.data_ptr()), _stream_ptr(self.device)), "ust_ncg_linesearch_lossy")
        return out

    def gn_hvp_lossy(self, v_s, v_k, jv=False):
        """Joint Gauss-Newton product on the state of the last ``fwi_loss_grad_lossy``: ``v_s``, ``v_k`` (ny, nx) real CUDA
        tensors -> ``(hv, jv2[, jv])`` with ``hv = Re(J^H J v)`` (2, ny, nx) = [s, kappa] blocks, ``jv2 = sum |J v|^2``
        (1-element float64 tensor) and, when ``jv``, ``J v`` at the kept receivers (nfreq, nt, nm) complex
        (``ust_fwi_gn_hvp_lossy``)."""
        torch = _torch()
        self._check_tensor(v_s, self.treal, self.nx * self.ny)
        self._check_tensor(v_k, self.treal, self.nx * self.ny)
        hv = torch.empty((2, self.ny, self.nx), dtype=self.treal, device=v_s.device)
        jv2 = torch.empty(1, dtype=torch.float64, device=v_s.device)
        jvt = torch.empty((getattr(self, "nfreq", 1), self.nt, getattr(self, "nm", 0)), dtype=self.tcplx, device=v_s.device) if jv else None
        _lib.check(self.L.ust_fwi_gn_hvp_lossy(self.h, C.c_void_p(v_s.data_ptr()), C.c_void_p(v_k.data_ptr()),
                                               C.c_void_p(hv[0].data_ptr()), C.c_void_p(hv[1].data_ptr()), C.c_void_p(jv2.data_ptr()),
                                               C.c_void_p(jvt.data_ptr()) if jv else None, _stream_ptr(self.device)),
                   "ust_fwi_gn_hvp_lossy")
        return (hv, jv2, jvt) if jv else (hv, jv2)

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

    def fwi_loss_grad_host(self, slow, rec, freqs, bde=None, out_grad=None):
        """slow (ny,nx) real host array, rec (nfreq, nt, nelem) complex host array (pinned or pageable)."""
        fr = np.ascontiguousarray(np.atleast_1d(np.asarray(freqs, dtype=np.float64)))
        slow = np.ascontiguousarray(np.asarray(slow, dtype=self.real))
        rec = np.ascontiguousarray(np.asarray(rec).astype(self.cplx, copy=False))
        if rec.size != fr.size * self.nt * self.nelem:
            raise ValueError("REC_DATA has the wrong shape for (nfreq, nt, nelem)")
        b = None if bde is None else np.ascontiguousarray(np.asarray(bde, dtype=np.float64).reshape(fr.size, 3))
        grad = out_grad if out_grad is not None else np.empty((self.ny, self.nx), dtype=self.real)
        loss = C.c_double(0.0)
        _lib.check(self.L.ust_fwi_loss_grad_host(self.h, slow.ctypes.data_as(C.c_void_p), rec.ctypes.data_as(C.c_void_p),
                                                 fr.size, _pd(fr), _pd(b), C.byref(loss), grad.ctypes.data_as(C.c_void_p)),
                   "ust_fwi_loss_grad_host")
        self.nfreq = fr.size
        self._factor_key = None
        self._eval_key = None
        return loss.value, grad

    def fwi_loss_grad_lossy_host(self, slow, kappa, rec, freqs, bde=None):
        """Host twin of ``fwi_loss_grad_lossy`` (``ust_fwi_loss_grad_lossy_host``): NumPy in, ``(loss, grad_s, grad_kappa)`` out."""
        fr = np.ascontiguousarray(np.atleast_1d(np.asarray(freqs, dtype=np.float64)))
        slow = np.ascontiguousarray(np.asarray(slow, dtype=self.real))
        kappa = np.ascontiguousarray(np.asarray(kappa, dtype=self.real))
        rec = np.ascontiguousarray(np.asarray(rec).astype(self.cplx, copy=False))
        if rec.size != fr.size * self.nt * self.nelem:
            raise ValueError("REC_DATA has the wrong shape for (nfreq, nt, nelem)")
        if slow.size != self.nx * self.ny or kappa.size != self.nx * self.ny:
            raise ValueError("slowness and kappa must have ny * nx entries")
        b = None if bde is None else np.ascontiguousarray(np.asarray(bde, dtype=np.float64).reshape(fr.size, 3))
        grad_s = np.empty((self.ny, self.nx), dtype=self.real)
        grad_k = np.empty((self.ny, self.nx), dtype=self.real)
        loss = C.c_double(0.0)
        _lib.check(self.L.ust_fwi_loss_grad_lossy_host(self.h, slow.ctypes.data_as(C.c_void_p), kappa.ctypes.data_as(C.c_void_p),
                                                       rec.ctypes.data_as(C.c_void_p), fr.size, _pd(fr), _pd(b), C.byref(loss),
                                                       grad_s.ctypes.data_as(C.c_void_p), grad_k.ctypes.data_as(C.c_void_p)),
                   "ust_fwi_loss_grad_lossy_host")
        self.nfreq = fr.size
        self._factor_key = None
        self._eval_key = None
        return loss.value, grad_s, grad_k

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
