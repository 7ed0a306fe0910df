"""ctypes binding of libustfwi.so (the C ABI in include/ustfwi.h).

The product path has no CPU fallback: if the CUDA library is missing or a call fails,
an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_LIB = None

EXPORTS = [
    "ust_last_error", "ust_version", "ust_plan_create", "ust_plan_destroy", "ust_plan_device_bytes",
    "ust_plan_set_groups", "ust_plan_set_gradient", "ust_plan_set_grid", "ust_plan_set_acquisition", "ust_factor", "ust_factor_lossy", "ust_solve",
    "ust_solve_helmholtz_host", "ust_fwi_loss_grad", "ust_fwi_loss_grad_host", "ust_fwi_loss_grad_lossy", "ust_fwi_loss_grad_lossy_host", "ust_ncg_linesearch", "ust_fwi_gn_hvp",
    "ust_ncg_linesearch_lossy", "ust_fwi_gn_hvp_lossy", "ust_get_bde", "ust_get_planes",
    "ust_get_src_est", "ust_get_wavefield", "ust_get_adjoint_wavefield", "ust_get_status",
    "ust_launch_count", "ust_launch_count_reset", "ust_profile", "ust_get_profile", "ust_test_cgemm", "ust_idtft", "ust_pack_f64_as_f32x2", "ust_residual_onehot",
]


class PlanDesc(C.Structure):
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("dtype", C.c_int), ("max_freq", C.c_int),
                ("max_nrhs", C.c_int), ("device", C.c_int), ("stencil", C.c_int), ("engine", C.c_int),
                ("fwi_buffers", C.c_int)]


class UstError(RuntimeError):
    pass


def lib():
    """Load libustfwi.so (built in-tree by ``build.build_library``).  Raises if absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIBPATH
    if not os.path.exists(path):
        raise UstError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)")
    L = C.CDLL(path)
    vp, i, d = C.c_void_p, C.c_int, C.c_double
    pd = C.POINTER(C.c_double)
    pi = C.POINTER(C.c_int32)
    L.ust_last_error.restype = C.c_char_p
    L.ust_version.restype = C.c_char_p
    L.ust_plan_create.argtypes = [C.POINTER(PlanDesc), C.POINTER(vp)]
    L.ust_plan_destroy.argtypes = [vp]
    L.ust_plan_device_bytes.argtypes = [vp]
    L.ust_plan_device_bytes.restype = C.c_size_t
    L.ust_plan_set_groups.argtypes = [vp, i]
    L.ust_plan_set_gradient.argtypes = [vp, i]
    L.ust_plan_set_grid.argtypes = [vp, pd, pd, d, d]
    L.ust_plan_set_acquisition.argtypes = [vp, i, pi, i, pi, i, pi]
    L.ust_factor.argtypes = [vp, vp, i, pd, pd, vp]
    L.ust_factor_lossy.argtypes = [vp, vp, vp, i, pd, pd, vp]
    L.ust_solve.argtypes = [vp, i, vp, i, i, vp]
    L.ust_solve_helmholtz_host.argtypes = [vp, vp, vp, vp, i, d, pd, i, i]
    L.ust_fwi_loss_grad.argtypes = [vp, vp, vp, i, pd, pd, vp, vp, vp]
    L.ust_fwi_loss_grad_host.argtypes = [vp, vp, vp, i, pd, pd, pd, vp]
    L.ust_fwi_loss_grad_lossy.argtypes = [vp, vp, vp, vp, i, pd, pd, vp, vp, vp, vp]
    L.ust_fwi_loss_grad_lossy_host.argtypes = [vp, vp, vp, vp, i, pd, pd, pd, vp, vp]
    L.ust_ncg_linesearch.argtypes = [vp, vp, vp, vp]
    L.ust_fwi_gn_hvp.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ust_ncg_linesearch_lossy.argtypes = [vp, vp, vp, vp, vp]
    L.ust_fwi_gn_hvp_lossy.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.ust_get_bde.argtypes = [vp, pd]
    L.ust_get_planes.argtypes = [vp, i, vp, vp]
    L.ust_get_src_est.argtypes = [vp, i, vp]
    L.ust_get_wavefield.argtypes = [vp, i]
    L.ust_get_wavefield.restype = vp
    L.ust_get_adjoint_wavefield.argtypes = [vp, i]
    L.ust_get_adjoint_wavefield.restype = vp
    L.ust_get_status.argtypes = [vp, C.POINTER(C.c_int)]
    L.ust_residual_onehot.argtypes = [vp, i, i, pd]
    L.ust_idtft.argtypes = [i, vp, i, C.c_longlong, pd, pd, d, pd, i, vp, vp]
    L.ust_pack_f64_as_f32x2.argtypes = [vp, vp, i, vp]
    L.ust_launch_count.restype = C.c_longlong
    L.ust_test_cgemm.argtypes = [i, i, i, i, i, vp, i, vp, i, vp, i, vp, i, C.c_float, i, i, i, i, vp]
    L.ust_profile.argtypes = [vp, i]
    L.ust_get_profile.argtypes = [vp, pd, C.POINTER(C.c_longlong)]
    _LIB = L
    return L


def check(rc, what=""):
    if rc != 0:
        msg = lib().ust_last_error()
        raise UstError(f"{what}: {msg.decode() if msg else 'unknown error'}")
